// polar_scl_api.cu -- the C entry points of the list decoder (include/polar_b200.h, polar_scl_*), for every arithmetic.
// A call is checked (check_scl_args), planned (scl_plan: which mapping runs, its grid and its workspace) and dispatched
// to scl3_kernel (polar_scl3.cu, min-sum only) or to scl2_kernel<L> of its arithmetic (polar_scl.cu: launch_scl2, and
// launch_scl2_boxplus from the same source compiled through polar_bp_wrap.cu).
//
// The hybrid SC -> SCL decoder lives here too: CRC-aided selection in the `use_hybrid_sc` mode of the Sionna-style
// SCL_Dec (my_sn/fec/polar/dec.py:437-470).  It decodes the whole batch with SC, keeps every SC decision whose CRC holds,
// and list-decodes only the rows whose CRC fails.  At a working Eb/N0 almost every SC decision passes, so the batch
// costs about one SC decode plus a partial wave of the list kernel instead of a full list decode.  Four stream-ordered
// operations, no host synchronisation:
//   1. polar_sc_decode_f32 / polar_sc_decode_boxplus_f32 over all B rows -> packed decisions and u_info
//   2. memset of the failing-row count
//   3. hybrid_crc_check_kernel: syndrome of each packed row, indices of the failing rows appended to fail_rows[]
//   4. scl2_kernel<L> of the arithmetic over fail_rows[0 .. count-1], overwriting those rows
// The list stage is the generic scl2 mapping in every arithmetic: its decisions equal scl3's bit for bit, and in the
// regime the hybrid is for it decodes a small fraction of the batch.
#include <algorithm>

#include "polar_common.cuh"
#include "polar_internal.h"
#include "polar_scl.h"

namespace polar {

static int scl_mode() { return env_int("POLAR_SCL_MODE", 2); }   // 2: scl3 where supported, else scl2 [default]; 1: scl2 always (tests)

int check_scl_shape(const char *who, int n, int L, int64_t B) {
  if (!is_pow2(n) || n < 2 || n > POLAR_SCL_MAX_N) return set_error(POLAR_EINVAL, "%s: n=%d must be a power of two in [2,%d]", who, n, POLAR_SCL_MAX_N);
  if (!is_pow2(L) || L > POLAR_SCL_MAX_L) return set_error(POLAR_EINVAL, "%s: list_size=%d must be a power of two <= %d", who, L, POLAR_SCL_MAX_L);
  if (B < 0) return set_error(POLAR_EINVAL, "%s: B=%lld < 0", who, (long long)B);
  return POLAR_OK;
}

// ws_bytes is what the mapping needs at its full grid.  For scl3 it is also at least one scl2 warp per SM: a caller
// sizes the workspace before it knows whether its rows will be 16-byte aligned, and on misaligned rows scl2 runs with
// as many warps as the workspace holds (its full-grid appetite is ~1.3 GB at n = 1024, L = 8, not worth reserving).
SclPlan scl_plan(int n, int L, int64_t B, SclArith arith, bool scl3_rows) {
  // scl2_kernel<L>, one warp per CTA: 4 KB of shared memory per warp hold the low LLR stages and, up to n = 128, the
  // partial-sum words; the other stages and words live in the workspace.  32 CTAs per SM fill the register file at 64
  // registers per thread.
  constexpr size_t kSmemPerWarp = 4096;
  constexpr int kWarpsPerSm = 32;
  SclPlan pl;
  const int m = ilog2(n);
  const size_t words = (size_t)32 * 2 * POLAR_WORDS(n) * 4;
  pl.words_global = words > 1024;
  const size_t wsm = pl.words_global ? 0 : words;
  int s_glob = m;
  while (s_glob > 0 && scl2_llr_smem_doubles(s_glob) * 8 + wsm > kSmemPerWarp) --s_glob;
  pl.s_glob = s_glob;
  pl.smem_per_warp = std::max<size_t>(16, (scl2_llr_smem_doubles(s_glob) * 8 + wsm + 15) / 16 * 16);
  pl.ws_bytes_per_warp = sizeof(double) * ((size_t)32 * ((1u << m) - (1u << s_glob)) + (pl.words_global ? words / 8 : 0));
  const int cpw = 32 / L;
  pl.grid = std::min((B + cpw - 1) / cpw, (int64_t)device_sm_count() * kWarpsPerSm);
  pl.ws_bytes = (size_t)pl.grid * pl.ws_bytes_per_warp;
  pl.scl3 = false;
  Scl3Plan p3;
  if (scl3_rows && arith == SclArith::minsum && scl_mode() == 2 && scl3_supported(n, L) &&
      launch_scl3(nullptr, nullptr, n, L, B, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, 0, nullptr, nullptr, &p3) == POLAR_OK) {
    const size_t floor2 = std::min(pl.ws_bytes, (size_t)device_sm_count() * pl.ws_bytes_per_warp);
    pl.scl3 = true;
    pl.grid = p3.grid;
    pl.ws_bytes_per_warp = p3.ws_bytes_per_warp;
    pl.ws_bytes = std::max((size_t)p3.grid * p3.ws_bytes_per_warp, floor2);
  }
  return pl;
}

namespace {

// The arguments of a list decode on device buffers.  A call with B == 0 launches nothing: it passes once n, L, B and,
// when a CRC is required (the hybrid), the CRC and k are valid, whatever its buffers.
int check_scl_args(const char *who, int n, int L, int64_t B, const float *logit, const uint32_t *fmask, bool has_output,
                   const float *u_info, const int32_t *info_pos, int k, const uint32_t *crc_rows, int crc_len, bool need_crc) {
  const int rc = check_scl_shape(who, n, L, B);
  if (rc != POLAR_OK) return rc;
  if (need_crc && (crc_len < 1 || crc_len > 32 || !crc_rows || k < 1 || k > n))
    return set_error(POLAR_EINVAL, "%s: needs a CRC (crc_len in [1,32] and crc_rows) and k in [1,%d], got crc_len=%d k=%d", who, n, crc_len, k);
  if (B == 0) return POLAR_OK;
  if (!logit || !fmask) return set_error(POLAR_EINVAL, "%s: null logit / frozen_mask", who);
  if (!has_output) return set_error(POLAR_EINVAL, "%s: no output buffer", who);
  if (u_info && (!info_pos || k < 0 || k > n)) return set_error(POLAR_EINVAL, "%s: u_info requested without valid info_pos/k", who);
  if (crc_len < 0 || crc_len > 32 || (crc_len > 0 && !crc_rows)) return set_error(POLAR_EINVAL, "%s: bad crc_len / crc_rows", who);
  if (crc_len > 0 && (k < 1 || k > n)) return set_error(POLAR_EINVAL, "%s: CRC-aided selection needs k (penalty 30 k, dec.py:517-518), got k=%d", who, k);
  return POLAR_OK;
}

// One list decode on device buffers: every polar_scl_decode* call, and the list stage of the hybrid, which passes the
// rows to decode (rows[0 .. min(*n_rows, B)-1], written earlier on the stream; only scl2 decodes a row list).
int scl_decode(SclArith arith, const float *logit, const uint32_t *fmask, int n, int L, int64_t B, uint32_t *best,
               float *u_info, const int32_t *info_pos, int k, double *pm, uint32_t *list, const uint32_t *crc_rows,
               int crc_len, void *ws, size_t ws_bytes, void *stream, const int32_t *rows = nullptr,
               const int32_t *n_rows = nullptr) {
  const int rc = check_scl_args("scl", n, L, B, logit, fmask, best || u_info || pm || list, u_info, info_pos, k, crc_rows,
                                crc_len, false);
  if (rc != POLAR_OK || B == 0) return rc;
  SclPlan pl = scl_plan(n, L, B, arith, !rows && ((uintptr_t)logit & 15) == 0);
  const size_t need = (size_t)pl.grid * pl.ws_bytes_per_warp;
  const cudaStream_t st = (cudaStream_t)stream;
  if (pl.scl3) {
    if (!ws || ws_bytes < need) return set_error(POLAR_ENOMEM, "scl: workspace %zu B < required %zu B", ws_bytes, need);
    if ((uintptr_t)ws & 255) return set_error(POLAR_EALIGN, "scl: workspace must be 256-byte aligned");
    return launch_scl3(logit, fmask, n, L, B, best, u_info, info_pos, k, pm, list, crc_rows, crc_len, ws, st, nullptr);
  }
  if (need > 0) {
    if (!ws) return set_error(POLAR_ENOMEM, "scl: workspace %zu B < required %zu B", (size_t)0, need);
    if ((uintptr_t)ws & 255) return set_error(POLAR_EALIGN, "scl: workspace must be 256-byte aligned");
    if (ws_bytes < need) {   // the kernel is persistent: run with as many warps as the workspace holds
      if (ws_bytes < pl.ws_bytes_per_warp) return set_error(POLAR_ENOMEM, "scl: workspace %zu B < required %zu B", ws_bytes, pl.ws_bytes_per_warp);
      pl.grid = (int64_t)(ws_bytes / pl.ws_bytes_per_warp);
    }
  }
  SclParams P;
  P.logit = logit; P.fmask = fmask; P.n = n; P.m = ilog2(n); P.B = B;
  P.best = best; P.u_info = u_info; P.info_pos = info_pos; P.k = k;
  P.pm_out = pm; P.list = list; P.crc_rows = crc_rows; P.crc_len = crc_len;
  P.ws = (double *)ws; P.ws_doubles_per_warp = pl.ws_bytes_per_warp / sizeof(double); P.s_glob = pl.s_glob;
  P.smem_per_warp = pl.smem_per_warp; P.words_global = pl.words_global; P.fast = arith == SclArith::boxplus_pruned;
  P.rows = rows; P.n_rows = n_rows;
  return arith == SclArith::minsum ? launch_scl2(P, pl, L, st) : launch_scl2_boxplus(P, pl, L, st);
}

constexpr unsigned kFull = 0xFFFFFFFFu;

inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Workspace layout of the hybrid, every region 256-byte aligned:
//   [0]          packed SC decisions [B, POLAR_WORDS(n)] uint32 (used when the caller passes no d_best_packed)
//   [count_off]  failing-row count, int32 (used when the caller passes no d_n_list_out)
//   [rows_off]   failing-row indices [B] int32
//   [scl_off]    scl2_kernel<L> workspace planned for B rows
struct HybridLayout { size_t count_off, rows_off, scl_off, total; };

HybridLayout hybrid_layout(int n, int L, int64_t B, SclArith arith) {
  HybridLayout h;
  h.count_off = align256((size_t)B * POLAR_WORDS(n) * sizeof(uint32_t));
  h.rows_off = h.count_off + 256;
  h.scl_off = h.rows_off + align256((size_t)B * sizeof(int32_t));
  h.total = h.scl_off + align256(scl_plan(n, L, B, arith, false).ws_bytes);
  return h;
}

// G = min(POLAR_WORDS(n), 32) lanes per row (a power of two), 32 / G rows per warp step.  A lane XORs crc_rows[i] over the
// set bits i of its words; the warp reduces per row; failing rows are appended with one atomic per warp step.
__global__ void __launch_bounds__(256) hybrid_crc_check_kernel(const uint32_t *__restrict__ packed, int n, int64_t B,
                                                               const uint32_t *__restrict__ crc_rows, int32_t *count,
                                                               int32_t *__restrict__ fail_rows) {
  const int nw = POLAR_WORDS(n);
  const int G = nw < 32 ? nw : 32;
  const int lane = threadIdx.x & 31, sub = lane / G, gl = lane & (G - 1);
  const int rpw = 32 / G;
  const int64_t nsteps = (B + rpw - 1) / rpw;
  const int64_t stride = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < nsteps; s += stride) {
    const int64_t b = s * rpw + sub;
    uint32_t syn = 0u;
    if (b < B) {
      const uint32_t *row = packed + b * nw;
      for (int w = gl; w < nw; w += G) {
        uint32_t uw = row[w];
        while (uw) {
          const int pos = w * 32 + __ffs(uw) - 1;
          uw &= uw - 1u;
          if (pos < n) syn ^= __ldg(crc_rows + pos);
        }
      }
    }
    for (int d = G >> 1; d > 0; d >>= 1) syn ^= __shfl_xor_sync(kFull, syn, d);
    const bool fail = b < B && gl == 0 && syn != 0u;
    const unsigned m = __ballot_sync(kFull, fail);
    if (m) {
      const int leader = __ffs(m) - 1;
      int base = 0;
      if (lane == leader) base = atomicAdd(count, __popc(m));
      base = __shfl_sync(kFull, base, leader);
      if (fail) fail_rows[base + __popc(m & ((1u << lane) - 1u))] = (int32_t)b;
    }
  }
}

}  // namespace

}  // namespace polar

using namespace polar;

extern "C" size_t polar_scl_workspace_bytes(int n, int L, int64_t B) {
  if (B <= 0 || check_scl_shape("scl", n, L, B) != POLAR_OK) return 0;
  return scl_plan(n, L, B, SclArith::minsum, true).ws_bytes;
}

extern "C" size_t polar_scl_boxplus_workspace_bytes(int n, int L, int64_t B) {
  if (B <= 0 || check_scl_shape("scl", n, L, B) != POLAR_OK) return 0;
  return scl_plan(n, L, B, SclArith::boxplus, true).ws_bytes;
}

extern "C" int polar_scl_decode(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                                uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                                double *d_pm_sorted, uint32_t *d_list_packed, const uint32_t *d_crc_rows, int crc_len,
                                void *d_workspace, size_t workspace_bytes, void *stream) {
  return scl_decode(SclArith::minsum, d_logit, d_frozen_mask, n, L, B, d_best_packed, d_u_info_f32, d_info_pos, k, d_pm_sorted,
                    d_list_packed, d_crc_rows, crc_len, d_workspace, workspace_bytes, stream);
}

extern "C" int polar_scl_decode_boxplus(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                                        uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                                        double *d_pm_sorted, uint32_t *d_list_packed, const uint32_t *d_crc_rows, int crc_len,
                                        void *d_workspace, size_t workspace_bytes, void *stream) {
  return scl_decode(SclArith::boxplus, d_logit, d_frozen_mask, n, L, B, d_best_packed, d_u_info_f32, d_info_pos, k, d_pm_sorted,
                    d_list_packed, d_crc_rows, crc_len, d_workspace, workspace_bytes, stream);
}

// use_fast_scl = True of the Sionna-style decoder: rate-0 / REP nodes update the path metric at node level
extern "C" int polar_scl_decode_boxplus_pruned(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                                               uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                                               double *d_pm_sorted, uint32_t *d_list_packed, const uint32_t *d_crc_rows, int crc_len,
                                               void *d_workspace, size_t workspace_bytes, void *stream) {
  return scl_decode(SclArith::boxplus_pruned, d_logit, d_frozen_mask, n, L, B, d_best_packed, d_u_info_f32, d_info_pos, k,
                    d_pm_sorted, d_list_packed, d_crc_rows, crc_len, d_workspace, workspace_bytes, stream);
}

extern "C" size_t polar_scl_hybrid_workspace_bytes(int n, int L, int64_t B, int cn_mode) {
  if (B <= 0 || B > INT32_MAX || cn_mode < 0 || cn_mode > 2 || check_scl_shape("hybrid", n, L, B) != POLAR_OK) return 0;
  return hybrid_layout(n, L, B, (SclArith)cn_mode).total;
}

extern "C" int polar_scl_decode_hybrid(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                                       uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                                       const uint32_t *d_crc_rows, int crc_len, int cn_mode, int32_t *d_n_list_out,
                                       void *d_workspace, size_t workspace_bytes, void *stream) {
  if (cn_mode < 0 || cn_mode > 2) return set_error(POLAR_EINVAL, "hybrid: cn_mode=%d must be 0 (min-sum), 1 (boxplus) or 2 (boxplus pruned)", cn_mode);
  if (B > INT32_MAX) return set_error(POLAR_EINVAL, "hybrid: B=%lld must be in [0, 2^31)", (long long)B);
  int rc = check_scl_args("hybrid", n, L, B, d_logit, d_frozen_mask, d_best_packed || d_u_info_f32, d_u_info_f32, d_info_pos, k,
                          d_crc_rows, crc_len, true);
  if (rc != POLAR_OK || B == 0) return rc;
  const SclArith arith = (SclArith)cn_mode;
  const HybridLayout h = hybrid_layout(n, L, B, arith);
  if (!d_workspace || workspace_bytes < h.total) return set_error(POLAR_ENOMEM, "hybrid: workspace %zu B < required %zu B", d_workspace ? workspace_bytes : (size_t)0, h.total);
  if ((uintptr_t)d_workspace & 255) return set_error(POLAR_EALIGN, "hybrid: workspace must be 256-byte aligned");

  unsigned char *ws = (unsigned char *)d_workspace;
  uint32_t *sc_packed = d_best_packed ? d_best_packed : (uint32_t *)ws;
  int32_t *count = d_n_list_out ? d_n_list_out : (int32_t *)(ws + h.count_off);
  int32_t *fail_rows = (int32_t *)(ws + h.rows_off);
  cudaStream_t st = (cudaStream_t)stream;

  rc = (arith == SclArith::minsum ? polar_sc_decode_f32 : polar_sc_decode_boxplus_f32)(d_logit, d_frozen_mask, n, B, sc_packed,
                                                                                        d_u_info_f32, d_info_pos, k, stream);
  if (rc != POLAR_OK) return rc;
  POLAR_CUDA(cudaMemsetAsync(count, 0, sizeof(int32_t), st));
  {
    const int rpw = 32 / (POLAR_WORDS(n) < 32 ? POLAR_WORDS(n) : 32);
    const int64_t warps = (B + rpw - 1) / rpw;
    int64_t grid = (warps + 7) / 8;
    const int64_t cap = (int64_t)device_sm_count() * 8;
    if (grid > cap) grid = cap;
    hybrid_crc_check_kernel<<<(unsigned)grid, 256, 0, st>>>(sc_packed, n, B, d_crc_rows, count, fail_rows);
    count_launch();
    POLAR_CHECK_LAUNCH("hybrid_crc_check_kernel");
  }
  return scl_decode(arith, d_logit, d_frozen_mask, n, L, B, d_best_packed, d_u_info_f32, d_info_pos, k, nullptr, nullptr,
                    d_crc_rows, crc_len, ws + h.scl_off, workspace_bytes - h.scl_off, stream, fail_rows, count);
}
