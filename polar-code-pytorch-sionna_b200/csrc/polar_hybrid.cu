// polar_hybrid.cu -- hybrid SC -> SCL decoding with CRC-aided selection (the `use_hybrid_sc` mode of the Sionna-style
// SCL_Dec, my_sn/fec/polar/dec.py:437-470): decode the whole batch with SC, keep every SC decision whose CRC holds, and
// list-decode only the rows whose CRC fails.  At a working Eb/N0 almost every SC decision passes, so the batch costs
// about one SC decode plus a partial wave of the list kernel instead of a full list decode.
//
// Four stream-ordered operations, no host synchronisation:
//   1. polar_sc_decode_f32 / polar_sc_decode_boxplus_f32 over all B rows -> packed decisions and u_info
//   2. memset of the failing-row count
//   3. hybrid_crc_check_kernel: syndrome of each packed row, indices of the failing rows appended to fail_rows[]
//   4. scl2_kernel<L> (polar_scl.cu, min-sum or boxplus build) over fail_rows[0 .. count-1], overwriting those rows
// The list stage is the generic scl2 mapping in every arithmetic: its decisions equal scl3's bit for bit, and in the
// regime the hybrid is for it decodes a small fraction of the batch.
#include "polar_hybrid.h"
#include "polar_internal.h"

namespace polar {

namespace {

constexpr unsigned kFull = 0xFFFFFFFFu;

inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Workspace layout, every region 256-byte aligned:
//   [0]          packed SC decisions [B, POLAR_WORDS(n)] uint32 (used when the caller passes no d_best_packed)
//   [count_off]  failing-row count, int32 (used when the caller passes no d_n_list_out)
//   [rows_off]   failing-row indices [B] int32
//   [scl_off]    scl2_kernel<L> workspace planned for B rows
struct HybridLayout { size_t count_off, rows_off, scl_off, total; };

HybridLayout hybrid_layout(int n, int L, int64_t B, int cn_mode) {
  HybridLayout h;
  h.count_off = align256((size_t)B * POLAR_WORDS(n) * sizeof(uint32_t));
  h.rows_off = h.count_off + 256;
  h.scl_off = h.rows_off + align256((size_t)B * sizeof(int32_t));
  const size_t scl = cn_mode == 0 ? polar::scl2_rows_workspace_bytes(n, L, B) : polar_bp::scl2_rows_workspace_bytes(n, L, B);
  h.total = h.scl_off + align256(scl);
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

extern "C" size_t polar_scl_hybrid_workspace_bytes(int n, int L, int64_t B, int cn_mode) {
  if (!is_pow2(n) || n < 2 || n > POLAR_SCL_MAX_N || !is_pow2(L) || L > POLAR_SCL_MAX_L || B <= 0 || B > INT32_MAX ||
      cn_mode < 0 || cn_mode > 2)
    return 0;
  return hybrid_layout(n, L, B, cn_mode).total;
}

extern "C" int polar_scl_decode_hybrid(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                                       uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                                       const uint32_t *d_crc_rows, int crc_len, int cn_mode, int32_t *d_n_list_out,
                                       void *d_workspace, size_t workspace_bytes, void *stream) {
  if (!is_pow2(n) || n < 2 || n > POLAR_SCL_MAX_N) return set_error(POLAR_EINVAL, "hybrid: n=%d must be a power of two in [2,%d]", n, POLAR_SCL_MAX_N);
  if (!is_pow2(L) || L > POLAR_SCL_MAX_L) return set_error(POLAR_EINVAL, "hybrid: list_size=%d must be a power of two <= %d", L, POLAR_SCL_MAX_L);
  if (cn_mode < 0 || cn_mode > 2) return set_error(POLAR_EINVAL, "hybrid: cn_mode=%d must be 0 (min-sum), 1 (boxplus) or 2 (boxplus pruned)", cn_mode);
  if (crc_len < 1 || crc_len > 32 || !d_crc_rows) return set_error(POLAR_EINVAL, "hybrid: needs a CRC (crc_len in [1,32] and crc_rows), got crc_len=%d", crc_len);
  if (k < 1 || k > n) return set_error(POLAR_EINVAL, "hybrid: k=%d must be in [1,%d]", k, n);
  if (B < 0 || B > INT32_MAX) return set_error(POLAR_EINVAL, "hybrid: B=%lld must be in [0, 2^31)", (long long)B);
  if (B == 0) return POLAR_OK;
  if (!d_logit || !d_frozen_mask) return set_error(POLAR_EINVAL, "hybrid: null logit / frozen_mask");
  if (!d_best_packed && !d_u_info_f32) return set_error(POLAR_EINVAL, "hybrid: no output buffer");
  if (d_u_info_f32 && !d_info_pos) return set_error(POLAR_EINVAL, "hybrid: u_info requested without info_pos");
  const HybridLayout h = hybrid_layout(n, L, B, cn_mode);
  if (!d_workspace || workspace_bytes < h.total) return set_error(POLAR_ENOMEM, "hybrid: workspace %zu B < required %zu B", d_workspace ? workspace_bytes : (size_t)0, h.total);
  if ((uintptr_t)d_workspace & 255) return set_error(POLAR_EALIGN, "hybrid: workspace must be 256-byte aligned");

  unsigned char *ws = (unsigned char *)d_workspace;
  uint32_t *sc_packed = d_best_packed ? d_best_packed : (uint32_t *)ws;
  int32_t *count = d_n_list_out ? d_n_list_out : (int32_t *)(ws + h.count_off);
  int32_t *fail_rows = (int32_t *)(ws + h.rows_off);
  cudaStream_t st = (cudaStream_t)stream;

  int rc = (cn_mode == 0 ? polar_sc_decode_f32 : polar_sc_decode_boxplus_f32)(d_logit, d_frozen_mask, n, B, sc_packed, d_u_info_f32,
                                                                               d_info_pos, k, stream);
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
  void *scl_ws = ws + h.scl_off;
  if (cn_mode == 0)
    return polar::launch_scl2_rows(d_logit, d_frozen_mask, n, L, B, fail_rows, count, d_best_packed, d_u_info_f32, d_info_pos, k,
                                   d_crc_rows, crc_len, scl_ws, 0, st);
  return polar_bp::launch_scl2_rows(d_logit, d_frozen_mask, n, L, B, fail_rows, count, d_best_packed, d_u_info_f32, d_info_pos, k,
                                    d_crc_rows, crc_len, scl_ws, cn_mode == 2, st);
}
