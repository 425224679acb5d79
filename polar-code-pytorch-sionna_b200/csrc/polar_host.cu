// polar_host.cu -- host-buffer entry points: the end-to-end path a caller with HOST tensors uses
// (SC_Dec.forward / SCL_Dec.forward on a CPU tensor, x_run_sn_polar/polar/polar_sc.py:113-133, polar_scl.py:210-234).
// The batch is cut into chunks; chunk c is copied H2D, decoded and copied back D2H on stream c%2, so the PCIe
// transfers of one chunk overlap the kernel of the other.  Page-locked caller buffers are DMA'd directly; pageable
// ones go through page-locked staging buffers filled / drained by a few host threads while the GPU works on the
// previous chunk.  Device and staging buffers are cached per device (grow-only).  One mutex per device; the caller's
// current device is restored; on an error both streams are drained before returning (no copy stays in flight on a
// caller buffer).
#include <string.h>

#include <mutex>
#include <thread>
#include <vector>

#include "polar_internal.h"
#include "polar_sc.h"
#include "polar_scl.h"

namespace polar {

struct HostCtx {
  std::mutex mu;
  cudaStream_t st[2] = {nullptr, nullptr};
  cudaEvent_t done[2] = {nullptr, nullptr};
  void *logit[2] = {nullptr, nullptr}; size_t logit_bytes = 0;
  void *out[2] = {nullptr, nullptr}; size_t out_bytes = 0;
  void *info[2] = {nullptr, nullptr}; size_t info_bytes = 0;
  void *pm[2] = {nullptr, nullptr}; size_t pm_bytes = 0;
  void *ws[2] = {nullptr, nullptr}; size_t ws_bytes = 0;
  void *mask = nullptr; size_t mask_bytes = 0;
  void *crc = nullptr; size_t crc_bytes = 0;
  void *pos = nullptr; size_t pos_bytes = 0;
  // page-locked staging for pageable caller buffers
  void *h_in[2] = {nullptr, nullptr}; size_t h_in_bytes = 0;
  void *h_out[2] = {nullptr, nullptr}; size_t h_out_bytes = 0;
  void *h_info[2] = {nullptr, nullptr}; size_t h_info_bytes = 0;
};
static HostCtx g_ctx[64];

static int grow(void **p, size_t *have, size_t need) {
  if (*have >= need) return POLAR_OK;
  if (*p) cudaFree(*p);
  *p = nullptr; *have = 0;
  if (cudaMalloc(p, need) != cudaSuccess) { (void)cudaGetLastError(); return set_error(POLAR_ENOMEM, "host path: cudaMalloc(%zu) failed", need); }
  *have = need;
  return POLAR_OK;
}
static int grow2(void *p[2], size_t *have, size_t need) {
  if (*have >= need) return POLAR_OK;
  *have = 0;
  for (int i = 0; i < 2; ++i) {
    if (p[i]) cudaFree(p[i]);
    p[i] = nullptr;
    if (cudaMalloc(&p[i], need) != cudaSuccess) { (void)cudaGetLastError(); return set_error(POLAR_ENOMEM, "host path: cudaMalloc(%zu) failed", need); }
  }
  *have = need;
  return POLAR_OK;
}
static int grow2_pinned(void *p[2], size_t *have, size_t need) {
  if (*have >= need) return POLAR_OK;
  *have = 0;
  for (int i = 0; i < 2; ++i) {
    if (p[i]) cudaFreeHost(p[i]);
    p[i] = nullptr;
    if (cudaHostAlloc(&p[i], need, cudaHostAllocDefault) != cudaSuccess) { (void)cudaGetLastError(); return set_error(POLAR_ENOMEM, "host path: cudaHostAlloc(%zu) failed", need); }
  }
  *have = need;
  return POLAR_OK;
}

static bool is_pinned(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// memcpy on a few host threads (a single core moves ~10 GB/s, a PCIe 5 x16 link ~55 GB/s)
static void par_memcpy(void *dst, const void *src, size_t bytes) {
  int nt = env_int("POLAR_HOST_COPY_THREADS", 4);
  if (nt < 1) nt = 1;
  if (nt > 16) nt = 16;
  if (bytes < ((size_t)4 << 20) || nt == 1) { memcpy(dst, src, bytes); return; }
  const size_t per = ((bytes / nt) + 4095) & ~(size_t)4095;
  std::vector<std::thread> th;
  for (int t = 1; t < nt; ++t) {
    const size_t off = per * t;
    if (off >= bytes) break;
    const size_t len = (off + per < bytes) ? per : bytes - off;
    th.emplace_back([=] { memcpy((char *)dst + off, (const char *)src + off, len); });
  }
  memcpy(dst, src, per < bytes ? per : bytes);
  for (auto &t : th) t.join();
}

// Chunk of the H2D / decode / D2H pipeline.  Page-locked input: 32 MB (the first H2D and the last D2H, which nothing
// overlaps, stay short: 81.7 ms per 4 GiB against 83.4 ms with 128 MB chunks); pageable input goes through the staging
// memcpy, whose threads want the larger pieces (128 MB: 37.8 ms per GiB against 49 ms with 32 MB).
static int64_t chunk_codewords(int n, int64_t B, bool staged) {
  int64_t c = env_int("POLAR_HOST_CHUNK_MB", 0);
  if (c <= 0) c = staged ? 128 : 32;
  c = c * (int64_t)(1 << 20) / ((int64_t)n * 4);
  if (c < 1) c = 1;
  if (c > B) c = B;
  return c;
}

struct DeviceGuard {               // run on `device`, restore the caller's current device on every exit path
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int device) { ok = cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(device) == cudaSuccess; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

struct HostJob {
  // caller buffers
  const float *h_logit; uint32_t *h_packed; float *h_info; double *h_pm;
  int n, k, L; int64_t B;
  bool scl; const uint32_t *crc_dev; int crc_len;
};

// The chunk loop shared by SC and SCL.  C is locked by the caller; `chunk` codewords per chunk.
static int run_chunks(HostCtx &C, const HostJob &J, int64_t chunk, size_t ws_need) {
  const int n = J.n, nw = POLAR_WORDS(n), k = J.k, L = J.L;
  const bool in_staged = !is_pinned(J.h_logit);
  const bool out_staged = J.h_packed && !is_pinned(J.h_packed);
  const bool info_staged = J.h_info && !is_pinned(J.h_info);
  int rc;
  if ((rc = grow2(C.logit, &C.logit_bytes, (size_t)chunk * n * 4))) return rc;
  if ((rc = grow2(C.out, &C.out_bytes, (size_t)chunk * nw * 4))) return rc;
  if (J.h_info && (rc = grow2(C.info, &C.info_bytes, (size_t)chunk * k * 4))) return rc;
  if (J.h_pm && (rc = grow2(C.pm, &C.pm_bytes, (size_t)chunk * L * 8))) return rc;
  if (ws_need && (rc = grow2(C.ws, &C.ws_bytes, ws_need))) return rc;
  if (in_staged && (rc = grow2_pinned(C.h_in, &C.h_in_bytes, (size_t)chunk * n * 4))) return rc;
  if (out_staged && (rc = grow2_pinned(C.h_out, &C.h_out_bytes, (size_t)chunk * nw * 4))) return rc;
  if (info_staged && (rc = grow2_pinned(C.h_info, &C.h_info_bytes, (size_t)chunk * k * 4))) return rc;
  struct Pending { int64_t b0 = 0, nb = 0; bool live = false; } pend[2];
  auto finish = [&](int idx) -> int {            // wait for chunk `idx` and drain its staging buffers into the caller's
    if (!pend[idx].live) return POLAR_OK;
    pend[idx].live = false;
    POLAR_CUDA(cudaEventSynchronize(C.done[idx]));
    const int64_t b0 = pend[idx].b0, nb = pend[idx].nb;
    if (out_staged) par_memcpy(J.h_packed + b0 * nw, C.h_out[idx], (size_t)nb * nw * 4);
    if (info_staged) par_memcpy(J.h_info + b0 * k, C.h_info[idx], (size_t)nb * k * 4);
    return POLAR_OK;
  };
  auto body = [&]() -> int {
    int idx = 0;
    for (int64_t b0 = 0; b0 < J.B; b0 += chunk, idx ^= 1) {
      const int64_t nb = (J.B - b0) < chunk ? (J.B - b0) : chunk;
      cudaStream_t st = C.st[idx];
      int r = finish(idx);                       // chunk c-2 used the same buffers
      if (r) return r;
      const float *src = J.h_logit + b0 * n;
      if (in_staged) { par_memcpy(C.h_in[idx], src, (size_t)nb * n * 4); src = (const float *)C.h_in[idx]; }
      POLAR_CUDA(cudaMemcpyAsync(C.logit[idx], src, (size_t)nb * n * 4, cudaMemcpyHostToDevice, st));
      uint32_t *d_out = J.h_packed ? (uint32_t *)C.out[idx] : nullptr;
      float *d_info = J.h_info ? (float *)C.info[idx] : nullptr;
      if (J.scl)
        r = polar_scl_decode((const float *)C.logit[idx], (const uint32_t *)C.mask, n, L, nb, d_out, d_info,
                             (const int32_t *)C.pos, k, J.h_pm ? (double *)C.pm[idx] : nullptr, nullptr, J.crc_dev, J.crc_len,
                             ws_need ? C.ws[idx] : nullptr, ws_need ? C.ws_bytes : 0, st);
      else
        r = sc_decode(Arith::minsum, (const float *)C.logit[idx], (const uint32_t *)C.mask, n, nb, d_out, d_info,
                      (const int32_t *)C.pos, k, st);
      if (r) return r;
      if (J.h_packed)
        POLAR_CUDA(cudaMemcpyAsync(out_staged ? C.h_out[idx] : (void *)(J.h_packed + b0 * nw), C.out[idx], (size_t)nb * nw * 4,
                                   cudaMemcpyDeviceToHost, st));
      if (J.h_info)
        POLAR_CUDA(cudaMemcpyAsync(info_staged ? C.h_info[idx] : (void *)(J.h_info + b0 * k), C.info[idx], (size_t)nb * k * 4,
                                   cudaMemcpyDeviceToHost, st));
      if (J.h_pm) POLAR_CUDA(cudaMemcpyAsync(J.h_pm + b0 * L, C.pm[idx], (size_t)nb * L * 8, cudaMemcpyDeviceToHost, st));
      POLAR_CUDA(cudaEventRecord(C.done[idx], st));
      pend[idx].b0 = b0; pend[idx].nb = nb; pend[idx].live = true;
    }
    int r = finish(idx);                         // older of the two chunks in flight first
    if (r) return r;
    return finish(idx ^ 1);
  };
  rc = body();
  if (rc) {                                      // drain: nothing may stay in flight on caller buffers after an error
    cudaStreamSynchronize(C.st[0]);
    cudaStreamSynchronize(C.st[1]);
    (void)cudaGetLastError();
  }
  return rc;
}

static int prepare(HostCtx &C, const uint32_t *h_mask, int n, const int32_t *h_info_pos, int k) {
  for (int i = 0; i < 2; ++i) {
    if (!C.st[i]) POLAR_CUDA(cudaStreamCreateWithFlags(&C.st[i], cudaStreamNonBlocking));
    if (!C.done[i]) POLAR_CUDA(cudaEventCreateWithFlags(&C.done[i], cudaEventDisableTiming));
  }
  const int nw = POLAR_WORDS(n);
  int rc;
  if ((rc = grow(&C.mask, &C.mask_bytes, (size_t)nw * 4))) return rc;
  POLAR_CUDA(cudaMemcpyAsync(C.mask, h_mask, (size_t)nw * 4, cudaMemcpyHostToDevice, C.st[0]));
  if (h_info_pos && k > 0) {
    if ((rc = grow(&C.pos, &C.pos_bytes, (size_t)k * 4))) return rc;
    POLAR_CUDA(cudaMemcpyAsync(C.pos, h_info_pos, (size_t)k * 4, cudaMemcpyHostToDevice, C.st[0]));
  }
  return POLAR_OK;
}

}  // namespace polar

using namespace polar;

extern "C" int polar_sc_decode_host_f32(const float *h_logit, const uint32_t *h_frozen_mask, int n, int64_t B,
                                        uint32_t *h_u_packed, float *h_u_info_f32, const int32_t *h_info_pos, int k,
                                        int device) {
  int rc = check_sc_args("sc host", n, B, h_logit, h_frozen_mask, h_u_packed || h_u_info_f32, h_u_info_f32, h_info_pos, k);
  if (rc != POLAR_OK || B == 0) return rc;
  if (h_u_info_f32 && k < 1) return set_error(POLAR_EINVAL, "sc host: u_info requested without valid info_pos/k");
  if (device < 0 || device >= 64) return set_error(POLAR_EINVAL, "sc host: bad device");
  HostCtx &C = g_ctx[device];
  std::lock_guard<std::mutex> lk(C.mu);
  DeviceGuard guard(device);
  if (!guard.ok) return set_error(POLAR_ECUDA, "sc host: cannot select device %d", device);
  rc = polar_init(device);
  if (rc) return rc;
  if ((rc = prepare(C, h_frozen_mask, n, h_u_info_f32 ? h_info_pos : nullptr, k))) return rc;
  POLAR_CUDA(cudaStreamSynchronize(C.st[0]));
  HostJob J{h_logit, h_u_packed, h_u_info_f32, nullptr, n, h_u_info_f32 ? k : 0, 0, B, false, nullptr, 0};
  return run_chunks(C, J, chunk_codewords(n, B, !is_pinned(h_logit)), 0);
}

extern "C" int polar_sc_decode_host(const float *h_logit, const uint32_t *h_frozen_mask, int n, int64_t B,
                                    uint32_t *h_u_packed, int device) {
  if (B != 0 && !h_u_packed) return set_error(POLAR_EINVAL, "sc host: null pointer");
  return polar_sc_decode_host_f32(h_logit, h_frozen_mask, n, B, h_u_packed, nullptr, nullptr, 0, device);
}

extern "C" int polar_scl_decode_host_f32(const float *h_logit, const uint32_t *h_frozen_mask, int n, int L, int64_t B,
                                         uint32_t *h_best_packed, float *h_u_info_f32, const int32_t *h_info_pos, int k,
                                         double *h_pm_sorted, const uint32_t *h_crc_rows, int crc_len, int device) {
  int rc = check_scl_shape("scl host", n, L, B);
  if (rc != POLAR_OK || B == 0) return rc;
  if (!h_logit || !h_frozen_mask || (!h_best_packed && !h_u_info_f32)) return set_error(POLAR_EINVAL, "scl host: null pointer");
  if (h_u_info_f32 && (!h_info_pos || k < 1 || k > n)) return set_error(POLAR_EINVAL, "scl host: u_info requested without valid info_pos/k");
  if (device < 0 || device >= 64) return set_error(POLAR_EINVAL, "scl host: bad device");
  HostCtx &C = g_ctx[device];
  std::lock_guard<std::mutex> lk(C.mu);
  DeviceGuard guard(device);
  if (!guard.ok) return set_error(POLAR_ECUDA, "scl host: cannot select device %d", device);
  rc = polar_init(device);
  if (rc) return rc;
  int64_t chunk = chunk_codewords(n, B, true);        // the list decoder's time per chunk is not hidden by the copy: large chunks
  const SclPlan whole = scl_plan(n, L, B, Arith::minsum, true);   // the chunk buffers are cudaMalloc'd: aligned rows
  if (whole.scl3 && chunk < B) {
    // the list kernel is persistent: every resident warp decodes the same number of 32/L-codeword groups, so a chunk
    // should be a whole number of such rounds (a 128 MB chunk of n = 1024 is 3.46 rounds: 13 % of the last one idle)
    const int64_t round = whole.grid * (32 / L);
    if (chunk > round) chunk = chunk / round * round;
  }
  const size_t ws_need = scl_plan(n, L, chunk, Arith::minsum, true).ws_bytes;
  if ((rc = prepare(C, h_frozen_mask, n, h_u_info_f32 ? h_info_pos : nullptr, k))) return rc;
  const bool crc = crc_len > 0 && h_crc_rows;
  if (crc) {
    if ((rc = grow(&C.crc, &C.crc_bytes, (size_t)n * 4))) return rc;
    POLAR_CUDA(cudaMemcpyAsync(C.crc, h_crc_rows, (size_t)n * 4, cudaMemcpyHostToDevice, C.st[0]));
  }
  POLAR_CUDA(cudaStreamSynchronize(C.st[0]));
  // k scales the CRC penalty (30 k, dec.py:517-518) even when no [B, k] tensor is requested: derive it from the mask then
  int k_eff = k;
  if (k_eff <= 0) {
    k_eff = n;
    for (int w = 0; w < POLAR_WORDS(n); ++w) k_eff -= __builtin_popcount(n < 32 ? (h_frozen_mask[w] & ((1u << n) - 1u)) : h_frozen_mask[w]);
  }
  HostJob J{h_logit, h_best_packed, h_u_info_f32, h_pm_sorted, n, k_eff, L, B, true,
            crc ? (const uint32_t *)C.crc : nullptr, crc ? crc_len : 0};
  return run_chunks(C, J, chunk, ws_need);
}

extern "C" int polar_scl_decode_host(const float *h_logit, const uint32_t *h_frozen_mask, int n, int L, int64_t B,
                                     uint32_t *h_best_packed, double *h_pm_sorted, const uint32_t *h_crc_rows,
                                     int crc_len, int device) {
  if (B != 0 && !h_best_packed) return set_error(POLAR_EINVAL, "scl host: null pointer");
  return polar_scl_decode_host_f32(h_logit, h_frozen_mask, n, L, B, h_best_packed, nullptr, nullptr, 0, h_pm_sorted, h_crc_rows,
                                   crc_len, device);
}
