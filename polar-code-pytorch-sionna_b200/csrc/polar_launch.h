// polar_launch.h -- host-side vocabulary of the C entry points: the arithmetic a decoder runs in, the shape check of a
// code length, and how a kernel's grid is sized and the kernel launched.  Kept apart from polar_internal.h, whose bytes
// stamp the profiler captures (bench.py KERNEL_SOURCES), so that host-side changes here leave the stamp alone.
#pragma once
#include "polar_internal.h"

namespace polar {

// Check-node arithmetic of a decode.  The values are the cn_mode of polar_scl_decode_hybrid.  Min-sum kernels live in
// namespace polar, the exact-boxplus builds of the same sources in namespace polar_bp (polar_bp_wrap.cu).
enum class Arith { minsum = 0, boxplus = 1, boxplus_pruned = 2 };

// n must be a power of two in [lo, hi]
inline int check_pow2_n(const char *who, int n, int lo, int hi) {
  if (!is_pow2(n) || n < lo || n > hi) return set_error(POLAR_EINVAL, "%s: n=%d must be a power of two in [%d,%d]", who, n, lo, hi);
  return POLAR_OK;
}

// ceil(work / per_cta) CTAs, at least one and at most ctas_per_sm per SM (grid-stride kernels loop over the rest)
inline unsigned grid_for(int64_t work, int per_cta, int ctas_per_sm) {
  int64_t g = (work + per_cta - 1) / per_cta;
  const int64_t cap = (int64_t)device_sm_count() * ctas_per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (unsigned)g;
}

// CTAs of `kernel` resident on one SM at `threads` threads and `smem` bytes of dynamic shared memory; 4 if the query fails
template <class K>
int resident_ctas(K kernel, int threads, size_t smem) {
  int r = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&r, kernel, threads, smem) != cudaSuccess || r <= 0) {
    (void)cudaGetLastError();
    r = 4;
  }
  return r;
}

// kernel<<<grid, block, smem, st>>>(args...), counted in polar_launch_count(); a launch error returns POLAR_ECUDA with the
// text "<what>: <CUDA error>"
template <class... P, class... A>
int launch(const char *what, void (*kernel)(P...), unsigned grid, int block, size_t smem, cudaStream_t st, A... args) {
  kernel<<<grid, block, smem, st>>>(args...);
  count_launch();
  POLAR_CHECK_LAUNCH(what);
  return POLAR_OK;
}

}  // namespace polar
