// polar_sc.cu -- SC decoder kernels for the short codes, n <= 64: one thread per codeword, the whole tree in registers
// (fp32 min-sum, bit-exact with the reference; exact boxplus in the polar_bp build, polar_bp_wrap.cu).
//
// Replaces x_run_sn_polar/polar/polar_sc.py:54-133 (recursion, f/g, leaf rule, partial sums, info gather).
// Semantics: SURVEY.md Appendix A.  The entry points and the choice of mapping by code length are in polar_sc_api.cu;
// the longer codes run on polar_sc4.cu (128 <= n <= 512) and polar_sc5.cu (n >= 1024).
// Rate-0 nodes (all frozen) are skipped and rate-1 subtrees take the hard-decision shortcut when no LLR is exactly 0 (both
// exact, see polar_common.cuh).
#include "polar_common.cuh"
#include "polar_internal.h"
#include "polar_sc.h"

namespace polar {

// ------------------------------------------------------------------ n <= 64: thread per codeword
template <int T>
__global__ void __launch_bounds__(128) sc_small_kernel(const float *__restrict__ logit,
                                                       const uint32_t *__restrict__ fmask, int64_t B,
                                                       uint32_t *__restrict__ u_packed,
                                                       float *__restrict__ u_info,
                                                       const int32_t *__restrict__ info_pos, int k) {
  constexpr int N = 1 << T;
  const uint32_t fm = __ldg(fmask);
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
    float x[N];
    const float *row = logit + b * N;
    if (N >= 4) {
#pragma unroll
      for (int q = 0; q < N / 4; ++q) {
        float4 v = __ldg(reinterpret_cast<const float4 *>(row) + q);
        x[4 * q + 0] = -v.x; x[4 * q + 1] = -v.y; x[4 * q + 2] = -v.z; x[4 * q + 3] = -v.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < N; ++j) x[j] = -__ldg(row + j);
    }
    uint32_t u;
    SubTree<T>::run(x, fm, u);
    if (u_packed) u_packed[b] = u;
    if (u_info)
      for (int t = 0; t < k; ++t) u_info[b * k + t] = (float)((u >> __ldg(info_pos + t)) & 1u);
  }
}

// n = 64: the two 32-leaf halves one after the other (f -> left subtree -> g -> right subtree, polar_sc.py:54-98); the
// decisions come straight out of the register subtrees (RollTree returns u next to the partial sums).
__global__ void __launch_bounds__(128) sc64_kernel(const float *__restrict__ logit, const uint32_t *__restrict__ fmask, int64_t B,
                                                   uint32_t *__restrict__ u_packed, float *__restrict__ u_info,
                                                   const int32_t *__restrict__ info_pos, int k) {
  const uint32_t fm0 = __ldg(fmask), fm1 = __ldg(fmask + 1);
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
    const float4 *row = reinterpret_cast<const float4 *>(logit + b * 64);
    float y[32];
    uint32_t u0 = 0, u1 = 0, bl = 0;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {                       // rolled: one copy of the 32-leaf subtree code
      const uint32_t fmc = h ? fm1 : fm0;
      if (fmc == 0xFFFFFFFFu) continue;                 // rate-0 half: decisions and partial sums are 0
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 a = __ldg(row + q), c = __ldg(row + 8 + q);        // logits: LLR = -logit (polar_sc.py:122)
        const float xa[4] = {-a.x, -a.y, -a.z, -a.w}, xc[4] = {-c.x, -c.y, -c.z, -c.w};
#pragma unroll
        for (int e = 0; e < 4; ++e)
          y[4 * q + e] = h ? g_minsum(xa[e], xc[e], (bl << (31 - (4 * q + e))) & 0x80000000u) : f_minsum(xa[e], xc[e]);
      }
      uint32_t u;
      const uint32_t beta = RollTree<5>::run(y, fmc, u);
      if (h == 0) { bl = beta; u0 = u; } else { u1 = u; }
    }
    if (u_packed) { u_packed[2 * b] = u0; u_packed[2 * b + 1] = u1; }
    if (u_info)
      for (int t = 0; t < k; ++t) {
        const int p = __ldg(info_pos + t);
        u_info[b * k + t] = (float)(((p < 32 ? u0 : u1) >> (p & 31)) & 1u);
      }
  }
}

int launch_sc_small(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
                    const int32_t *info_pos, int k, cudaStream_t st) {
  const unsigned grid = grid_for(B, 128, 16);
  if (n == 64) return launch("sc64_kernel", sc64_kernel, grid, 128, 0, st, logit, fmask, B, u_packed, u_info, info_pos, k);
  const auto kern = n == 2 ? sc_small_kernel<1> : n == 4 ? sc_small_kernel<2> : n == 8 ? sc_small_kernel<3>
                    : n == 16 ? sc_small_kernel<4> : sc_small_kernel<5>;
  return launch("sc_small_kernel", kern, grid, 128, 0, st, logit, fmask, B, u_packed, u_info, info_pos, k);
}

}  // namespace polar
