// polar_belief.cu -- belief-propagation (BP) polar decoder with soft output and a fixed number of iterations
// (Sionna's PolarBPDecoder, dec_type="BP" of its Polar5GDecoder).  Compiled twice: with the min-sum f into namespace
// polar (polar::launch_belief) and, through polar_bp_wrap.cu, with the exact boxplus f into namespace polar_bp
// (polar_bp::launch_belief).  The C entry point is polar_belief_decode_f32 (polar_belief_api.cu).
//
// Factor graph: the encoder's butterfly (polar_enc.cu) in natural order, columns 0 (u side) .. m (channel side).  Stage
// s joins columns s and s+1 through the processing elements (PEs) (i, j = i + 2^s), one for every i with bit s clear.
// Lm[s] is the leftward message column, Rm[s] the rightward one: Lm[m] = channel LLR (-logit), Rm[0] = +30 at frozen
// positions and 0 at information positions, every other column starts at 0.  One iteration:
//   right to left, s = m-1 .. 0:  Lm[s][i]   = f(Lm[s+1][i], Lm[s+1][j] + Rm[s][j])
//                                 Lm[s][j]   = f(Rm[s][i], Lm[s+1][i]) + Lm[s+1][j]
//   left to right, s = 0 .. m-2:  Rm[s+1][i] = f(Rm[s][i], Lm[s+1][j] + Rm[s][j])
//                                 Rm[s+1][j] = f(Rm[s][i], Lm[s+1][i]) + Rm[s][j]
// f is the SC decoder's f of the same arithmetic (polar_common.cuh), additions are fp32 and unclipped.  Output: soft
// = -(Lm[0][i] + Rm[0][i]) in the logit convention, hard bit = [soft > 0].  Lm[0] is read by nothing but the output,
// so only the last iteration forms it; the last iteration also skips its left-to-right sweep, and Rm[m] is never
// formed.  None of these skips changes an output.
//
// Mapping: n/2 threads per codeword, thread p runs PE p of every stage; 512/n codewords per CTA of 256 threads below
// n = 1024, one codeword per CTA of 512 threads at n = 1024.  The live state Lm[1..m-1], Rm[1..m-1] sits in shared
// memory: 2(m-1) n floats per codeword, 72 KB at n = 1024 (three codewords per SM).  The channel row Lm[m] is re-read
// from global memory (L1/L2) on every iteration.  At every stage s <= 5 the 32 PEs of a warp touch one 64-position
// block and nothing else, so two consecutive stages that are both <= 5 are ordered by __syncwarp; every other stage
// boundary is a CTA barrier.
#include "polar_common.cuh"
#include "polar_internal.h"
#include "polar_launch.h"
#include "polar_belief.h"

namespace polar {

namespace {

constexpr int kBeliefMaxThreads = 512;

// orders stage s_next after stage s_done (see the mapping above)
__device__ __forceinline__ void stage_barrier(int s_done, int s_next) {
  if (s_done <= 5 && s_next <= 5) __syncwarp(); else __syncthreads();
}

// PE p of stage s: the pair (i, i + 2^s)
__device__ __forceinline__ int pe_low(int p, int s) { return ((p >> s) << (s + 1)) | (p & ((1 << s) - 1)); }

__global__ void __launch_bounds__(kBeliefMaxThreads) belief_kernel(const BeliefParams P) {
  extern __shared__ float smem[];
  const int n = P.n, m = ilog2(n), half = n >> 1;
  const int cpb = blockDim.x / half;
  const int c = threadIdx.x / half, p = threadIdx.x - c * half;
  // per codeword: Lm[s] (s = 1 .. m-1) at base + (s-1) n, then Rm[s] at base + (m-2+s) n.  The soft output of the last
  // iteration goes where Rm[1] was (nothing reads Rm[1] after the last right-to-left stage 1); n = 2 has only that row.
  float *const base = smem + (size_t)c * (m > 1 ? 2 * (m - 1) : 1) * n;
  float *const rm1 = base + (size_t)(m > 1 ? m - 1 : 0) * n;
  const auto Lc = [&](int s) { return base + (size_t)(s - 1) * n; };
  const auto Rc = [&](int s) { return rm1 + (size_t)(s - 1) * n; };

  const uint32_t fw = __ldg(P.fmask + ((2 * p) >> 5)) >> ((2 * p) & 31);       // frozen bits of stage 0's pair
  const float r0i = (fw & 1u) ? kLlrMax : 0.0f, r0j = (fw & 2u) ? kLlrMax : 0.0f;

  for (int64_t b0 = (int64_t)blockIdx.x * cpb; b0 < P.B; b0 += (int64_t)gridDim.x * cpb) {
    const int64_t b = b0 + c;
    const bool valid = b < P.B;
    const float *row = P.logit + (valid ? b : 0) * n;                            // a partial CTA decodes row 0 again
    for (int q = p; q < (m - 1) * n; q += half) rm1[q] = 0.0f;                  // Rm[1 .. m-1] start at 0
    __syncthreads();

    for (int it = 0;; ++it) {
#pragma unroll 1
      for (int s = m - 1; s >= 1; --s) {                                          // right to left; stage 0 below
        const int i = pe_low(p, s), j = i + (1 << s);
        float li, lj;
        if (s == m - 1) { li = -__ldg(row + i); lj = -__ldg(row + j); }
        else { li = Lc(s + 1)[i]; lj = Lc(s + 1)[j]; }
        const float *R = Rc(s);
        const float ri = R[i], rj = R[j];
        float *L = Lc(s);
        L[i] = f_minsum(li, lj + rj);
        L[j] = f_minsum(ri, li) + lj;
        stage_barrier(s, s - 1);
      }
      if (it == P.iters - 1) break;
#pragma unroll 1
      for (int s = 0; s <= m - 2; ++s) {                                          // left to right
        const int i = pe_low(p, s), j = i + (1 << s);
        const float *L = Lc(s + 1);
        const float li = L[i], lj = L[j];
        float ri, rj;
        if (s == 0) { ri = r0i; rj = r0j; }
        else { ri = Rc(s)[i]; rj = Rc(s)[j]; }
        float *R = Rc(s + 1);
        R[i] = f_minsum(ri, lj + rj);
        R[j] = f_minsum(ri, li) + rj;
        stage_barrier(s, s + 1);
      }
    }
    {                                                                             // last iteration, stage 0: the output
      float li, lj;
      if (m == 1) { li = -__ldg(row); lj = -__ldg(row + 1); }
      else { li = Lc(1)[2 * p]; lj = Lc(1)[2 * p + 1]; }
      const float l0i = f_minsum(li, lj + r0j), l0j = f_minsum(r0i, li) + lj;
      rm1[2 * p] = -(l0i + r0i);
      rm1[2 * p + 1] = -(l0j + r0j);
    }
    __syncthreads();
    if (valid) {
      const float *soft = rm1;
      if (P.u_info || P.llr_info)
        for (int t = p; t < P.k; t += half) {
          const float v = soft[__ldg(P.info_pos + t)];
          if (P.llr_info) P.llr_info[b * P.k + t] = v;
          if (P.u_info) P.u_info[b * P.k + t] = v > 0.0f ? 1.0f : 0.0f;
        }
      if (P.u_packed) {
        const int nw = POLAR_WORDS(n), len = n < 32 ? n : 32;
        for (int w = p; w < nw; w += half) {
          uint32_t word = 0;
          for (int q0 = 0; q0 < len; ++q0) {
            const int q = (q0 + w) & (len - 1);                                   // staggered: no bank conflicts
            word |= (uint32_t)(soft[32 * w + q] > 0.0f) << q;
          }
          P.u_packed[b * nw + w] = word & ~__ldg(P.fmask + w);                    // frozen positions are 0
        }
      }
    }
    __syncthreads();                                                              // the next codeword clears Rm[1]
  }
}

}  // namespace

int launch_belief(const BeliefParams &P, cudaStream_t st) {
  const int m = ilog2(P.n), half = P.n / 2;
  const int threads = half > 256 ? half : 256;
  const int cpb = threads / half;
  const size_t smem = (size_t)cpb * (m > 1 ? 2 * (m - 1) : 1) * P.n * sizeof(float);
  int64_t grid = (P.B + cpb - 1) / cpb;
  if (grid > ((int64_t)1 << 30)) grid = (int64_t)1 << 30;                        // the kernel loops over the rest
  POLAR_CUDA(cudaFuncSetAttribute(belief_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return launch("belief_kernel", belief_kernel, (unsigned)grid, threads, smem, st, P);
}

}  // namespace polar
