// polar_scl.cu -- SCL decoder (list size L = 1..32) for sm_100a, optional CRC-aided selection.
//
// Replaces x_run_sn_polar/polar/polar_scl.py:49-234 (2L decoder slots, full-tree copy per info bit)
// and my_sn/fec/polar/dec.py:507-527 (CRC-aided candidate selection).  Semantics: SURVEY.md Appendix A,
// L-survivor formulation (A9): pm = [0,30,..,30]; frozen leaf pm += log(1+exp(-x)); info leaf: fork,
// sort the 2L candidates ascending, keep L.  Arithmetic is fp64 like the reference (numpy float64):
// min-sum f with +-30 clip, g = (1-2u)a+b, exact softplus path metric.
//
// This file: the GENERIC list kernel scl2_kernel<L> and its launcher (lane = (codeword, path): a warp
// decodes 32/L codewords, every lane walks all elements of its own path's nodes; nothing is copied on a fork -- a stage is
// always rewritten by every path at the same time, so a path writes its own slot and a fork only permutes packed pointer
// rows with a warp shuffle; decisions are recovered at the end from the root partial sums; the 2L candidates are ranked by
// a bitonic network on (pm, index)).  It serves what the default mapping does not: n < 64 or n > 4096, L = 1, rows that
// are not 16-byte aligned, and the exact-boxplus variant.  The default is polar_scl3.cu (virtual top stages, compile-time
// tree, counting rank); both return identical bits (tests/test_gpu_parity.py).
#include <math.h>

#include "polar_internal.h"
#include "polar_scl.h"
#include "polar_warp.cuh"

namespace polar {

constexpr double kLlrMaxD = 30.0;

#if defined(POLAR_F_BOXPLUS)
// exact boxplus of the Sionna-style list decoder (my_sn/fec/polar/dec.py:331-340, numpy float64): clip to +-30,
// ln(1+e^(x+y)) - ln(e^x+e^y).  Selected by polar_bp_wrap.cu (namespace polar_bp, launcher launch_scl2_boxplus).
__device__ __forceinline__ double f_minsum_d(double a, double b) {
  const double x = fmax(fmin(a, 30.0), -30.0), y = fmax(fmin(b, 30.0), -30.0);
  return log(1.0 + exp(x + y)) - log(exp(x) + exp(y));
}
#else
__device__ __forceinline__ double f_minsum_d(double a, double b) {   // polar_scl.py:93-106
  const double mag = fmin(fmin(fabs(a), fabs(b)), kLlrMaxD);
  const unsigned long long sgn = (unsigned long long)(__double_as_longlong(a) ^ __double_as_longlong(b)) & 0x8000000000000000ull;
  return __longlong_as_double((long long)((unsigned long long)__double_as_longlong(mag) | sgn));
}
#endif
__device__ __forceinline__ double g_minsum_d(double a, double b, unsigned u) {   // polar_scl.py:107-108
  const unsigned long long sm = (unsigned long long)(u & 1u) << 63;
  return __longlong_as_double((long long)((unsigned long long)__double_as_longlong(a) ^ sm)) + b;
}
// polar_scl.py:81-83 with u_hat: log(1 + exp(-(1-2u).clip(x)))
__device__ __forceinline__ double pm_penalty(double x_clipped, unsigned u) {
  const double v = u ? x_clipped : -x_clipped;
  return log(1.0 + exp(v));
}

// =====================================================================================================
// scl2_kernel: lane = (codeword, path).  A warp decodes 32/L codewords at once, every lane owns one path of
// one codeword and walks ALL elements of its nodes itself.  Same lazy-copy bookkeeping as scl_kernel above
// (per-stage slot pointers packed 5 bits per stage; slots are now the 32 lanes, a path only ever points at
// slots of its own codeword group), but no lane is idle on the narrow stages and at the leaves, which is where
// the one-codeword-per-warp mapping spent most of its issue slots (ncu: 518 warp instructions per leaf, 72 %
// issue utilisation -> the kernel was instruction bound).  Per-stage arrays are [element][32 lanes] doubles:
// a warp access touches 32 consecutive doubles, conflict free.
// =====================================================================================================
#ifndef SCL2_MINB
#define SCL2_MINB 8   // 64 registers per thread: occupancy (latency hiding of the workspace traffic) beats registers
#endif
template <int L>
__global__ void __launch_bounds__(128, SCL2_MINB) scl2_kernel(const SclParams P) {
  constexpr int CPW = 32 / L;                                   // codewords per warp
  constexpr int LOGL = (L == 1) ? 0 : (L == 2) ? 1 : (L == 4) ? 2 : (L == 8) ? 3 : (L == 16) ? 4 : 5;
  constexpr unsigned FULL = 0xFFFFFFFFu;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int p = lane & (L - 1), gbase = lane & ~(L - 1), cwl = lane >> LOGL;
  const int n = P.n, m = P.m, nw = n < 32 ? 1 : n >> 5;
  const int s_glob = P.s_glob;

  unsigned char *base = smem_raw + (size_t)warp * P.smem_per_warp;
  double *llr_s = reinterpret_cast<double *>(base);
  const int64_t gwarp = (int64_t)blockIdx.x * nwarps + warp;
  double *llr_g = P.ws ? P.ws + (size_t)gwarp * P.ws_doubles_per_warp : nullptr;
  const unsigned g_off = 32u * ((1u << s_glob) - 1u);
  // partial-sum words: stage s>=5 at (2^(s-5)-1)*32, then the root region [nw][32].  They are touched once per
  // 32 leaves, so by default they live in the global workspace and shared memory only holds the hot low LLR stages.
  uint32_t *bl = P.words_global ? reinterpret_cast<uint32_t *>(llr_g + (size_t)32 * ((1u << m) - (1u << s_glob)))
                                : reinterpret_cast<uint32_t *>(llr_s + scl2_llr_smem_doubles(s_glob));
  uint32_t *rootw = bl + (size_t)32 * nw;                                                // [nw][32]

  auto stage_ptr = [&](int s) -> double * {   // array [2^s elements][32 slots] of LLR stage s (< m)
    const unsigned off = 32u * ((1u << s) - 1u);
    return (s < s_glob) ? (llr_s + off) : (llr_g + (off - g_off));
  };
  const unsigned long long idrow = (unsigned long long)p * 0x0084210842108421ull;   // field s (5 bits) = p, s = 0..11
  // number of codewords and the row of codeword j; re-read from memory where needed rather than kept live across the
  // leaf loop, which runs at the 64-register cap
  auto n_codewords = [&]() -> int64_t {
    if (!P.rows) return P.B;
    const int64_t c = *P.n_rows;                                 // written by the previous kernel on the stream
    return c < 0 ? 0 : (c < P.B ? c : P.B);
  };
  auto row_of = [&](int64_t j) -> int64_t { return P.rows ? (int64_t)P.rows[j] : j; };

  for (int64_t bb = gwarp; bb < (n_codewords() + CPW - 1) / CPW; bb += (int64_t)gridDim.x * nwarps) {
    const float *ch;
    {
      const int64_t nb = n_codewords(), j = bb * CPW + cwl;
      ch = P.logit + row_of(j < nb ? j : nb - 1) * (int64_t)n;   // idle lanes of the last group redo a real codeword
    }
    double pm = (p == 0) ? 0.0 : kLlrMaxD;                       // polar_scl.py:192-194
    unsigned long long rowL = idrow, rowB = idrow;
    uint32_t small = 0u, rootreg = 0u, fword = 0u;

    for (int i = 0; i < n;) {
      if ((i & 31) == 0) fword = __ldg(P.fmask + (i >> 5));
      // Fast-SCL node shortcuts of the Sionna-style decoder (my_sn/fec/polar/dec.py:269-306, 354-376, use_fast_scl=True):
      // a rate-0 node (all leaves frozen) or a REP node (only the last leaf carries information) of 2^s0 leaves is not
      // descended into; its path-metric update is taken from the node's own stage-s0 LLRs.  Exact under the boxplus f
      // (SURVEY App. C) -- and only there, so the min-sum build never prunes.  Nodes up to 32 leaves (one mask word).
      int sn = 0;                                               // stage of the pruned node (0: plain leaf)
      bool rep = false;
#if defined(POLAR_F_BOXPLUS)
      if (P.fast) {
        const int tmax = (i == 0) ? (m < 5 ? m : 5) : ((__ffs(i) - 1) < 5 ? (__ffs(i) - 1) : 5);
        for (int s = tmax; s >= 1; --s) {
          const uint32_t wbits = 1u << s;
          const uint32_t full = (wbits == 32u) ? 0xFFFFFFFFu : ((1u << wbits) - 1u);
          const uint32_t fm = (fword >> (i & 31)) & full;
          if (fm == full) { sn = s; break; }
          if (fm == (full >> 1)) { sn = s; rep = true; break; }
        }
      }
#endif
      // ------------------------------------------------------------------ descent to leaf i (to the node (s0, i) when pruning)
      int t;
      if (i == 0) {
        t = m;
      } else {
        t = __ffs(i) - 1;
        // g step: stage t+1 -> t, beta = left sibling's partial sums (polar_scl.py:140-144)
        const int h = 1 << t;
        double *dst = stage_ptr(t) + lane;
        if (t < 5) {
          const uint32_t ub = small >> ((1u << t) - 1u);
          if (t + 1 == m) {
            for (int e = 0; e < h; ++e)
              dst[e * 32] = g_minsum_d((double)(-__ldg(ch + e)), (double)(-__ldg(ch + e + h)), (ub >> e) & 1u);
          } else {
            const double *src = stage_ptr(t + 1) + gbase + (unsigned)((rowL >> (5 * (t + 1))) & 31u);
#pragma unroll 4
            for (int e = 0; e < h; ++e) dst[e * 32] = g_minsum_d(src[e * 32], src[(e + h) * 32], (ub >> e) & 1u);
          }
        } else {
          const uint32_t *bw = bl + (size_t)((1u << (t - 5)) - 1u) * 32 + gbase + (unsigned)((rowB >> (5 * t)) & 31u);
          if (t + 1 == m) {
            for (int w = 0; w < (h >> 5); ++w) {
              const uint32_t ub = bw[w * 32];
#pragma unroll 4
              for (int e = 0; e < 32; ++e) {
                const int ee = w * 32 + e;
                dst[ee * 32] = g_minsum_d((double)(-__ldg(ch + ee)), (double)(-__ldg(ch + ee + h)), (ub >> e) & 1u);
              }
            }
          } else {
            const double *src = stage_ptr(t + 1) + gbase + (unsigned)((rowL >> (5 * (t + 1))) & 31u);
            for (int w = 0; w < (h >> 5); ++w) {
              const uint32_t ub = bw[w * 32];
#pragma unroll 4
              for (int e = 0; e < 32; ++e) {
                const int ee = w * 32 + e;
                dst[ee * 32] = g_minsum_d(src[ee * 32], src[(ee + h) * 32], (ub >> e) & 1u);
              }
            }
          }
        }
      }
      // f steps: stage s -> s-1 along left children (polar_scl.py:134-137); inputs are this path's own slot
      // (lane-private data from here on: no synchronisation needed)
      for (int s = (t < m ? t : m); s >= sn + 1; --s) {
        const int h = 1 << (s - 1);
        double *dst = stage_ptr(s - 1) + lane;
        if (s == m) {
          for (int e = 0; e < h; ++e) dst[e * 32] = f_minsum_d((double)(-__ldg(ch + e)), (double)(-__ldg(ch + e + h)));
        } else {
          const double *src = stage_ptr(s) + lane;
#pragma unroll 4
          for (int e = 0; e < h; ++e) dst[e * 32] = f_minsum_d(src[e * 32], src[(e + h) * 32]);
        }
      }
      {  // stages sn..min(t, m-1) were rewritten by this path into its own slot
        const int top = (t < m ? t : m - 1);
        unsigned long long msk = (top >= 11) ? 0x0FFFFFFFFFFFFFFFull : ((1ull << (5 * (top + 1))) - 1ull);
        if (sn > 0) msk &= ~((1ull << (5 * sn)) - 1ull);
        rowL = (rowL & ~msk) | (idrow & msk);
      }
      // ------------------------------------------------------------------ leaf (or pruned node)
      unsigned bit = 0u;
      bool fork = false;
      double k0, k1;
      if (sn > 0) {
        // dec.py:269-280 (rate-0): pm += sum_j log(1+exp(-llr_j)); dec.py:281-306 (REP): the same sum for the u = 0
        // branch, the sum with the LLR signs flipped for the u = 1 branch, then sort and keep L
        const double *node = stage_ptr(sn) + lane;
        double a0 = 0.0, a1 = 0.0;
        for (int e = 0; e < (1 << sn); ++e) {
          const double xe = fmax(fmin(node[e * 32], kLlrMaxD), -kLlrMaxD);
          a0 += pm_penalty(xe, 0u);
          if (rep) a1 += pm_penalty(xe, 1u);
        }
        if (rep) { fork = true; k0 = pm + a0; k1 = pm + a1; }
        else pm += a0;
      } else {
        double x = stage_ptr(0)[lane];
        x = fmax(fmin(x, kLlrMaxD), -kLlrMaxD);                  // polar_scl.py:81
        if ((fword >> (i & 31)) & 1u) {
          pm += pm_penalty(x, 0u);                                 // frozen: u = 0
        } else {
          fork = true; k0 = pm + pm_penalty(x, 0u); k1 = pm + pm_penalty(x, 1u);
        }
      }
      if (fork) {
        // fork: candidate E = u*L + p  (reference slot order [u=0 paths | u=1 paths], polar_scl.py:49-68);
        // two candidates per lane, bitonic sort of the 2L candidates of each codeword inside its lane group
        int s0 = p, s1 = L + p;
#pragma unroll
        for (int k = 2; k <= 2 * L; k <<= 1) {
#pragma unroll
          for (int d = k >> 1; d > 0; d >>= 1) {
            if (d == L) {   // partner is the other register; k == 2L: ascending
              const bool less10 = (k1 < k0) || (k1 == k0 && s1 < s0);
              if (less10) { const double tk = k0; k0 = k1; k1 = tk; const int ts = s0; s0 = s1; s1 = ts; }
            } else {
              const double pk0 = __shfl_xor_sync(FULL, k0, d), pk1 = __shfl_xor_sync(FULL, k1, d);
              const int ps0 = __shfl_xor_sync(FULL, s0, d), ps1 = __shfl_xor_sync(FULL, s1, d);
              const bool lower = ((p & d) == 0);
              const bool up0 = (k == 2 * L) ? true : (k == L) ? true : ((p & k) == 0);
              const bool up1 = (k == 2 * L) ? true : (k == L) ? false : ((p & k) == 0);
              const bool less0 = (pk0 < k0) || (pk0 == k0 && ps0 < s0);
              const bool less1 = (pk1 < k1) || (pk1 == k1 && ps1 < s1);
              if ((lower == up0) == less0) { k0 = pk0; s0 = ps0; }
              if ((lower == up1) == less1) { k1 = pk1; s1 = ps1; }
            }
          }
        }
        const int parent = gbase + (s0 & (L - 1));
        bit = (unsigned)(s0 >> LOGL) & 1u;
        pm = k0;
        rowL = __shfl_sync(FULL, rowL, parent);
        rowB = __shfl_sync(FULL, rowB, parent);
        small = __shfl_sync(FULL, small, parent);
      }
      __syncwarp();   // forked paths read their parents' slots from here on
      // ------------------------------------------------------------------ partial-sum cascade
      // z = number of completed right children above the node that just finished -- leaf i, or the pruned node of 2^sn
      // leaves whose partial sums are all `bit` (rate-0: 0; REP: x_hat = u.(1,...,1))  (polar_scl.py:147-153, [bl ^ br, br])
      const int iend = i + (1 << sn) - 1;
      const int z = (iend == n - 1) ? m : (__ffs(~iend) - 1);
      uint32_t cur = (sn == 0) ? bit : (bit ? ((sn == 5) ? 0xFFFFFFFFu : ((1u << (1u << sn)) - 1u)) : 0u);
      const int zs = z < 5 ? z : 5;
      for (int s = sn; s < zs; ++s) {
        const uint32_t w = 1u << s;
        const uint32_t field = (small >> (w - 1u)) & ((1u << w) - 1u);
        cur = (field ^ cur) | (cur << w);
      }
      if (z < 5) {
        if (z < m) {
          const uint32_t w = 1u << z, off = w - 1u, msk = ((1u << w) - 1u) << off;
          small = (small & ~msk) | (cur << off);
        } else {
          rootreg = cur;                                           // n < 32: whole codeword
        }
      } else {
        const int nwz = 1 << (z - 5);
        uint32_t *dest = ((z < m) ? (bl + (size_t)(nwz - 1) * 32) : rootw) + lane;
        dest[(nwz - 1) * 32] = cur;
        for (int s = 5; s < z; ++s) {
          const int hw = 1 << (s - 5);
          const uint32_t *bls = bl + (size_t)(hw - 1) * 32 + gbase + (unsigned)((rowB >> (5 * s)) & 31u);
          for (int w = 0; w < hw; ++w) dest[(nwz - 2 * hw + w) * 32] = bls[w * 32] ^ dest[(nwz - hw + w) * 32];
        }
        if (z < m) rowB = (rowB & ~(31ull << (5 * z))) | ((unsigned long long)p << (5 * z));
        __syncwarp();
      }
      i = iend + 1;
    }  // leaves

    // ---------------------------------------------------------------------- epilogue
    // root partial sums = codeword estimate x_hat; u_hat = T(x_hat) (involution); lane-private words
    if (m < 5) {
      rootw[lane] = ptransform_rt(rootreg, m);
    } else {
      for (int w = 0; w < nw; ++w) rootw[w * 32 + lane] = ptransform_rt(rootw[w * 32 + lane], 5);
      for (int d = 1; d < nw; d <<= 1)
        for (int w = 0; w < nw; ++w)
          if (!(w & d)) rootw[w * 32 + lane] ^= rootw[(w + d) * 32 + lane];
    }
    __syncwarp();
    // final sort by path metric inside each codeword group (polar_scl.py:204)
    double key = pm;
    int src = p;
    if constexpr (L > 1) {
#pragma unroll
      for (int k = 2; k <= L; k <<= 1) {
#pragma unroll
        for (int d = k >> 1; d > 0; d >>= 1) {
          const double pk = __shfl_xor_sync(FULL, key, d);
          const int ps = __shfl_xor_sync(FULL, src, d);
          const bool take_min = (((p & d) == 0) == ((p & k) == 0 || k == L));
          const bool partner_less = (pk < key) || (pk == key && ps < src);
          if (take_min == partner_less) { key = pk; src = ps; }
        }
      }
    }
    // lane p of each group now holds rank p: (pm ascending, source path)
    const int64_t j = bb * CPW + cwl;
    const bool valid = j < n_codewords();
    const int64_t b = valid ? row_of(j) : 0;
    if (P.pm_out && valid) P.pm_out[b * L + p] = key;
    const int slot = gbase + src;                                  // slot holding the decisions of rank p
    if (P.list && valid)
      for (int w = 0; w < nw; ++w) P.list[((size_t)b * L + p) * nw + w] = rootw[w * 32 + slot];
    // CRC-aided selection (my_sn/fec/polar/dec.py:507-520): pm += 30*k for candidates failing the CRC
    double pen = key;
    if (P.crc_len > 0 && P.crc_rows) {
      uint32_t syn = 0u;
      for (int w = 0; w < nw; ++w) {
        uint32_t uw = rootw[w * 32 + slot];
        while (uw) {
          const int bpos = __ffs(uw) - 1;
          uw &= uw - 1u;
          const int pos = w * 32 + bpos;
          if (pos < n) syn ^= __ldg(P.crc_rows + pos);
        }
      }
      if (syn != 0u) pen = key + kLlrMaxD * (double)P.k;
    }
    // argmin over the L sorted candidates, first minimum wins (np.argmin, dec.py:520)
    double bk = pen;
    int bi = p;
#pragma unroll
    for (int d = L >> 1; d > 0; d >>= 1) {
      const double ok = __shfl_xor_sync(FULL, bk, d);
      const int oi = __shfl_xor_sync(FULL, bi, d);
      if (ok < bk || (ok == bk && oi < bi)) { bk = ok; bi = oi; }
    }
    const int best_slot = gbase + __shfl_sync(FULL, src, gbase + bi);
    if (valid) {
      if (P.best)
        for (int w = p; w < nw; w += L) P.best[(size_t)b * nw + w] = rootw[w * 32 + best_slot];
      if (P.u_info) {
        float *row = P.u_info + b * (int64_t)P.k;
        for (int tt = p; tt < P.k; tt += L) {
          const int pos = __ldg(P.info_pos + tt);
          row[tt] = (float)((rootw[(pos >> 5) * 32 + best_slot] >> (pos & 31)) & 1u);
        }
      }
    }
    __syncwarp();
  }
}

}  // namespace polar

using namespace polar;

// launch_scl2 (launch_scl2_boxplus in the boxplus build), declared in polar_scl.h.  At most 4 KB of dynamic shared
// memory per warp (scl_plan), under the default limit.
int launch_scl2(const SclParams &P, const SclPlan &pl, int L, cudaStream_t st) {
  void (*kern)(const SclParams) = L == 1 ? scl2_kernel<1> : L == 2 ? scl2_kernel<2> : L == 4 ? scl2_kernel<4>
                                  : L == 8 ? scl2_kernel<8> : L == 16 ? scl2_kernel<16> : scl2_kernel<32>;
  kern<<<(unsigned)pl.grid, 32, P.smem_per_warp, st>>>(P);
  count_launch();
  POLAR_CHECK_LAUNCH("scl2_kernel");
  return POLAR_OK;
}
