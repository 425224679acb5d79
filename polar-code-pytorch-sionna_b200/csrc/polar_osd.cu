// polar_osd.cu -- ordered-statistics decoder (SURVEY 8f row N4; reference my_sn/fec/osd/dec.py:8-192).
//
// One CTA per codeword, the whole decode in shared memory:
//   1. clip the logits to +-100 (dec.py:155) and order the positions by |llr|, most reliable first (dec.py:157;
//      equal magnitudes keep their index order -- torch.argsort makes no promise there);
//   2. the generator matrix with its columns in that order, one bit-packed ROW per information bit: a column
//      permutation is a bit gather, a row operation of the elimination a word-wise XOR;
//   3. most-reliable basis exactly as dec.py:99-117 forms it: for row c = 0 .. k-1 the pivot is the FIRST set position
//      of row c, and that column is cleared from every other row (so the basis depends on the row order of G);
//   4. the k pivot positions are hard-decided (llr > 0 -> 1, sim.py:4-6) and re-encoded (dec.py:171-174); every error
//      pattern of weight 1 .. t on the pivots is tested in the reference's order (itertools.combinations, dec.py:57-62)
//      with the LLR distance mean_j log(1 + exp(llr_j (1 - 2 c_j))) (dec.py:64-79, fp32, literal); within one weight
//      the first minimum wins (argmin, dec.py:93), across weights only a strictly smaller distance (dec.py:181-184);
//   5. the winner goes back to the original positions (dec.py:186-188).
// The reference permutes the matrix a second time to [pivots | parity] order (dec.py:118-134); that only reorders the
// terms of the distance sum, so it is not done here.  Distances are fp32 sums in sorted-position order: they agree with
// the reference's to rounding, and so does the decision except where two candidates are closer than that (the tests
// skip exactly those, like the list decoder's ill-conditioned lists).
#include "polar_common.cuh"
#include "polar_launch.h"

namespace polar {
namespace {

constexpr int kOsdThreads = 128;
constexpr int kOsdWarps = kOsdThreads / 32;
constexpr int kOsdMaxT = 6;

struct OsdLayout {
  int nw, np2;
  size_t rows_off, key_off, idx_off, cost_off, vec_off, piv_off, flag_off, red_off, total;
};
__host__ __device__ inline OsdLayout osd_layout(int n, int k) {
  OsdLayout l;
  l.nw = (n + 31) >> 5;
  int p = 1;
  while (p < n) p <<= 1;
  l.np2 = p;
  size_t o = 0;
  auto take = [&o](size_t bytes) { const size_t at = o; o += (bytes + 15) / 16 * 16; return at; };   // 16-byte aligned pieces
  l.rows_off = take((size_t)k * l.nw * 4);         // G, columns in sorted order, bit-packed rows
  l.key_off = take((size_t)l.np2 * 4);             // |llr| (sort keys); afterwards the clipped logits in sorted order
  l.idx_off = take((size_t)l.np2 * 4);             // original position of sorted position j
  l.cost_off = take((size_t)n * 8);                // {log(1+exp(+llr_j)), log(1+exp(-llr_j))}: cost of c_j = 0 / 1
  l.vec_off = take((size_t)3 * l.nw * 4);          // order-0 codeword, prefix candidate, output words
  l.piv_off = take((size_t)k * 4);
  l.flag_off = take((size_t)k * 4);
  l.red_off = take(256);
  l.total = (o + 15) / 16 * 16;
  return l;
}

struct Cand {                    // a tested pattern: distance, position in the reference's pattern list, the flipped pivots
  float d;
  unsigned rank;
  int e[kOsdMaxT];
};
// ordered like the reference's argmin: smaller distance first, then the earlier pattern
PDEV bool cand_less(float d, unsigned r, float d2, unsigned r2) { return d < d2 || (d == d2 && r < r2); }

// mean_j of the position costs of the codeword a ^ b (dec.py:64-79), summed in position order
PDEV float osd_distance(const uint32_t *a, const uint32_t *b, const float2 *cost, int n, int nw) {
  float acc = 0.0f;
  for (int w = 0; w < nw; ++w) {
    uint32_t x = a[w] ^ (b ? b[w] : 0u);
    const int jend = min(32, n - 32 * w);
    const float2 *cw = cost + 32 * w;
    for (int j = 0; j < jend; ++j, x >>= 1) {
      const float2 c = cw[j];
      acc += (x & 1u) ? c.y : c.x;
    }
  }
  return acc / (float)n;
}

__global__ void __launch_bounds__(kOsdThreads) osd_kernel(const float *__restrict__ logit, const uint32_t *__restrict__ gm,
                                                           int n, int k, int t, int64_t B, uint32_t *__restrict__ c_packed,
                                                           float *__restrict__ c_f32, float *__restrict__ dist_out) {
  extern __shared__ __align__(16) unsigned char osd_smem[];
  const OsdLayout lay = osd_layout(n, k);
  const int nw = lay.nw, np2 = lay.np2, tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  uint32_t *rows = reinterpret_cast<uint32_t *>(osd_smem + lay.rows_off);
  float *key = reinterpret_cast<float *>(osd_smem + lay.key_off);
  int *idx = reinterpret_cast<int *>(osd_smem + lay.idx_off);
  float2 *cost = reinterpret_cast<float2 *>(osd_smem + lay.cost_off);
  uint32_t *base = reinterpret_cast<uint32_t *>(osd_smem + lay.vec_off);
  uint32_t *pref = base + nw, *outw = base + 2 * nw;
  int *piv = reinterpret_cast<int *>(osd_smem + lay.piv_off);
  int *flag = reinterpret_cast<int *>(osd_smem + lay.flag_off);
  float *red_d = reinterpret_cast<float *>(osd_smem + lay.red_off);          // per warp: best distance ...
  unsigned *red_r = reinterpret_cast<unsigned *>(red_d + kOsdWarps);          // ... its rank ...
  int *red_e = reinterpret_cast<int *>(red_r + kOsdWarps);                    // ... its pattern [warp][kOsdMaxT]
  int *ctl = red_e + kOsdWarps * kOsdMaxT;                                    // [0] pivot of the current row

  for (int64_t cw = blockIdx.x; cw < B; cw += gridDim.x) {
    const float *x = logit + cw * (int64_t)n;
    // 1. keys |clip(llr)|, padding sorts last; bitonic network, ties by position
    for (int j = tid; j < np2; j += T) {
      key[j] = j < n ? fabsf(fminf(fmaxf(x[j], -100.0f), 100.0f)) : -1.0f;
      idx[j] = j;
    }
    __syncthreads();
    for (int sz = 2; sz <= np2; sz <<= 1)
      for (int st = sz >> 1; st > 0; st >>= 1) {
        for (int i = tid; i < np2 / 2; i += T) {
          const int lo = ((i & ~(st - 1)) << 1) | (i & (st - 1)), hi = lo | st;
          const bool first_wins = (lo & sz) == 0;    // this block is sorted most-reliable-first
          const float a = key[lo], b = key[hi];
          const int ia = idx[lo], ib = idx[hi];
          const bool a_first = a > b || (a == b && ia < ib);
          if (a_first != first_wins) { key[lo] = b; key[hi] = a; idx[lo] = ib; idx[hi] = ia; }
        }
        __syncthreads();
      }
    // sorted logits and the per-position costs (dec.py:75-78: llr_sign = llr (1 - 2c); d = log(1 + exp(llr_sign)))
    for (int j = tid; j < n; j += T) {
      const float v = fminf(fmaxf(x[idx[j]], -100.0f), 100.0f);
      key[j] = v;
      cost[j] = make_float2(logf(1.0f + expf(v)), logf(1.0f + expf(-v)));
    }
    // 2. rows of G with the columns in sorted order
    for (int q = tid; q < k * nw; q += T) {
      const int r = q / nw, w = q - r * nw;
      const uint32_t *g = gm + (size_t)r * nw;
      uint32_t acc = 0;
      const int jend = min(32, n - 32 * w);
      for (int b = 0; b < jend; ++b) {
        const int src = idx[32 * w + b];
        acc |= ((__ldg(g + (src >> 5)) >> (src & 31)) & 1u) << b;
      }
      rows[q] = acc;
    }
    __syncthreads();
    // 3. most-reliable basis (dec.py:99-117)
    for (int c = 0; c < k; ++c) {
      if (warp == 0) {
        int p = 0x7fffffff;
        for (int w = lane; w < nw && p == 0x7fffffff; w += 32) {
          const uint32_t v = rows[c * nw + w];
          if (v) p = 32 * w + __ffs(v) - 1;
        }
        for (int o = 16; o > 0; o >>= 1) p = min(p, __shfl_xor_sync(0xffffffffu, p, o));
        if (lane == 0) { p = (p == 0x7fffffff) ? 0 : p; ctl[0] = p; piv[c] = p; }   // all-zero row: argmax gives 0
      }
      __syncthreads();
      const int p = ctl[0];
      for (int r = tid; r < k; r += T) flag[r] = (r != c) && ((rows[r * nw + (p >> 5)] >> (p & 31)) & 1u);
      __syncthreads();
      for (int q = tid; q < k * nw; q += T) {
        const int r = q / nw, w = q - r * nw;
        if (flag[r]) rows[q] ^= rows[c * nw + w];
      }
      __syncthreads();
    }
    // 4. order-0 codeword: hard decisions on the pivots, re-encoded
    for (int w = tid; w < nw; w += T) {
      uint32_t acc = 0;
      for (int r = 0; r < k; ++r)
        if (key[piv[r]] > 0.0f) acc ^= rows[r * nw + w];
      base[w] = acc;
    }
    __syncthreads();
    Cand win;                                       // best candidate so far (identical in every thread)
    win.d = osd_distance(base, nullptr, cost, n, nw);
    win.rank = 0;
    int win_w = 0;
    for (int wt = 1; wt <= t && wt <= k; ++wt) {
      Cand mine;
      mine.d = __int_as_float(0x7fc00000); mine.rank = 0xffffffffu;     // nothing tested yet (NaN never wins a comparison)
      bool have = false;
      int e[kOsdMaxT];
#pragma unroll
      for (int i = 0; i < kOsdMaxT; ++i) { e[i] = i; mine.e[i] = 0; }
      unsigned rank0 = 0;                           // rank of the pattern (e[0..wt-2], e[wt-2]+1)
      bool more = true;
      while (more) {
        // prefix codeword base ^ rows[e[0]] ^ .. ^ rows[e[wt-2]] (uniform over the CTA)
        if (wt > 1) {
          __syncthreads();
          for (int w = tid; w < nw; w += T) {
            uint32_t acc = base[w];
#pragma unroll
            for (int i = 0; i < kOsdMaxT - 1; ++i)
              if (i < wt - 1) acc ^= rows[e[i] * nw + w];
            pref[w] = acc;
          }
          __syncthreads();
        }
        const int first = wt > 1 ? e[wt - 2] + 1 : 0;
        const uint32_t *pv = wt > 1 ? pref : base;
        for (int last = first + tid; last < k; last += T) {
          const float d = osd_distance(pv, rows + last * nw, cost, n, nw);
          const unsigned rk = rank0 + (unsigned)(last - first);
          if (!have || cand_less(d, rk, mine.d, mine.rank)) {
            have = true; mine.d = d; mine.rank = rk;
#pragma unroll
            for (int i = 0; i < kOsdMaxT; ++i) mine.e[i] = i < wt - 1 ? e[i] : last;
          }
        }
        rank0 += (unsigned)(k - first);
        // next prefix in lexicographic order: e[i] may reach k - wt + i (the last index needs room above it)
        more = false;
        if (wt > 1) {
          int i = wt - 2;
          while (i >= 0 && e[i] + 1 > k - wt + i) --i;
          if (i >= 0) {
            ++e[i];
            for (int j = i + 1; j < wt - 1; ++j) e[j] = e[j - 1] + 1;
            more = true;
          }
        }
      }
      // CTA minimum by (distance, rank)
      for (int o = 16; o > 0; o >>= 1) {
        const float d2 = __shfl_xor_sync(0xffffffffu, mine.d, o);
        const unsigned r2 = __shfl_xor_sync(0xffffffffu, mine.rank, o);
        const bool h2 = __shfl_xor_sync(0xffffffffu, (int)have, o) != 0;
        int e2[kOsdMaxT];
#pragma unroll
        for (int i = 0; i < kOsdMaxT; ++i) e2[i] = __shfl_xor_sync(0xffffffffu, mine.e[i], o);
        if (h2 && (!have || cand_less(d2, r2, mine.d, mine.rank))) {
          have = true; mine.d = d2; mine.rank = r2;
#pragma unroll
          for (int i = 0; i < kOsdMaxT; ++i) mine.e[i] = e2[i];
        }
      }
      __syncthreads();
      if (lane == 0) {
        red_d[warp] = mine.d; red_r[warp] = have ? mine.rank : 0xffffffffu;
#pragma unroll
        for (int i = 0; i < kOsdMaxT; ++i) red_e[warp * kOsdMaxT + i] = mine.e[i];
      }
      __syncthreads();
      int bw = -1;
      for (int w = 0; w < kOsdWarps; ++w)
        if (red_r[w] != 0xffffffffu && (bw < 0 || cand_less(red_d[w], red_r[w], red_d[bw], red_r[bw]))) bw = w;
      if (bw >= 0 && red_d[bw] < win.d) {            // dec.py:181-184: strictly smaller only
        win.d = red_d[bw]; win_w = wt;
#pragma unroll
        for (int i = 0; i < kOsdMaxT; ++i) win.e[i] = red_e[bw * kOsdMaxT + i];
      }
    }
    // 5. winner back to the original positions
    __syncthreads();
    for (int w = tid; w < nw; w += T) {
      uint32_t acc = base[w];
#pragma unroll
      for (int i = 0; i < kOsdMaxT; ++i)
        if (i < win_w) acc ^= rows[win.e[i] * nw + w];
      pref[w] = acc;
      outw[w] = 0u;
    }
    __syncthreads();
    for (int j = tid; j < n; j += T) {
      const uint32_t bit = (pref[j >> 5] >> (j & 31)) & 1u;
      const int dst = idx[j];
      if (c_f32) c_f32[cw * (int64_t)n + dst] = bit ? 1.0f : 0.0f;
      if (bit) atomicOr(&outw[dst >> 5], 1u << (dst & 31));
    }
    __syncthreads();
    if (c_packed)
      for (int w = tid; w < nw; w += T) c_packed[cw * (int64_t)nw + w] = outw[w];
    if (dist_out && tid == 0) dist_out[cw] = win.d;
    __syncthreads();
  }
}

}  // namespace
}  // namespace polar

extern "C" int polar_osd_decode(const float *d_logit, const uint32_t *d_gm_rows, int n, int k, int t, int64_t B,
                                uint32_t *d_c_packed, float *d_c_f32, float *d_dist, void *stream) {
  using namespace polar;
  if (!d_logit || !d_gm_rows || (!d_c_packed && !d_c_f32)) return set_error(POLAR_EINVAL, "osd: null pointer");
  if (n < 2 || n > 1024 || k < 1 || k > n) return set_error(POLAR_EINVAL, "osd: need 2 <= n <= 1024 and 1 <= k <= n (got n=%d k=%d)", n, k);
  if (t < 0 || t > kOsdMaxT) return set_error(POLAR_EINVAL, "osd: order t=%d outside [0, %d]", t, kOsdMaxT);
  if (B < 0) return set_error(POLAR_EINVAL, "osd: B < 0");
  double pat = 1.0;                                   // C(k, t) patterns must be countable in 32 bits
  for (int i = 0; i < t && i < k; ++i) pat = pat * (double)(k - i) / (double)(i + 1);
  if (pat > 2.0e9) return set_error(POLAR_EINVAL, "osd: C(%d, %d) error patterns are too many", k, t);
  if (B == 0) return POLAR_OK;
  const OsdLayout lay = osd_layout(n, k);
  if (lay.total > (size_t)device_max_smem_optin()) return set_error(POLAR_ENOMEM, "osd: n=%d k=%d does not fit in shared memory", n, k);
  POLAR_CUDA(cudaFuncSetAttribute(osd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.total));
  // persistent CTAs: as many as are resident at once, queried on every call because the shared memory depends on n and k
  const unsigned grid = grid_for(B, 1, resident_ctas(osd_kernel, kOsdThreads, lay.total));
  return launch("osd_kernel", osd_kernel, grid, kOsdThreads, lay.total, (cudaStream_t)stream, d_logit, d_gm_rows, n, k, t, B,
                d_c_packed, d_c_f32, d_dist);
}
