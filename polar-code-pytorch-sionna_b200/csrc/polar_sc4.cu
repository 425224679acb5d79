// polar_sc4.cu -- SC decoder, warp-autonomous mapping for 128 <= n <= 512 (everything on chip; n >= 1024: polar_sc5.cu).
//
// Same algorithm and exact semantics as polar_sc.cu / polar_sc3.cu (x_run_sn_polar/polar/polar_sc.py:54-133,
// SURVEY.md Appendix A).  Measurements of polar_sc3.cu (CTA per 32 codewords: one warp walks the 64-leaf
// subtrees while three helper warps wait at a barrier) showed that the decoder is bound by the latency of
// that serial walk and that co-resident CTAs do not slow each other down -- throughput is simply (serial
// chains in flight per SM) / (latency of a chain).  So here EVERY warp is a chain:
//   * a warp owns 32 codewords for the whole decode and never synchronises with another warp
//     (__syncwarp only); one persistent CTA per SM holds as many such warps as on-chip storage allows
//     (n=1024: 7 warps = 224 codewords in flight per SM instead of 96..128);
//   * wide stages are processed cooperatively by the 32 lanes (4 elements per lane and round), the 64-leaf
//     subtrees with one lane per codeword, entirely in registers (BetaTree, polar_common.cuh);
//   * storage per codeword, n = 1024: channel stage in global memory / L2; stage 9 virtual (recomputed from
//     the channel, see polar_sc3.cu); stage 8 in TENSOR MEMORY (tcgen05.st/ld 32x32b -- lane l of warp w owns
//     TMEM lane 32(w%4)+l, 256 columns per warp; the tensor cores are idle, their 256 KB per SM is free
//     storage); stages 7 and 6 plus the partial-sum words in shared memory (916 B per codeword).
//   * only partial sums are produced on the serial path; the decisions are recovered once per codeword as
//     u = T(x_hat).
// the 32-leaf level as two separate calls (its children then know at compile time whether their LLRs come from an f and
// skip the clip): +1.5 % here; the larger polar_sc5.cu kernel loses 5 % to the extra code (instruction cache) and keeps it rolled
#define POLAR_BT5_UNROLL 1
#include "polar_common.cuh"
#include "polar_internal.h"
#include "polar_launch.h"

namespace polar {

// phase timeline of warp 0 of CTA 0 (cycles), filled only when POLAR_SC3_DBG=1 (tools/perf_probe.py):
// 0 virtual steps, 1 g steps, 2 f steps, 3 64-leaf subtrees, 4 merges, 5 outputs, 6 total, 7 batches
__device__ unsigned long long g_sc4_dbg[8];

namespace {

constexpr unsigned FULLMASK = 0xFFFFFFFFu;
#define SC4_T(slot)                                                                   \
  do {                                                                                \
    if (DBG && threadIdx.x == 0 && blockIdx.x == 0) {                                 \
      const long long t__ = clock64(); g_sc4_dbg[slot] += (unsigned long long)(t__ - tlast); tlast = t__; \
    }                                                                                 \
  } while (0)


struct Sc4Layout {
  int nw, nws, n64, top, stride;
  size_t nz_off, warp_off, per_warp, total;
};
__host__ __device__ inline Sc4Layout sc4_layout(int m, int top, int bot, int warps) {
  Sc4Layout l;
  const int n = 1 << m;
  l.nw = n >> 5; l.nws = l.nw + 1; l.n64 = n >> bot;    // n64: number of 2^bot-leaf blocks
  l.top = top;                                        // highest stage kept in shared memory (>= 6)
  l.stride = (2 << l.top) - (1 << bot) + 4;           // floats per codeword row (stages bot..top); stride/4 is odd
  l.nz_off = (size_t)((l.nw * 4 + 15) / 16) * 16;
  l.warp_off = l.nz_off + (size_t)((2 * l.n64 + 15) / 16) * 16 + 16;   // +16: tensor-memory base address slot
  l.per_warp = (((size_t)32 * l.stride * 4 + (size_t)32 * l.nws * 4) + 15) / 16 * 16;
  l.total = l.warp_off + (size_t)warps * l.per_warp;
  return l;
}

PDEV float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
PDEV float4 lds4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
PDEV void sts4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }
PDEV float4 f4(const float4 a, const float4 b) {
  float4 o;
  o.x = f_minsum(a.x, b.x); o.y = f_minsum(a.y, b.y); o.z = f_minsum(a.z, b.z); o.w = f_minsum(a.w, b.w);
  return o;
}
PDEV float4 f4neg(const float4 a, const float4 b) {   // f on logits (see f_minsum_neg)
  float4 o;
  o.x = f_minsum_neg(a.x, b.x); o.y = f_minsum_neg(a.y, b.y); o.z = f_minsum_neg(a.z, b.z); o.w = f_minsum_neg(a.w, b.w);
  return o;
}
PDEV float4 g4(const float4 a, const float4 b, const uint32_t bits) {   // bit e of `bits` = partial sum of element e
  float4 o;
  o.x = g_minsum(a.x, b.x, (bits << 31) & 0x80000000u);
  o.y = g_minsum(a.y, b.y, (bits << 30) & 0x80000000u);
  o.z = g_minsum(a.z, b.z, (bits << 29) & 0x80000000u);
  o.w = g_minsum(a.w, b.w, (bits << 28) & 0x80000000u);
  return o;
}
// g(-a, -b, u): the operands are logits, the LLR is their negation (polar_sc.py:122)
PDEV float gneg(float a, float b, uint32_t signmask) { return u2f(f2u(a) ^ signmask ^ 0x80000000u) - b; }
PDEV float4 g4neg(const float4 a, const float4 b, const uint32_t bits) {
  float4 o;
  o.x = gneg(a.x, b.x, (bits << 31) & 0x80000000u);
  o.y = gneg(a.y, b.y, (bits << 30) & 0x80000000u);
  o.z = gneg(a.z, b.z, (bits << 29) & 0x80000000u);
  o.w = gneg(a.w, b.w, (bits << 28) & 0x80000000u);
  return o;
}

// ---- tensor memory as per-thread scratch (32x32b: lane l of the warp owns TMEM lane base+l) -----
PDEV void tmem_st8(uint32_t taddr, const float4 a, const float4 b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(f2u(a.x)), "r"(f2u(a.y)), "r"(f2u(a.z)), "r"(f2u(a.w)), "r"(f2u(b.x)), "r"(f2u(b.y)),
               "r"(f2u(b.z)), "r"(f2u(b.w)) : "memory");
}
PDEV void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
struct Tm8 { uint32_t r[8]; };
PDEV void tmem_ld8_issue(uint32_t taddr, Tm8 &v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v.r[0]), "=r"(v.r[1]), "=r"(v.r[2]), "=r"(v.r[3]), "=r"(v.r[4]), "=r"(v.r[5]), "=r"(v.r[6]), "=r"(v.r[7])
               : "r"(taddr) : "memory");
}
// the registers are defined only after the wait; tying them to it keeps every use behind it
PDEV void tmem_ld_wait(Tm8 &a, Tm8 &b) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a.r[0]), "+r"(a.r[1]), "+r"(a.r[2]), "+r"(a.r[3]), "+r"(a.r[4]), "+r"(a.r[5]), "+r"(a.r[6]), "+r"(a.r[7]),
                 "+r"(b.r[0]), "+r"(b.r[1]), "+r"(b.r[2]), "+r"(b.r[3]), "+r"(b.r[4]), "+r"(b.r[5]), "+r"(b.r[6]), "+r"(b.r[7])
               :: "memory");
}
PDEV float4 tm_lo(const Tm8 &v) { return make_float4(u2f(v.r[0]), u2f(v.r[1]), u2f(v.r[2]), u2f(v.r[3])); }
PDEV float4 tm_hi(const Tm8 &v) { return make_float4(u2f(v.r[4]), u2f(v.r[5]), u2f(v.r[6]), u2f(v.r[7])); }

// ---- cooperative steps of ONE warp over its 32 codewords ------------------------------------------
// stage S+1 -> S inside shared memory.  out[j] = f(a[j], a[j+H]) or g(a[j], a[j+H], beta_left[j]).
template <int S, bool IS_G, int BOT>
PDEV void step_smem(float *L, const uint32_t *beta, int stride, int nws, int lane, int left_word) {
  constexpr int H = 1 << S, HQ = H >> 2, ITEMS = 32 * HQ;
  float *dst = L + (H - (1 << BOT));
  const float *src = L + (2 * H - (1 << BOT));
#pragma unroll 4
  for (int it = lane; it < ITEMS; it += 32) {
    const int c = (int)((unsigned)it / (unsigned)HQ), j = (int)((unsigned)it % (unsigned)HQ) << 2;
    const float4 a = lds4(src + c * stride + j), b = lds4(src + c * stride + j + H);
    float4 o;
    if (IS_G) o = g4(a, b, beta[c * nws + left_word + (j >> 5)] >> (j & 31));
    else o = f4(a, b);
    sts4(dst + c * stride + j, o);
  }
}
template <int SMAX, bool IS_G, int BOT>
PDEV void step_smem_any(int s, float *L, const uint32_t *beta, int stride, int nws, int lane, int left_word) {
  if constexpr (SMAX >= BOT) {
    if (s == SMAX) step_smem<SMAX, IS_G, BOT>(L, beta, stride, nws, lane, left_word);
    else step_smem_any<SMAX - 1, IS_G, BOT>(s, L, beta, stride, nws, lane, left_word);
  }
}

// channel (global, stage M) -> stage M-1 in shared memory (n <= 512: everything fits in shared memory).
template <int M, bool IS_G, int BOT>
__device__ __noinline__ void step_glob(const float *__restrict__ logit, int64_t cw0, int nvalid, float *L,
                                       const uint32_t *beta, int stride, int nws, int lane) {
  constexpr int N = 1 << M, H = N >> 1, HQ = H >> 2, ITEMS = 32 * HQ;
  constexpr int U = 4;        // items per round: 8 independent 128-bit loads in flight per lane
  float *dst = L + (H - (1 << BOT));
#pragma unroll 1
  for (int it0 = lane; it0 < ITEMS; it0 += U * 32) {
    float4 a[U], b[U];
#pragma unroll
    for (int r = 0; r < U; ++r) {
      const int it = it0 + r * 32;
      const int c = (int)((unsigned)it / (unsigned)HQ), j = (int)((unsigned)it % (unsigned)HQ) << 2;
      const int cl = c < nvalid ? c : nvalid - 1;
      const float *row = logit + (cw0 + cl) * (int64_t)N + j;
      a[r] = ldg4(row); b[r] = ldg4(row + H);
    }
#pragma unroll
    for (int r = 0; r < U; ++r) {
      const int it = it0 + r * 32;
      const int c = (int)((unsigned)it / (unsigned)HQ), j = (int)((unsigned)it % (unsigned)HQ) << 2;
      float4 o;
      if (IS_G) o = g4neg(a[r], b[r], beta[c * nws + (j >> 5)] >> (j & 31));
      else o = f4neg(a[r], b[r]);                       // f(-a,-b) == f(a,b) for min-sum
      sts4(dst + c * stride + j, o);
    }
  }
}

// channel (global, stage M) -> stage M-1 in TENSOR MEMORY (n = 512: no virtual stage needed).
// Work item p = lane + 32k = (codeword c, pair q): the float4 at elements 4q and 4q + H/2 of the stage M-1 node.
template <int M, bool IS_G>
__device__ __noinline__ void step_glob_tmem(const float *__restrict__ logit, int64_t cw0, int nvalid, const uint32_t *beta,
                                            int nws, int lane, uint32_t tm_base) {
  constexpr int N = 1 << M, H = N >> 1, PQ = H >> 3;   // PQ pairs per codeword (multiple of 32)
  constexpr int KMAX = PQ, VU = 4;
#pragma unroll 1
  for (int k0 = 0; k0 < KMAX; k0 += VU) {
    float4 a[VU][2], b[VU][2];
#pragma unroll
    for (int r = 0; r < VU; ++r) {
      const int p = lane + 32 * (k0 + r);
      const int c = (int)((unsigned)p / (unsigned)PQ), q = (int)((unsigned)p % (unsigned)PQ);
      const int cl = c < nvalid ? c : nvalid - 1;
      const float *row = logit + (cw0 + cl) * (int64_t)N + 4 * q;
#pragma unroll
      for (int e = 0; e < 2; ++e) { a[r][e] = ldg4(row + e * (H / 2)); b[r][e] = ldg4(row + e * (H / 2) + H); }
    }
#pragma unroll
    for (int r = 0; r < VU; ++r) {
      const int p = lane + 32 * (k0 + r);
      const int c = (int)((unsigned)p / (unsigned)PQ), q = (int)((unsigned)p % (unsigned)PQ);
      float4 o[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int j = 4 * q + e * (H / 2);
        if (IS_G) o[e] = g4neg(a[r][e], b[r][e], beta[c * nws + (j >> 5)] >> (j & 31));
        else o[e] = f4neg(a[r][e], b[r][e]);              // f(-a,-b) == f(a,b) for min-sum
      }
      tmem_st8(tm_base + 8 * (k0 + r), o[0], o[1]);
    }
  }
  tmem_wait_st();
}

// stage TS (tensor memory, lane-private pairs) -> stage TS-1 in shared memory.
template <int TS, bool IS_G, int BOT>   // TS = stage held in tensor memory; writes stage TS-1
PDEV void step_tmem(float *L, const uint32_t *beta, int stride, int nws, int lane, uint32_t tm_base, int left_word) {
  constexpr int H = 1 << (TS - 1), PQ = H >> 2;        // H outputs per codeword = PQ float4
  constexpr int KMAX = PQ;
  float *dst = L + (H - (1 << BOT));
#pragma unroll 2
  for (int k0 = 0; k0 < KMAX; k0 += 2) {
    Tm8 v0, v1;
    tmem_ld8_issue(tm_base + 8 * k0, v0);
    tmem_ld8_issue(tm_base + 8 * (k0 + 1), v1);
    tmem_ld_wait(v0, v1);
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int p = lane + 32 * (k0 + r);
      const int c = (int)((unsigned)p / (unsigned)PQ), j = (int)((unsigned)p % (unsigned)PQ) << 2;
      const float4 a = tm_lo(r ? v1 : v0), b = tm_hi(r ? v1 : v0);
      float4 o;
      if (IS_G) o = g4(a, b, beta[c * nws + left_word + (j >> 5)] >> (j & 31));
      else o = f4(a, b);
      sts4(dst + c * stride + j, o);
    }
  }
}

// ---- one lane per codeword: the 64-leaf subtree below the lane's stage-6 node (shared memory) -----
PDEV uint2 bottom64(const float *node, uint32_t fm0, uint32_t fm1) {
  uint32_t bl = 0, bc = 0;
#pragma unroll 1
  for (int h = 0; h < 2; ++h) {      // rolled: one copy of the 32-leaf subtree code
    const uint32_t fmc = h ? fm1 : fm0;
    if (fmc == FULLMASK) { bc = 0; continue; }
    float x[32];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 a = lds4(node + 4 * q), b = lds4(node + 32 + 4 * q);
      const float4 o = h ? g4(a, b, bl >> (4 * q)) : f4(a, b);
      x[4 * q] = o.x; x[4 * q + 1] = o.y; x[4 * q + 2] = o.z; x[4 * q + 3] = o.w;
    }
    bc = BetaTree<5>::run(x, fmc);
    if (h == 0) bl = bc;
  }
  return make_uint2(bl ^ bc, bc);
}

// MODE 0: stages 6..M-1 in shared memory (n <= 256).  MODE 1: stage M-1 in tensor memory (n = 512).
// the 128-leaf subtree below the lane's stage-7 node: both 64-leaf halves in registers (x[64] + the BetaTree levels),
// so that shared memory only has to hold stage 7 (one more warp per SM) and stage 6 costs no LDS/STS round trip.
PDEV uint64_t tree64(const float (&x)[64], uint64_t fm) {
  uint32_t bl = 0, bc = 0;
#pragma unroll 1
  for (int h = 0; h < 2; ++h) {
    const uint32_t fmc = h ? (uint32_t)(fm >> 32) : (uint32_t)fm;
    if (fmc == FULLMASK) { bc = 0; continue; }
    float y[32];
#pragma unroll
    for (int j = 0; j < 32; ++j)
      y[j] = h ? g_minsum(x[j], x[j + 32], (bl << (31 - j)) & 0x80000000u) : f_minsum(x[j], x[j + 32]);
    bc = BetaTree<5>::run(y, fmc);
    if (h == 0) bl = bc;
  }
  return (uint64_t)(bl ^ bc) | ((uint64_t)bc << 32);
}
PDEV uint4 bottom128(const float *node, uint64_t fm0, uint64_t fm1) {
  uint64_t bl = 0, bc = 0;
#pragma unroll 1
  for (int h = 0; h < 2; ++h) {
    const uint64_t fmc = h ? fm1 : fm0;
    if (fmc == ~0ull) { bc = 0; continue; }
    float x[64];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const float4 a = lds4(node + 4 * q), b = lds4(node + 64 + 4 * q);
      const float4 o = h ? g4(a, b, (uint32_t)(bl >> (4 * q))) : f4(a, b);
      x[4 * q] = o.x; x[4 * q + 1] = o.y; x[4 * q + 2] = o.z; x[4 * q + 3] = o.w;
    }
    bc = tree64(x, fmc);
    if (h == 0) bl = bc;
  }
  const uint64_t lo = bl ^ bc;
  return make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)bc, (uint32_t)(bc >> 32));
}

// DBG: per-phase timeline of warp 0 of CTA 0 (POLAR_SC3_DBG=1) as a separate instantiation: the product kernel carries no timer code
template <int M, int MODE, bool DBG>
__global__ void __launch_bounds__(256, 1) sc4_kernel(const float *__restrict__ logit, const uint32_t *__restrict__ fmask_g,
                                                     int64_t B, int64_t nbatches,
                                                     uint32_t *__restrict__ u_packed, float *__restrict__ u_info,
                                                     const int32_t *__restrict__ info_pos, int k) {
  constexpr bool TM = MODE == 1;
  constexpr int TS = M - 1;                                 // stage held in tensor memory (TM only)
  static_assert(MODE == 0 ? (M >= 7) : (TS >= 8 && TS <= 9), "sc4: the bottom stage must exist in shared memory; a warp reaches 512 TMEM columns");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int BOT = (M >= 8) ? 7 : 6;                      // stage of the node the per-lane subtree starts from
  constexpr int WB = 1 << (BOT - 5);                         // 32-bit words per bottom block
  constexpr int N = 1 << M, NW = N >> 5, NWS = NW + 1, N64 = N >> BOT, TOP = TM ? TS - 1 : M - 1;
  constexpr int TM_COLS_WARP = TM ? (1 << TS) : 32;         // 32 codewords x 2^TS floats / 32 lanes
  // lane-0 broadcasts: warp index and frozen-pattern words are warp uniform, and the shuffle lets the compiler know
  // (uniform branches instead of potentially divergent ones in the register subtrees; see polar_sc5.cu)
  const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(FULLMASK, tid >> 5, 0), nwarps = blockDim.x >> 5;
  const Sc4Layout lay = sc4_layout(M, TOP, BOT, nwarps);
  constexpr int stride = (2 << TOP) - (1 << BOT) + 4;   // == lay.stride, compile-time so that row offsets fold into immediates
  uint32_t *fmask = reinterpret_cast<uint32_t *>(smem_raw);
  unsigned char *nz = smem_raw + lay.nz_off;    // nz[(N64 >> lv) + (i >> lv)]: node of 2^lv 64-blocks at block i is rate-0
  uint32_t *tm_slot = reinterpret_cast<uint32_t *>(smem_raw + lay.warp_off - 16);
  float *L = reinterpret_cast<float *>(smem_raw + lay.warp_off + (size_t)warp * lay.per_warp);
  uint32_t *beta = reinterpret_cast<uint32_t *>(L + 32 * stride);

  uint32_t tm_base = 0;
  if (TM) {
    if (warp == 0) {          // the CTA is alone on its SM (shared memory): take all 512 columns
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                   ::"r"((uint32_t)__cvta_generic_to_shared(tm_slot)), "n"(512) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  for (int i = tid; i < NW; i += blockDim.x) fmask[i] = __ldg(fmask_g + i);
  __syncthreads();
  if (TM) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // warp w: TMEM lanes 32(w%4)..+31 (the only ones it can address), column block w/4
    tm_base = *tm_slot + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * TM_COLS_WARP);
  }
  for (int i = tid; i < N64; i += blockDim.x) {
    uint32_t all = FULLMASK;
    for (int w = 0; w < WB; ++w) all &= fmask[WB * i + w];
    nz[N64 + i] = all == FULLMASK;
  }
  __syncthreads();
  if (tid == 0)
    for (int idx = N64 - 1; idx >= 1; --idx) nz[idx] = nz[2 * idx] & nz[2 * idx + 1];
  __syncthreads();

  long long tlast = DBG ? clock64() : 0;
  const long long tstart = tlast;
  const int64_t wstride = (int64_t)gridDim.x * nwarps;
  for (int64_t batch = (int64_t)warp * gridDim.x + blockIdx.x; batch < nbatches; batch += wstride) {
    const int64_t cw0 = batch * 32;
    const int nvalid = (int)((B - cw0) < 32 ? (B - cw0) : 32);
    int i = 0;                                   // current 64-leaf block
    while (i < N64) {
      // node entered at block i: the root, or the right child whose left sibling just finished
      const int S = (i == 0) ? M : BOT + (__ffs(i) - 1);
      int s = S;
      bool zeroed = nz[(N64 >> (S - BOT)) + (i >> (S - BOT))] != 0;
      if (!zeroed && S < M) {
        // g step into (S, i) from its parent at stage S+1; the left sibling's beta starts at word 2*(i - 2^(S-6))
        const int left_word = WB * (i - (1 << (S - BOT)));
        if (TM && S == M - 1) {
          step_glob_tmem<M, true>(logit, cw0, nvalid, beta, NWS, lane, tm_base);
        } else if (TM && S == TS - 1) {
          step_tmem<TS, true, BOT>(L, beta, stride, NWS, lane, tm_base, left_word);
        } else if (!TM && S == M - 1) {
          step_glob<M, true, BOT>(logit, cw0, nvalid, L, beta, stride, NWS, lane);
        } else {
          step_smem_any<TOP - 1, true, BOT>(S, L, beta, stride, NWS, lane, left_word);
        }
        __syncwarp();
        SC4_T(1);
      }
      while (!zeroed && s > BOT) {
        if (nz[(N64 >> (s - 1 - BOT)) + (i >> (s - 1 - BOT))]) { zeroed = true; --s; break; }   // left child is rate-0
        if (TM && s == M) {
          step_glob_tmem<M, false>(logit, cw0, nvalid, beta, NWS, lane, tm_base);
        } else if (TM && s == TS) {
          step_tmem<TS, false, BOT>(L, beta, stride, NWS, lane, tm_base, 0);
        } else if (!TM && s == M) {
          step_glob<M, false, BOT>(logit, cw0, nvalid, L, beta, stride, NWS, lane);
        } else {
          step_smem_any<TOP - 1, false, BOT>(s - 1, L, beta, stride, NWS, lane, 0);
        }
        __syncwarp();
        SC4_T(2);
        --s;
      }
      const int lv0 = s - BOT;                   // the finished node covers 2^lv0 bottom blocks starting at i
      if (zeroed) {
        const int nwd = WB << lv0;
        for (int q = lane; q < 32 * nwd; q += 32) {
          const int c = q / nwd, w = q & (nwd - 1);
          beta[c * NWS + WB * i + w] = 0u;
        }
      } else if (BOT == 7) {
        const uint32_t *fmw = fmask + 4 * i;
        const uint32_t f0 = __shfl_sync(FULLMASK, fmw[0], 0), f1 = __shfl_sync(FULLMASK, fmw[1], 0);
        const uint32_t f2 = __shfl_sync(FULLMASK, fmw[2], 0), f3 = __shfl_sync(FULLMASK, fmw[3], 0);
        const uint4 b = bottom128(L + lane * stride, (uint64_t)f0 | ((uint64_t)f1 << 32), (uint64_t)f2 | ((uint64_t)f3 << 32));
        uint32_t *bp = beta + lane * NWS + 4 * i;
        bp[0] = b.x; bp[1] = b.y; bp[2] = b.z; bp[3] = b.w;
      } else {
        const uint2 b = bottom64(L + lane * stride, __shfl_sync(FULLMASK, fmask[2 * i], 0), __shfl_sync(FULLMASK, fmask[2 * i + 1], 0));
        uint32_t *bp = beta + lane * NWS + 2 * i;
        bp[0] = b.x; bp[1] = b.y;
      }
      __syncwarp();
      SC4_T(3);
      {  // merge partial sums upward while the finished node is a right child: [bl ^ br, br] (polar_sc.py:83-89)
        int lv = lv0, a = i;
        while (lv < M - BOT && ((a >> lv) & 1)) {
          const int nwd = WB << lv, left = a - (1 << lv);
          for (int q = lane; q < 32 * nwd; q += 32) {
            const int c = q / nwd, w = q & (nwd - 1);
            beta[c * NWS + WB * left + w] ^= beta[c * NWS + WB * a + w];
          }
          __syncwarp();
          a = left; ++lv;
        }
      }
      SC4_T(4);
      i += 1 << lv0;
    }
    // beta now holds the re-encoded codeword x_hat of every codeword; the decisions are u = T(x_hat)
    // (my_sn/fec/polar/enc.py:85-96 is an involution): 5 stages inside each word, M-5 across words.
    for (int q = lane; q < 32 * NW; q += 32) {
      const int c = q / NW, w = q % NW;
      beta[c * NWS + w] = ptransform<5>(beta[c * NWS + w]);
    }
    __syncwarp();
#pragma unroll 1
    for (int st = 0; st < M - 5; ++st) {
      for (int q = lane; q < 32 * (NW / 2); q += 32) {
        const int c = q / (NW / 2), r = q % (NW / 2);
        const int w = ((r >> st) << (st + 1)) | (r & ((1 << st) - 1));     // word index with bit st clear
        beta[c * NWS + w] ^= beta[c * NWS + w + (1 << st)];
      }
      __syncwarp();
    }
    if (u_packed) {
      for (int q = lane; q < 32 * NW; q += 32) {
        const int c = q / NW, w = q % NW;
        if (c < nvalid) u_packed[(cw0 + c) * NW + w] = beta[c * NWS + w];
      }
    }
    if (u_info) {
      // the API tensor [B, k] fp32 (polar_sc.py:127-133): a codeword's row at a time, one float4 per lane and round
      // (bit -> 0.f / 1.f by masking the bit pattern of 1.0f: no int-to-float conversion on the slow pipe)
      if ((k & 3) == 0 && (reinterpret_cast<uintptr_t>(u_info) & 15) == 0 && (reinterpret_cast<uintptr_t>(info_pos) & 15) == 0) {
        const int k4 = k >> 2;
        const int4 *ip = reinterpret_cast<const int4 *>(info_pos);
        for (int c = 0; c < nvalid; ++c) {
          float4 *row = reinterpret_cast<float4 *>(u_info + (cw0 + c) * (int64_t)k);
          const uint32_t *bw = beta + c * NWS;
          for (int t4 = lane; t4 < k4; t4 += 32) {
            const int4 p = __ldg(ip + t4);
            float4 o;
            o.x = u2f((0u - ((bw[p.x >> 5] >> (p.x & 31)) & 1u)) & 0x3f800000u);
            o.y = u2f((0u - ((bw[p.y >> 5] >> (p.y & 31)) & 1u)) & 0x3f800000u);
            o.z = u2f((0u - ((bw[p.z >> 5] >> (p.z & 31)) & 1u)) & 0x3f800000u);
            o.w = u2f((0u - ((bw[p.w >> 5] >> (p.w & 31)) & 1u)) & 0x3f800000u);
            __stcs(row + t4, o);
          }
        }
      } else {
        for (int q = lane; q < nvalid * k; q += 32) {
          const int c = q / k, t = q - c * k;
          const int p = __ldg(info_pos + t);
          u_info[(cw0 + c) * (int64_t)k + t] = (float)((beta[c * NWS + (p >> 5)] >> (p & 31)) & 1u);
        }
      }
    }
    __syncwarp();
    SC4_T(5);
    if (DBG && tid == 0 && blockIdx.x == 0) g_sc4_dbg[7] += 1;
  }
  if (DBG && tid == 0 && blockIdx.x == 0) g_sc4_dbg[6] += (unsigned long long)(clock64() - tstart);
  if (TM) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tm_slot), "n"(512) : "memory");
  }
}

}  // namespace

namespace {

template <int M, int MODE>
int launch_sc4_t(const float *logit, const uint32_t *fmask, int64_t B, uint32_t *u_packed, float *u_info,
                 const int32_t *info_pos, int k, int warps, cudaStream_t st) {
  const int max_smem = device_max_smem_optin();
  constexpr bool TM = MODE >= 1;
  constexpr int TS = M - 1;
  int wmax = 8;
  if (TM) wmax = 4 * (512 >> TS);               // TMEM columns: 2^TS per warp, 512 per lane quarter
  if (wmax > 8) wmax = 8;
  if (warps <= 0 || warps > wmax) warps = wmax;
  constexpr int TOP = TM ? TS - 1 : M - 1, BOT = (M >= 8) ? 7 : 6;
  while (warps > 1 && sc4_layout(M, TOP, BOT, warps).total > (size_t)max_smem) --warps;
  const Sc4Layout lay = sc4_layout(M, TOP, BOT, warps);
  if (lay.total > (size_t)max_smem) return set_error(POLAR_ENOMEM, "sc: n=%d needs %zu B shared memory per CTA", 1 << M, lay.total);
  auto kern = env_int("POLAR_SC3_DBG", 0) != 0 ? sc4_kernel<M, MODE, true> : sc4_kernel<M, MODE, false>;
  // one persistent CTA per SM.  With tensor memory the CTA takes all 512 columns, so a second CTA must never
  // become resident on the same SM: pad the request above half of the SM's shared memory.
  size_t smem = lay.total;
  if (TM && smem < (size_t)116 * 1024) smem = (size_t)116 * 1024;
  POLAR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t nbatches = (B + 31) / 32;
  return launch("sc4_kernel", kern, grid_for(nbatches, warps, 1), warps * 32, smem, st, logit, fmask, B, nbatches, u_packed,
                u_info, info_pos, k);
}

}  // namespace

// n in [128, 512].  warps = autonomous warps per SM (0 = as many as shared memory / tensor memory hold).
int launch_sc4(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
               const int32_t *info_pos, int k, int warps, cudaStream_t st) {
  switch (ilog2(n)) {
    case 7: return launch_sc4_t<7, 0>(logit, fmask, B, u_packed, u_info, info_pos, k, warps, st);
    case 8: return launch_sc4_t<8, 0>(logit, fmask, B, u_packed, u_info, info_pos, k, warps, st);
    case 9: return launch_sc4_t<9, 1>(logit, fmask, B, u_packed, u_info, info_pos, k, warps, st);
    default: return set_error(POLAR_EINVAL, "sc4: n=%d not supported by this mapping", n);
  }
}

}  // namespace polar

// debug only (not part of include/polar_b200.h): read and clear the phase timeline of warp 0 of CTA 0
extern "C" int polar_sc4_debug_read(unsigned long long *h_out8) {
  unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (cudaMemcpyFromSymbol(h_out8, polar::g_sc4_dbg, sizeof(z)) != cudaSuccess) return POLAR_ECUDA;
  if (cudaMemcpyToSymbol(polar::g_sc4_dbg, z, sizeof(z)) != cudaSuccess) return POLAR_ECUDA;
  return POLAR_OK;
}
