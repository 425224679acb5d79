// polar_sc5.cu -- SC decoder for n = 1024 .. 8192: warp-autonomous like polar_sc4.cu, with
//   (1) every global read of the top stages STAGED THROUGH SHARED MEMORY BY THE TMA ENGINE (cp.async.bulk + mbarrier):
//       four 4 KB slots per warp (its own stage-7 buffer, dead during a descent), 16 KB in flight per descending warp.
//       ncu of the register-landing version showed the row passes waiting on loads whose scoreboards serialise (8 KB in
//       flight per warp); a bulk copy needs no register and no scoreboard;
//   (2) a scratch HIERARCHY for the stages that do not fit on chip: the stage-8 node of every codeword lives in tensor
//       memory (256 columns per warp -> 8 warps per SM for every n), stage 7 + partial sums in shared memory, the
//       128-leaf subtrees in registers -- and the live node of each stage 9 .. m-1 in a per-warp global scratch
//       (L2-resident for n = 1024, L2 + HBM above).  Each scratch node is written once, by the fused descent that
//       forms it, and read once, by the descent into its right sibling; consumed lines are dropped from the L2
//       (discard.global.L2) so that they are never written back.
// Same algorithm and exact semantics as the other SC units (x_run_sn_polar/polar/polar_sc.py:54-133, SURVEY App. A).
//
// Descent: entering the node (S, i) -- the root, or a right child whose left sibling has just been decoded -- one pass
// reads the parent (channel row or scratch node of stage S+1), applies g (f at the root), stores the stage-S node, and
// keeps going down the LEFT spine with f, storing every stage >= 9 it passes and ending with the stage-8 node in tensor
// memory.  All of that happens in registers on data that crossed the memory system once.
#include <atomic>
#include <mutex>

#include "polar_common.cuh"
#include "polar_internal.h"

namespace polar {

#if !defined(POLAR_F_BOXPLUS)     // one scratch per device for the whole library: the boxplus unit uses ::polar's
namespace {
__global__ void nsmid_kernel(unsigned *out) {
  unsigned v;
  asm volatile("mov.u32 %0, %%nsmid;" : "=r"(v));
  *out = v;
}
std::mutex g_scr_mu;
std::atomic<float *> g_scr_buf[64];
}  // namespace

// Per-device stage scratch of the SC decoder for n >= 1024: %nsmid slots of kScScratchPerSm (the live nodes of stages
// 9 .. m-1 of every codeword in flight on an SM; 592 MB on a 148-SM part, of which n = 1024 touches 76 MB -- small enough
// to stay resident in the L2).  Allocated once by polar_init(device) (which may allocate and synchronise; the decode
// entry points never do) and kept for the life of the process.
int sc_scratch_init(int device) {
  if (device < 0 || device >= 64) return set_error(POLAR_EINVAL, "init: bad device %d", device);
  std::lock_guard<std::mutex> lk(g_scr_mu);
  if (g_scr_buf[device].load(std::memory_order_acquire)) return POLAR_OK;
  unsigned *d_n = nullptr, h_n = 0;
  POLAR_CUDA(cudaMalloc(&d_n, sizeof(unsigned)));
  nsmid_kernel<<<1, 1>>>(d_n);
  const cudaError_t e = cudaMemcpy(&h_n, d_n, sizeof(unsigned), cudaMemcpyDeviceToHost);
  cudaFree(d_n);
  if (e != cudaSuccess) return set_error(POLAR_ECUDA, "init: %s", cudaGetErrorString(e));
  if (h_n == 0 || h_n > 1024) return set_error(POLAR_ECUDA, "init: implausible %%nsmid = %u", h_n);
  void *p = nullptr;
  if (cudaMalloc(&p, (size_t)h_n * kScScratchPerSm) != cudaSuccess) {
    (void)cudaGetLastError();
    return set_error(POLAR_ENOMEM, "init: cudaMalloc of the %zu-byte SC stage scratch failed", (size_t)h_n * kScScratchPerSm);
  }
  g_scr_buf[device].store((float *)p, std::memory_order_release);
  return POLAR_OK;
}
float *sc_scratch() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  return g_scr_buf[dev].load(std::memory_order_acquire);
}
#endif

// phase timeline of warp 0 of CTA 0 (cycles), filled only when POLAR_SC3_DBG=1 (tools/perf_probe.py):
// 0 descents from the channel, 1 descents from the scratch, 2 tensor-memory steps, 3 128-leaf subtrees, 4 merges, 5 outputs, 6 total, 7 batches
__device__ unsigned long long g_sc5_dbg[8];

namespace {

constexpr unsigned FULLMASK = 0xFFFFFFFFu;
constexpr int kSlotFloats = 1024, kSlotBytes = 4096;
constexpr int kSlots = 6;            // at most: 4 = the warp's own stage-7 buffer (dead during a descent), 6 where spare shared memory allows
constexpr int kHeaderBytes = 1024;   // + frozen mask words and block flags for n > 1024 (sc5_layout)

#define SC5_T(slot)                                                                   \
  do {                                                                                \
    if (DBG && threadIdx.x == 0 && blockIdx.x == 0) {                                 \
      const long long t__ = clock64(); g_sc5_dbg[slot] += (unsigned long long)(t__ - tlast); tlast = t__; \
    }                                                                                 \
  } while (0)

struct Ctl {                        // control block (start of shared memory)
  unsigned long long bar[8 * kSlots];   // mbarrier of staging slot j of warp w at [kSlots w + j]
  uint32_t tm_addr;                 // tcgen05.alloc result
  uint32_t pad[3];
};
static_assert(sizeof(Ctl) + 128 + 8 <= kHeaderBytes, "sc5: header");

struct Sc5Layout {
  int nw, nws, n64, stride, slots;
  size_t fmask_off, nz_off, warp_off, per_warp, beta_off, total;
};
__host__ __device__ inline Sc5Layout sc5_layout(int m, int warps, int slots) {
  Sc5Layout l;
  const int n = 1 << m;
  l.nw = n >> 5; l.nws = l.nw + 1; l.n64 = n >> 7; l.slots = slots;
  l.stride = 128 + 4;                                   // stage-7 row of a codeword; stride/4 is odd
  l.fmask_off = (sizeof(Ctl) + 15) / 16 * 16;
  l.nz_off = l.fmask_off + (size_t)l.nw * 4;
  l.warp_off = (l.nz_off + (size_t)l.n64 + 1023) / 1024 * 1024;
  // per-warp region: staging slots (the first 32 x 132 floats double as the stage-7 rows), then the partial sums
  l.beta_off = (size_t)slots * kSlotBytes > (size_t)32 * l.stride * 4 ? (size_t)slots * kSlotBytes : (size_t)32 * l.stride * 4;
  l.per_warp = (l.beta_off + (size_t)32 * l.nws * 4 + 127) / 128 * 128;
  l.total = l.warp_off + (size_t)warps * l.per_warp;
  return l;
}

// ---- small PTX wrappers ---------------------------------------------------------------------------------------
PDEV uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
PDEV void mbar_init(unsigned long long *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
PDEV void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
PDEV void mbar_wait(unsigned long long *bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "SC5_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
      "@P1 bra SC5_DONE;\n\t"
      "bra SC5_WAIT;\n\t"
      "SC5_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
}
PDEV void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
PDEV uint64_t l2_policy_evict_last() {
  uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p;
}
PDEV uint64_t l2_policy_evict_first() {
  uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p;
}
PDEV uint64_t l2_policy_evict_normal() {
  uint64_t p; asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p)); return p;
}
PDEV void stg4_hint(float *p, const float4 v, uint64_t policy) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;"
               ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(policy) : "memory");
}
PDEV float4 lds4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
PDEV void sts4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }
PDEV float4 f4(const float4 a, const float4 b) {
  float4 o;
  o.x = f_minsum(a.x, b.x); o.y = f_minsum(a.y, b.y); o.z = f_minsum(a.z, b.z); o.w = f_minsum(a.w, b.w);
  return o;
}
PDEV float4 f4nc(const float4 a, const float4 b) {        // inputs are outputs of f: already inside [-30, 30]
  float4 o;
  o.x = f_minsum_noclip(a.x, b.x); o.y = f_minsum_noclip(a.y, b.y); o.z = f_minsum_noclip(a.z, b.z); o.w = f_minsum_noclip(a.w, b.w);
  return o;
}
PDEV float4 f4neg(const float4 a, const float4 b) {       // f on logits (LLR = -logit, polar_sc.py:122)
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
PDEV float gneg(float a, float b, uint32_t signmask) { return u2f(f2u(a) ^ signmask ^ 0x80000000u) - b; }   // g(-a, -b, u)
PDEV float4 g4neg(const float4 a, const float4 b, const uint32_t bits) {
  float4 o;
  o.x = gneg(a.x, b.x, (bits << 31) & 0x80000000u);
  o.y = gneg(a.y, b.y, (bits << 30) & 0x80000000u);
  o.z = gneg(a.z, b.z, (bits << 29) & 0x80000000u);
  o.w = gneg(a.w, b.w, (bits << 28) & 0x80000000u);
  return o;
}

// ---- tensor memory as per-thread scratch (32x32b: lane l of the warp owns TMEM lane base+l) ----------------------
PDEV void tmem_st8(uint32_t taddr, const float4 a, const float4 b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(f2u(a.x)), "r"(f2u(a.y)), "r"(f2u(a.z)), "r"(f2u(a.w)), "r"(f2u(b.x)), "r"(f2u(b.y)),
               "r"(f2u(b.z)), "r"(f2u(b.w)) : "memory");
}
PDEV void tmem_st4(uint32_t taddr, const float4 a) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(f2u(a.x)), "r"(f2u(a.y)), "r"(f2u(a.z)), "r"(f2u(a.w)) : "memory");
}
PDEV void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
struct Tm16 { uint32_t r[16]; };    // 16 columns = the stage-8 pairs of two consecutive codewords
PDEV void tmem_ld16_issue(uint32_t taddr, Tm16 &v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(v.r[0]), "=r"(v.r[1]), "=r"(v.r[2]), "=r"(v.r[3]), "=r"(v.r[4]), "=r"(v.r[5]), "=r"(v.r[6]), "=r"(v.r[7]),
                 "=r"(v.r[8]), "=r"(v.r[9]), "=r"(v.r[10]), "=r"(v.r[11]), "=r"(v.r[12]), "=r"(v.r[13]), "=r"(v.r[14]), "=r"(v.r[15])
               : "r"(taddr) : "memory");
}
PDEV void tmem_ld_wait_all() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
PDEV void tmem_tie(Tm16 &v) {      // after tmem_ld_wait_all(): keeps every use of v behind the wait (volatile asm keeps its order)
  asm volatile(""
               : "+r"(v.r[0]), "+r"(v.r[1]), "+r"(v.r[2]), "+r"(v.r[3]), "+r"(v.r[4]), "+r"(v.r[5]), "+r"(v.r[6]), "+r"(v.r[7]),
                 "+r"(v.r[8]), "+r"(v.r[9]), "+r"(v.r[10]), "+r"(v.r[11]), "+r"(v.r[12]), "+r"(v.r[13]), "+r"(v.r[14]), "+r"(v.r[15]));
}

// ---- staging ------------------------------------------------------------------------------------------------------
// While a warp runs a descent its own stage-7 buffer is dead (it is rewritten by the tensor-memory step that follows), so
// it serves as kSlots = 4 staging slots of 4 KB: 16 KB of bulk copies in flight per descending warp, no sharing, no
// atomics.  (A pool of extra slots in the CTA's spare shared memory, shared by the warps, was measured and removed: with
// 2 or 4 more slots per warp the passes were SLOWER -- the memory system, not the number of requests in flight, bounds
// them.)  Each slot has its own mbarrier; `par` holds the parity its next completion will have, kept by the warp across
// descents.
//
// Fused descent (file header).  D = stages between the source (stage 8 + D: channel row or scratch node) and the stage-8
// node that ends in tensor memory; FIRST_G: the first update is g with the partial sums of the left sibling (entering a
// right child), else f (root); FROM_CH: the source is the channel (logits = -LLR, rows past `nvalid` repeat the last one).
// Sub-unit of the staging stream = one 4 KB slot:
//   D == 1: the source nodes (512 floats) of TWO consecutive codewords (they are adjacent in the scratch);
//   D == 2: the whole source node of one codeword; lane l owns columns {4l..4l+3} and {4l+128..} of every 256-column block;
//   D >= 3: one half h of the 256 columns (lane l: columns 128h + 4l..+3) of 8 source blocks {4q+r, 2^(D-1)+4q+r : r < 4}
//           of one codeword -- exactly the operands of the first update of 4 blocks -- gathered by 8 bulk copies of 512 B.
// A step consumes TWO slots so that several independent dependency chains are in flight between the barrier wait and the
// stores: the warp shares its scheduler with one other warp only.
// Scratch of stage t (9 <= t < 8 + D) for this warp: scr + 32 (2^t - 512) + c 2^t  (c = codeword in the batch).
// All addresses that advance with the codeword are kept as running pointers (the first version recomputed them per use
// and spent more integer instructions on that than on the f / g arithmetic).
template <int D, bool FIRST_G, bool FROM_CH, int NS>
__device__ __noinline__ void descent(const float *__restrict__ src, const int nvalid, const uint32_t *beta, const int nws,
                                     const int left_word, float *scr, const uint32_t tm_base, float *Lw, const uint32_t bar_a,
                                     uint32_t &par, const int lane, const bool discard) {
  constexpr int NB = 1 << D;                       // 256-column source blocks per codeword
  constexpr int HB = NB / 2;                       // blocks of the stage 8+D-1 node
  constexpr int SRC = 256 * NB;                    // floats per codeword in the source
  constexpr bool WIDE = D <= 2;                    // whole node(s) per slot
  constexpr int CPS = D == 1 ? 2 : 1;              // codewords per slot (WIDE)
  constexpr int NQ = WIDE ? 1 : (1 << (D - 3));    // steps per codeword (D >= 3)
  constexpr int K = WIDE ? 32 / CPS : 64 * NQ;     // slots per pass
  constexpr int T1 = 8 + D - 1;                    // stage of the node the first update produces
  // channel rows are streamed (nobody comes back within the L2's reach); a scratch node must stay in the L2 until the
  // discard that follows its only read -- reading it evict_first would get the dirty line written back before that
  const uint64_t pol_src = FROM_CH ? l2_policy_evict_first() : (D == 1 ? l2_policy_evict_last() : l2_policy_evict_normal());
  const uint64_t pol_s9 = l2_policy_evict_last(), pol_sx = l2_policy_evict_normal();
  if (!FROM_CH) asm volatile("fence.proxy.async.global;" ::: "memory");   // generic-proxy scratch writes -> bulk-copy reads
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");            // the stage-7 buffer (generic writes) becomes staging space
  __syncwarp();
  const uint32_t slot_a = smem_u32(Lw);
  // `par` is a reference into the caller's stack frame (this function is not inlined): read through it, every slot wait
  // of a step reloads it from local memory, with L1 almost all carved out as shared memory.  The whole-node loops keep a
  // register copy; the D >= 3 loop (n >= 2048) keeps the reference: its copy spills in the boxplus build at n = 8192.
  uint32_t par_reg = par;
  uint32_t &pr = WIDE ? par_reg : par;

  // refill slots ring, ring+1 (ring in {0, 2, ..}) with sub-units k, k+1 (all lanes call it)
  auto issue2 = [&](const int k, const int ring) {
    if (WIDE) {
      if (lane < 2) {
        const int s = ring + lane;
        int c = (k + lane) * CPS;
        if (FROM_CH && c >= nvalid) c = nvalid - 1;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a + 8 * s), "r"(4096) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                     ::"r"(slot_a + 4096 * s), "l"(src + (size_t)c * SRC), "r"(4096), "r"(bar_a + 8 * s), "l"(pol_src) : "memory");
      }
    } else {
      if (lane < 2)
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a + 8 * (ring + lane)), "r"(4096) : "memory");
      __syncwarp();
      if (lane < 16) {                               // lanes 0..7: the 8 pieces of sub-unit k (h = 0), 8..15: of k+1 (h = 1)
        const int h = lane >> 3, p = lane & 7, s = ring + h;
        int c = k / (2 * NQ);
        const int q = (k >> 1) % NQ;
        if (FROM_CH && c >= nvalid) c = nvalid - 1;
        const int blk = (p & 3) + 4 * q + ((p >> 2) ? HB : 0);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                     ::"r"(slot_a + 4096 * s + 512 * p), "l"(src + (size_t)c * SRC + blk * 256 + h * 128), "r"(512), "r"(bar_a + 8 * s),
                     "l"(pol_src) : "memory");
      }
    }
  };
  auto wait = [&](const int s) -> const float * {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "SC5_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
        "@P1 bra SC5_DONE;\n\t"
        "bra SC5_WAIT;\n\t"
        "SC5_DONE:\n\t"
        "}" ::"r"(bar_a + 8 * s), "r"((pr >> s) & 1u), "r"(0x989680u) : "memory");
    return Lw + s * kSlotFloats;
  };

#pragma unroll
  for (int r = 0; r < NS; r += 2) issue2(r, r);
  int ring = 0;
  const int col = 4 * lane;                                            // this lane's columns: col .. col+3 (+128 for the upper half)
  float *st1 = scr + (size_t)32 * ((1 << T1) - 512) + col;            // stage T1 scratch, advances by one codeword per unit
  const uint32_t *bp = beta + left_word + (col >> 5);                   // partial sums of the left sibling, word of column `col`
  const int sh = col & 31;                                              // (columns col and col+128 share the bit position)
  const float *dp = src + lane * 32;                                    // discard cursor (scratch sources only)
  if constexpr (WIDE) {
    constexpr int CW = 2 * CPS;                      // codewords per step
    int tcol = 0;                                    // tensor-memory column of the step's first codeword
#pragma unroll 1
    for (int k = 0; k < K; k += 2) {
      const float *sl[2];
      sl[0] = wait(ring); sl[1] = wait(ring + 1);
      float4 v[CW][2][NB];
#pragma unroll
      for (int u = 0; u < CW; ++u)
#pragma unroll
        for (int e = 0; e < 2; ++e)
#pragma unroll
          for (int i = 0; i < NB; ++i) v[u][e][i] = lds4(sl[u / CPS] + (u % CPS) * SRC + i * 256 + col + 128 * e);
      float4 out[CW][2];
#pragma unroll
      for (int u = 0; u < CW; ++u) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          float4 r1[HB];
#pragma unroll
          for (int i = 0; i < HB; ++i) {
            if (FIRST_G) {
              const uint32_t bits = bp[u * nws + i * 8 + e * 4] >> sh;
              r1[i] = FROM_CH ? g4neg(v[u][e][i], v[u][e][i + HB], bits) : g4(v[u][e][i], v[u][e][i + HB], bits);
            } else {
              r1[i] = FROM_CH ? f4neg(v[u][e][i], v[u][e][i + HB]) : f4(v[u][e][i], v[u][e][i + HB]);
            }
            if (D >= 2) stg4_hint(st1 + u * (1 << T1) + i * 256 + e * 128, r1[i], T1 == 9 ? pol_s9 : pol_sx);
          }
          if (D == 2) out[u][e] = FIRST_G ? f4(r1[0], r1[HB - 1]) : f4nc(r1[0], r1[HB - 1]);
          else out[u][e] = r1[0];
        }
      }
      if (!FROM_CH && discard) {                       // consumed scratch lines never need to reach HBM: 2 x 4 KB = 64 lines
        asm volatile("discard.global.L2 [%0], 128;" ::"l"(dp) : "memory");
        asm volatile("discard.global.L2 [%0], 128;" ::"l"(dp + 1024) : "memory");
      }
      st1 += CW << T1; bp += CW * nws; dp += 2048;
      __syncwarp();                                    // every lane has consumed both slots
      pr ^= 3u << ring;
      if (k + NS < K) issue2(k + NS, ring);
#pragma unroll
      for (int u = 0; u < CW; ++u) tmem_st8(tm_base + tcol + 8 * u, out[u][0], out[u][1]);
      tcol += 8 * CW;
      ring = (ring + 2 == NS) ? 0 : ring + 2;
    }
  } else {
    const int piece = (lane >> 2) & 7, line = lane & 3;                  // discard: 2 x 8 pieces x 4 lines, two lines per lane
    dp = src + ((piece & 3) + ((piece >> 2) ? HB : 0)) * 256 + line * 32;
#pragma unroll 1
    for (int c = 0; c < 32; ++c) {
      float4 R[2][HB];                                 // [column half][block of the stage 8+D-1 node]
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        const int k = (c * NQ + q) * 2;
        const float *sl[2];
        sl[0] = wait(ring); sl[1] = wait(ring + 1);
        float4 v[2][8];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int p = 0; p < 8; ++p) v[h][p] = lds4(sl[h] + p * 128 + col);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int blk = 4 * q + t;
            if (FIRST_G) {
              const uint32_t bits = bp[blk * 8 + h * 4] >> sh;
              R[h][blk] = FROM_CH ? g4neg(v[h][t], v[h][4 + t], bits) : g4(v[h][t], v[h][4 + t], bits);
            } else {
              R[h][blk] = FROM_CH ? f4neg(v[h][t], v[h][4 + t]) : f4(v[h][t], v[h][4 + t]);
            }
            stg4_hint(st1 + blk * 256 + h * 128, R[h][blk], T1 == 9 ? pol_s9 : pol_sx);
          }
        }
        if (!FROM_CH && discard) {
          asm volatile("discard.global.L2 [%0], 128;" ::"l"(dp + 4 * q * 256) : "memory");
          asm volatile("discard.global.L2 [%0], 128;" ::"l"(dp + 4 * q * 256 + 128) : "memory");
        }
        __syncwarp();
        pr ^= 3u << ring;
        if (k + NS < K) issue2(k + NS, ring);
        ring = (ring + 2 == NS) ? 0 : ring + 2;
      }
      // the rest of the left spine in registers: stage 8+D-1 -> ... -> 8; only the first of these f's can see inputs
      // outside [-30, 30] (outputs of g); everything below consumes outputs of f
#pragma unroll
      for (int lv = D - 1; lv >= 1; --lv) {
        const int half = 1 << (lv - 1);
        float *stl = scr + (size_t)32 * ((1 << (8 + lv - 1)) - 512) + (size_t)c * (1 << (8 + lv - 1)) + col;
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int i = 0; i < half; ++i) {
            R[h][i] = (FIRST_G && lv == D - 1) ? f4(R[h][i], R[h][i + half]) : f4nc(R[h][i], R[h][i + half]);
            if (lv - 1 >= 1) stg4_hint(stl + i * 256 + h * 128, R[h][i], (8 + lv - 1) == 9 ? pol_s9 : pol_sx);
          }
      }
      tmem_st8(tm_base + 8 * c, R[0][0], R[1][0]);
      st1 += 1 << T1; bp += nws; dp += SRC;
    }
  }
  if (WIDE) par = par_reg;
  tmem_wait_st();
  __syncwarp();
}

// stage 8 (tensor memory, lane-private pairs) -> stage 7 in shared memory: f, or g with the partial sums of block i-1
template <bool IS_G>
PDEV void step_tmem(float *L, const uint32_t *beta, const int stride, const int nws, const int lane, const uint32_t tm_base,
                    const int left_word) {
  // 128 outputs per codeword = 32 float4; codeword k, lane = float4 column.  Two register sets of G = 4 codewords (two
  // 32x32b.x16 loads each): tcgen05.wait::ld waits for every load issued before it, so the loads of the next set are
  // issued right AFTER the wait for this one and fly while its codewords are computed.  The g pass reads the partial-sum
  // bits of a set together with its loads -- read per codeword, each read queued behind the previous codeword's store and
  // the whole g chain waited on it.  (Sets of 8: the pass is as short, the kernel 1.4 % slower -- 200 more instructions.)
  constexpr int G = 4;
  const int j = lane << 2;
  const uint32_t *bp = beta + left_word + (j >> 5);
  const int sh = j & 31;
  float *dst = L + j;
  Tm16 a[G / 2], b[G / 2];
  uint32_t ba[G], bb[G];
  auto issue = [&](const int k0, Tm16 (&v)[G / 2], uint32_t (&bits)[G]) {
#pragma unroll
    for (int q = 0; q < G / 2; ++q) tmem_ld16_issue(tm_base + 8 * (k0 + 2 * q), v[q]);
    if (IS_G) {
#pragma unroll
      for (int r = 0; r < G; ++r) bits[r] = bp[(k0 + r) * nws] >> sh;
    }
  };
  auto wait = [&](Tm16 (&v)[G / 2]) {
    tmem_ld_wait_all();
#pragma unroll
    for (int q = 0; q < G / 2; ++q) tmem_tie(v[q]);
  };
  auto compute = [&](const int k0, const Tm16 (&v)[G / 2], const uint32_t (&bits)[G]) {
#pragma unroll
    for (int r = 0; r < G; ++r) {
      const uint32_t *w = v[r >> 1].r + 8 * (r & 1);
      const float4 x = make_float4(u2f(w[0]), u2f(w[1]), u2f(w[2]), u2f(w[3]));
      const float4 y = make_float4(u2f(w[4]), u2f(w[5]), u2f(w[6]), u2f(w[7]));
      sts4(dst + (k0 + r) * stride, IS_G ? g4(x, y, bits[r]) : f4(x, y));
    }
  };
  issue(0, a, ba);
#pragma unroll 1
  for (int k0 = 0; k0 < 32; k0 += 2 * G) {
    wait(a);
    issue(k0 + G, b, bb);
    compute(k0, a, ba);
    wait(b);
    if (k0 + 2 * G < 32) issue(k0 + 2 * G, a, ba);
    compute(k0 + G, b, bb);
  }
}

// the 128-leaf subtree below the lane's stage-7 node: both 64-leaf halves in registers (see polar_sc4.cu)
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

// DBG: the per-phase timeline of warp 0 of CTA 0 (POLAR_SC3_DBG=1); a separate instantiation, so the product kernel carries
// none of the timer code (the block loop is sensitive to every instruction it does not need)
template <int M, int NS, bool DBG>
__global__ void __launch_bounds__(256, 1) sc5_kernel(const float *__restrict__ logit, const uint32_t *__restrict__ fmask_g,
                                                     int64_t B, int64_t nbatches, float *scratch, size_t scratch_per_sm,
                                                     int scr_discard, uint32_t *__restrict__ u_packed, float *__restrict__ u_info,
                                                     const int32_t *__restrict__ info_pos, int k) {
  static_assert(M >= 10 && M <= 13, "sc5: n = 1024 .. 8192");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int N = 1 << M, NW = N >> 5, NWS = NW + 1, N64 = N >> 7, stride = 132;
  // warp index and everything derived from the frozen pattern go through a lane-0 broadcast: the values are warp
  // uniform anyway, but only the shuffle lets the compiler KNOW it -- branches on them become uniform branches instead of
  // potentially divergent ones that need a convergence barrier each (the 128-leaf subtree nests a dozen of them; when the
  // barrier registers run out the compiler spills them with BMOV and the subtree phase gets 1.5x slower)
  const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(FULLMASK, tid >> 5, 0), nwarps = blockDim.x >> 5;
  Sc5Layout lay = sc5_layout(M, nwarps, NS);
  Ctl *P = reinterpret_cast<Ctl *>(smem_raw);
  uint32_t *fmask = reinterpret_cast<uint32_t *>(smem_raw + lay.fmask_off);
  unsigned char *nz = smem_raw + lay.nz_off;            // nz[i]: 128-leaf block i is rate-0
  float *L = reinterpret_cast<float *>(smem_raw + lay.warp_off + (size_t)warp * lay.per_warp);
  uint32_t *beta = reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(L) + lay.beta_off);
  const uint32_t bar_a = smem_u32(&P->bar[kSlots * warp]);   // this warp's four slot barriers
  uint32_t par = 0;                                          // parity the next completion of each will have

  if (warp == 0) {          // the CTA is alone on its SM (shared memory): take all 512 tensor-memory columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(&P->tm_addr)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    for (int s = 0; s < 8 * kSlots; ++s) mbar_init(&P->bar[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  for (int i = tid; i < NW; i += blockDim.x) fmask[i] = __ldg(fmask_g + i);
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  // warp w: TMEM lanes 32(w%4)..+31 (the only ones it can address), column block w/4 (256 columns: the stage-8 node)
  const uint32_t tm_base = P->tm_addr + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * 256);
  for (int i = tid; i < N64; i += blockDim.x)
    nz[i] = (fmask[4 * i] & fmask[4 * i + 1] & fmask[4 * i + 2] & fmask[4 * i + 3]) == FULLMASK;
  __syncthreads();

  // per-warp scratch for stages 9 .. M-1, indexed by the PHYSICAL SM (only one CTA of this kernel fits on an SM, so
  // concurrent launches on other streams can never share a slot)
  uint32_t smid;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
  float *scr = scratch + (size_t)smid * (scratch_per_sm / 4) + (size_t)warp * 32 * (N - 512);
  long long tlast = DBG ? clock64() : 0;
  const long long tstart = tlast;
  const int64_t wstride = (int64_t)gridDim.x * nwarps;
  for (int64_t batch = (int64_t)warp * gridDim.x + blockIdx.x; batch < nbatches; batch += wstride) {
    const int64_t cw0 = batch * 32;
    const int nvalid = (int)((B - cw0) < 32 ? (B - cw0) : 32);
#pragma unroll 1
    for (int i = 0; i < N64; ++i) {               // 128-leaf blocks, left to right
      const bool zero_blk = __shfl_sync(FULLMASK, (int)nz[i], 0) != 0;      // warp uniform, and known to be
      if ((i & 1) == 0) {
        // a new stage-8 node starts here.  S = stage of the node entered at block i (the root, or the right child whose left
        // sibling has just finished); nodes of stage >= 8 are always materialised (rate-0 is only exploited per block)
        const int S = (i == 0) ? M : 7 + (__ffs(i) - 1);
        const bool dead = __shfl_sync(FULLMASK, (int)(nz[i] & nz[i + 1]), 0) != 0;       // nobody will read this stage-8 node
        if (S == M) {
          descent<M - 8, false, true, NS>(logit + cw0 * (int64_t)N, nvalid, beta, NWS, 0, scr, tm_base, L, bar_a, par, lane, false);
        } else if (S == M - 1) {
          descent<M - 8, true, true, NS>(logit + cw0 * (int64_t)N, nvalid, beta, NWS, 0, scr, tm_base, L, bar_a, par, lane, false);
        } else {
          const int left_word = 4 * (i - (1 << (S - 7)));      // the left sibling's partial sums start at that block
          const float *sp = scr + (size_t)32 * ((1 << (S + 1)) - 512);
          const bool dis = scr_discard != 0;
          switch (S) {                                         // source = scratch node of stage S+1, D = S+1-8
            case 8: if (!dead) descent<1, true, false, NS>(sp, 32, beta, NWS, left_word, scr, tm_base, L, bar_a, par, lane, dis); break;
            case 9: if (M > 10) descent<(M > 10 ? 2 : 1), true, false, NS>(sp, 32, beta, NWS, left_word, scr, tm_base, L, bar_a, par, lane, dis); break;
            case 10: if (M > 11) descent<(M > 11 ? 3 : 1), true, false, NS>(sp, 32, beta, NWS, left_word, scr, tm_base, L, bar_a, par, lane, dis); break;
            case 11: if (M > 12) descent<(M > 12 ? 4 : 1), true, false, NS>(sp, 32, beta, NWS, left_word, scr, tm_base, L, bar_a, par, lane, dis); break;
            default: break;
          }
        }
        __syncwarp();
        if (S >= M - 1) SC5_T(0); else SC5_T(1);
        if (!zero_blk) {
          step_tmem<false>(L, beta, stride, NWS, lane, tm_base, 0);
          __syncwarp();
        }
        SC5_T(2);
      } else if (!zero_blk) {
        step_tmem<true>(L, beta, stride, NWS, lane, tm_base, 4 * (i - 1));
        __syncwarp();
        SC5_T(2);
      }
      if (zero_blk) {
        for (int q = lane; q < 128; q += 32) beta[(q >> 2) * NWS + 4 * i + (q & 3)] = 0u;
      } else {
        const uint32_t *fmw = fmask + 4 * i;
        const uint32_t f0 = __shfl_sync(FULLMASK, fmw[0], 0), f1 = __shfl_sync(FULLMASK, fmw[1], 0);
        const uint32_t f2 = __shfl_sync(FULLMASK, fmw[2], 0), f3 = __shfl_sync(FULLMASK, fmw[3], 0);
        const uint4 b = bottom128(L + lane * stride, (uint64_t)f0 | ((uint64_t)f1 << 32), (uint64_t)f2 | ((uint64_t)f3 << 32));
        uint32_t *bp = beta + lane * NWS + 4 * i;
        bp[0] = b.x; bp[1] = b.y; bp[2] = b.z; bp[3] = b.w;
      }
      __syncwarp();
      SC5_T(3);
      {  // merge partial sums upward while the finished node is a right child: [bl ^ br, br] (polar_sc.py:83-89).
         // Lane c owns the partial-sum row of codeword c (odd row stride: conflict free); the cooperative readers (g bits
         // of the tensor-memory steps and the descents) come after the __syncwarp below.
        uint32_t *bw = beta + lane * NWS;
        int lv = 0, a = i;
        while (lv < M - 7 && ((a >> lv) & 1)) {
          const int nwd = 4 << lv, left = a - (1 << lv);
#pragma unroll 1
          for (int w = 0; w < nwd; w += 4) {          // loads first: the compiler cannot prove the two ranges distinct
            const uint32_t r0 = bw[4 * a + w], r1 = bw[4 * a + w + 1], r2 = bw[4 * a + w + 2], r3 = bw[4 * a + w + 3];
            const uint32_t l0 = bw[4 * left + w], l1 = bw[4 * left + w + 1], l2 = bw[4 * left + w + 2], l3 = bw[4 * left + w + 3];
            bw[4 * left + w] = l0 ^ r0; bw[4 * left + w + 1] = l1 ^ r1; bw[4 * left + w + 2] = l2 ^ r2; bw[4 * left + w + 3] = l3 ^ r3;
          }
          a = left; ++lv;
        }
        __syncwarp();
      }
      SC5_T(4);
    }
    // beta now holds the re-encoded codeword x_hat of every codeword; the decisions are u = T(x_hat)
    // (my_sn/fec/polar/enc.py:85-96 is an involution): 5 stages inside each word, M-5 across words.
    if constexpr (NW <= 64) {
      // lane c transforms the row of codeword c entirely in registers and writes its NW words itself
      uint32_t *bw = beta + lane * NWS;
      uint32_t w[NW];
#pragma unroll
      for (int t = 0; t < NW; ++t) w[t] = ptransform<5>(bw[t]);
#pragma unroll
      for (int st = 0; st < M - 5; ++st)
#pragma unroll
        for (int t = 0; t < NW; ++t)
          if (!(t & (1 << st))) w[t] ^= w[t + (1 << st)];
      if (u_packed && lane < nvalid) {
        uint32_t *dst = u_packed + (cw0 + lane) * NW;
        if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
          for (int t = 0; t < NW; t += 4) __stcs(reinterpret_cast<uint4 *>(dst + t), make_uint4(w[t], w[t + 1], w[t + 2], w[t + 3]));
        } else {
#pragma unroll
          for (int t = 0; t < NW; ++t) dst[t] = w[t];
        }
      }
      if (u_info) {
#pragma unroll
        for (int t = 0; t < NW; ++t) bw[t] = w[t];
      }
      __syncwarp();
    } else {
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
    }
    if (u_info) {
      // the API tensor [B, k] fp32 (polar_sc.py:127-133): a codeword's row at a time, one float4 per lane and round
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
    SC5_T(5);
    if (DBG && tid == 0 && blockIdx.x == 0) g_sc5_dbg[7] += 1;
  }
  if (DBG && tid == 0 && blockIdx.x == 0) g_sc5_dbg[6] += (unsigned long long)(clock64() - tstart);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(P->tm_addr), "n"(512) : "memory");
}

template <int M>
int launch_sc5_t(const float *logit, const uint32_t *fmask, int64_t B, uint32_t *u_packed, float *u_info,
                 const int32_t *info_pos, int k, int warps, cudaStream_t st) {
  const int max_smem = device_max_smem_optin();
  constexpr int N = 1 << M;
  int wmax = 8;                                         // tensor memory: 256 columns per warp, 512 per lane quarter
  if (warps <= 0 || warps > wmax) warps = wmax;
  while (warps > 1 && (sc5_layout(M, warps, 4).total > (size_t)max_smem ||
                       (size_t)warps * 32 * (N - 512) * 4 > kScScratchPerSm)) --warps;
  int ns = env_int("POLAR_SC5_SLOTS", 6);               // staging slots per warp: 6 where the spare shared memory allows
  if (ns != 6 || sc5_layout(M, warps, 6).total > (size_t)max_smem) ns = 4;
  const Sc5Layout lay = sc5_layout(M, warps, ns);
  if (lay.total > (size_t)max_smem) return set_error(POLAR_ENOMEM, "sc: n=%d needs more shared memory per CTA than the device has", N);
  float *scratch = sc_scratch();
  if (!scratch)
    return set_error(POLAR_EINVAL, "sc: n=%d needs the per-device stage scratch -- call polar_init(device) once before decoding", N);
  const bool dbg = env_int("POLAR_SC3_DBG", 0) != 0;
  auto kern = dbg ? (ns == 6 ? sc5_kernel<M, 6, true> : sc5_kernel<M, 4, true>) : (ns == 6 ? sc5_kernel<M, 6, false> : sc5_kernel<M, 4, false>);
  // one persistent CTA per SM: it takes all 512 tensor-memory columns, so a second CTA must never become resident on the
  // same SM: the shared-memory request is padded above half of the SM's
  size_t smem = lay.total;
  if (smem < (size_t)116 * 1024) smem = (size_t)116 * 1024;
  POLAR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int sms = device_sm_count();
  const int64_t nbatches = (B + 31) / 32;
  int64_t grid = (nbatches + warps - 1) / warps;
  if (grid > sms) grid = sms;
  if (grid < 1) grid = 1;
  kern<<<(unsigned)grid, warps * 32, smem, st>>>(logit, fmask, B, nbatches, scratch,
                                              // slots packed back to back: what this launch uses is one dense range (76 MB for
                                              // n = 1024, L2 resident); a sparse 4 MB stride made the L2 write every line back
                                              (size_t)warps * 32 * (N - 512) * 4,
                                                      env_int("POLAR_SC4_DISCARD", 1), u_packed, u_info, info_pos, k);
  count_launch();
  POLAR_CHECK_LAUNCH("sc5_kernel");
  return POLAR_OK;
}

}  // namespace

// n in [1024, 8192].  warps = autonomous warps per SM (0 = as many as shared memory and the scratch slot hold).
int launch_sc5(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
               const int32_t *info_pos, int k, int warps, cudaStream_t st) {
  switch (ilog2(n)) {
    case 10: return launch_sc5_t<10>(logit, fmask, B, u_packed, u_info, info_pos, k, warps, st);
    case 11: return launch_sc5_t<11>(logit, fmask, B, u_packed, u_info, info_pos, k, warps, st);
    case 12: return launch_sc5_t<12>(logit, fmask, B, u_packed, u_info, info_pos, k, warps, st);
    case 13: return launch_sc5_t<13>(logit, fmask, B, u_packed, u_info, info_pos, k, warps, st);
    default: return set_error(POLAR_EINVAL, "sc5: n=%d not supported by this mapping", n);
  }
}

}  // namespace polar

// debug only (not part of include/polar_b200.h): read and clear the phase timeline of warp 0 of CTA 0
extern "C" int polar_sc5_debug_read(unsigned long long *h_out8) {
  unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (cudaMemcpyFromSymbol(h_out8, polar::g_sc5_dbg, sizeof(z)) != cudaSuccess) return POLAR_ECUDA;
  if (cudaMemcpyToSymbol(polar::g_sc5_dbg, z, sizeof(z)) != cudaSuccess) return POLAR_ECUDA;
  return POLAR_OK;
}
