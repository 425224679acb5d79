// polar_count.cu -- bit / block error counters (sm_100a).
// Replaces count_errors / count_block_errors (my_sn/sim.py:7-18): sum(b != b_hat) and
// sum(any(b != b_hat, -1)).  Popcount over packed words (or a compare over the fp32 API tensors),
// per-warp accumulation in registers, one atomicAdd pair per warp at the end.
#include "polar_launch.h"

namespace polar {

constexpr int kMcGroupMax = POLAR_MC_GROUP_MAX;

__device__ __forceinline__ unsigned warp_sum(unsigned v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
  return v;
}

__global__ void __launch_bounds__(256) count_packed_kernel(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b,
                                                           const uint32_t *__restrict__ mask, int nw, int64_t B,
                                                           unsigned long long *__restrict__ counters) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  unsigned long long bit_acc = 0, blk_acc = 0;
  for (int64_t row = warp0; row < B; row += nwarps) {
    unsigned cnt = 0;
    for (int w = lane; w < nw; w += 32) {
      uint32_t d = __ldg(a + row * nw + w) ^ __ldg(b + row * nw + w);
      if (mask) d &= __ldg(mask + w);
      cnt += __popc(d);
    }
    cnt = warp_sum(cnt);
    bit_acc += cnt; blk_acc += (cnt != 0);
  }
  if (lane == 0 && (bit_acc | blk_acc)) {
    atomicAdd(counters, bit_acc);
    atomicAdd(counters + 1, blk_acc);
  }
}

// Same counters for rows of nw = 4 .. 128 words (n = 128 .. 4096): the two arrays are read as flat streams of 16-byte
// pieces, G = nw/4 consecutive lanes share a row (the one-warp-per-row version above keeps two 4-byte loads per lane in
// flight and ran at 1.5 TB/s).  The mask repeats every G pieces.
template <int G>
__global__ void __launch_bounds__(256) count_packed_vec_kernel(const uint4 *__restrict__ a, const uint4 *__restrict__ b,
                                                               const uint4 *__restrict__ mask, int64_t pieces,
                                                               unsigned long long *__restrict__ counters) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;            // a multiple of 32 >= G: a thread keeps its mask piece
  const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint4 m = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
  if (mask) m = __ldg(mask + (i0 & (G - 1)));
  unsigned long long bit_acc = 0, blk_acc = 0;
  for (int64_t base = i0 - lane; base < pieces; base += stride) {      // whole warps iterate together (shuffles below)
    const int64_t i = base + lane;
    unsigned cnt = 0;
    if (i < pieces) {
      const uint4 x = __ldg(a + i), y = __ldg(b + i);
      cnt = __popc((x.x ^ y.x) & m.x) + __popc((x.y ^ y.y) & m.y) + __popc((x.z ^ y.z) & m.z) + __popc((x.w ^ y.w) & m.w);
    }
    unsigned rowc = cnt;
#pragma unroll
    for (int d = 1; d < G; d <<= 1) rowc += __shfl_xor_sync(0xFFFFFFFFu, rowc, d);
    bit_acc += cnt;
    blk_acc += ((lane & (G - 1)) == 0 && rowc != 0);
  }
  bit_acc = warp_sum((unsigned)bit_acc);                                // < 2^32 per warp and launch: 128 bits x 2^24 pieces per lane at most
  blk_acc = warp_sum((unsigned)blk_acc);
  if (lane == 0 && (bit_acc | blk_acc)) {
    atomicAdd(counters, bit_acc);
    atomicAdd(counters + 1, blk_acc);
  }
}

__global__ void __launch_bounds__(256) count_f32_kernel(const float *__restrict__ a, const float *__restrict__ b, int k,
                                                        int64_t B, unsigned long long *__restrict__ counters) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  unsigned long long bit_acc = 0, blk_acc = 0;
  const bool vec = (k & 3) == 0 && (((uintptr_t)a | (uintptr_t)b) & 15) == 0;        // rows of float4: 128-bit loads
  for (int64_t row = warp0; row < B; row += nwarps) {
    unsigned cnt = 0;
    if (vec) {
      const float4 *pa = reinterpret_cast<const float4 *>(a + row * k), *pb = reinterpret_cast<const float4 *>(b + row * k);
      for (int t = lane; t < (k >> 2); t += 32) {
        const float4 x = __ldg(pa + t), y = __ldg(pb + t);
        cnt += (x.x != y.x) + (x.y != y.y) + (x.z != y.z) + (x.w != y.w);
      }
    } else {
      for (int t = lane; t < k; t += 32) cnt += (__ldg(a + row * k + t) != __ldg(b + row * k + t));
    }
    cnt = warp_sum(cnt);
    bit_acc += cnt; blk_acc += (cnt != 0);
  }
  if (lane == 0 && (bit_acc | blk_acc)) {
    atomicAdd(counters, bit_acc);
    atomicAdd(counters + 1, blk_acc);
  }
}

// Stop rules of sim_ber (my_sn/sim.py:90-133) evaluated on the device, one thread, for a GROUP of queued iterations that
// may span SNR points (my_sn/sim.py::sim_ber_device packs several iterations -- of one point, or of consecutive points
// that are predicted to stop -- into one decoder launch so that a small per-rank batch still fills the GPU).
// state (int64[P,8], one row per point): [0] bit errors [1] block errors [2] bits [3] blocks [4] stop flag [5] status code
// [6] iterations counted.  delta (uint64[G,4]): each iteration's (bit errors, block errors, bits, blocks), summed over
// ranks when sharded.  Once a point's stop flag is set its later iterations are ignored, so the host may enqueue
// iterations ahead of the counters.  Iteration j of the group was simulated at the noise level of point
// item.point[j] with the random numbers of sequence position expect_q + j.  It counts only if it is what the sequential
// loop (sim.py:79-133) would have run at that position: the sweep has not ended, every earlier iteration of the group
// counted, and the loop is at that point.  The first iteration that does not count ends the group (its successors sit at
// positions the loop will reach with other parameters); the host re-plans from the state it reads back.
struct McItems { int point[kMcGroupMax]; };
__global__ void mc_control_group_kernel(unsigned long long *__restrict__ delta, McItems item, int G, long long *__restrict__ state,
                                        long long *__restrict__ sweep, long long expect_q, int P, long long target_bit,
                                        long long target_block, long long max_iter, int early_stop) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  long long consumed = 0;
  if (!sweep[1] && sweep[2] == expect_q) {
    for (int j = 0; j < G; ++j) {
      const long long pc = sweep[0];
      if (pc >= P || item.point[j] != pc) break;
      long long *st = state + 8 * pc;
      st[0] += (long long)delta[4 * j]; st[1] += (long long)delta[4 * j + 1];
      st[2] += (long long)delta[4 * j + 2]; st[3] += (long long)delta[4 * j + 3];
      const long long it = ++st[6];
      ++sweep[2]; ++consumed;
      if (target_bit >= 0 && st[0] >= target_bit) { st[5] = 3; st[4] = 1; }             // sim.py:107-112
      else if (target_block >= 0 && st[1] >= target_block) { st[5] = 4; st[4] = 1; }    // sim.py:113-118
      else if (it >= max_iter) { st[5] = 1; st[4] = 1; }                                // sim.py:120-123
      if (st[4]) {
        if (early_stop && st[1] == 0) { st[5] = 2; sweep[1] = 1; break; }               // sim.py:128-133
        sweep[0] = pc + 1;
        if (pc + 1 >= P) { sweep[1] = 1; break; }
      }
    }
  }
  sweep[3] += 1; sweep[4] = consumed;
  for (int j = 0; j < 4 * G; ++j) delta[j] = 0;
}

}  // namespace polar

using namespace polar;

extern "C" int polar_mc_control_group(unsigned long long *d_delta, const int32_t *h_item_point, int n_items,
                                      long long *d_state, int n_points, long long *d_sweep8, long long expect_q,
                                      long long target_bit_errs, long long target_block_errs, long long max_mc_iter,
                                      int early_stop, void *stream) {
  if (!d_delta || !h_item_point || !d_state || !d_sweep8) return set_error(POLAR_EINVAL, "mc_control_group: null pointer");
  if (n_items < 1 || n_items > kMcGroupMax) return set_error(POLAR_EINVAL, "mc_control_group: 1 <= n_items <= %d", kMcGroupMax);
  if (max_mc_iter < 1 || n_points < 1) return set_error(POLAR_EINVAL, "mc_control_group: max_mc_iter < 1 or n_points < 1");
  McItems it;
  for (int j = 0; j < kMcGroupMax; ++j) it.point[j] = j < n_items ? h_item_point[j] : -1;
  return launch("mc_control_group", mc_control_group_kernel, 1, 32, 0, (cudaStream_t)stream, d_delta, it, n_items, d_state,
                d_sweep8, expect_q, n_points, target_bit_errs, target_block_errs, max_mc_iter, early_stop);
}

extern "C" int polar_count_errors_packed(const uint32_t *d_a, const uint32_t *d_b, const uint32_t *d_mask, int n,
                                         int64_t B, unsigned long long *d_counters, void *stream) {
  if (n < 1 || B < 0) return set_error(POLAR_EINVAL, "count: bad n/B");
  if (B == 0) return POLAR_OK;
  if (!d_a || !d_b || !d_counters) return set_error(POLAR_EINVAL, "count: null pointer");
  const int nw = POLAR_WORDS(n);
  const bool vec = nw >= 4 && nw <= 128 && ((((uintptr_t)d_a | (uintptr_t)d_b | (uintptr_t)d_mask) & 15) == 0) && B * (int64_t)nw < ((int64_t)1 << 36);
  const cudaStream_t st = (cudaStream_t)stream;
  if (vec) {
    const int64_t pieces = B * (int64_t)(nw / 4);
    const int q = nw / 4;
    const auto kern = q == 1 ? count_packed_vec_kernel<1> : q == 2 ? count_packed_vec_kernel<2> : q == 4 ? count_packed_vec_kernel<4>
                      : q == 8 ? count_packed_vec_kernel<8> : q == 16 ? count_packed_vec_kernel<16> : count_packed_vec_kernel<32>;
    return launch("count_packed", kern, grid_for(pieces, 256, 8), 256, 0, st, reinterpret_cast<const uint4 *>(d_a),
                  reinterpret_cast<const uint4 *>(d_b), reinterpret_cast<const uint4 *>(d_mask), pieces, d_counters);
  }
  return launch("count_packed", count_packed_kernel, grid_for(B, 8, 8), 256, 0, st, d_a, d_b, d_mask, nw, B, d_counters);
}

extern "C" int polar_count_errors_f32(const float *d_b, const float *d_b_hat, int k, int64_t B,
                                      unsigned long long *d_counters, void *stream) {
  if (k < 1 || B < 0) return set_error(POLAR_EINVAL, "count: bad k/B");
  if (B == 0) return POLAR_OK;
  if (!d_b || !d_b_hat || !d_counters) return set_error(POLAR_EINVAL, "count: null pointer");
  return launch("count_f32", count_f32_kernel, grid_for(B, 8, 8), 256, 0, (cudaStream_t)stream, d_b, d_b_hat, k, B, d_counters);
}
