// polar_frontend.cu -- BPSK/AWGN LLR front end (sm_100a): random info bits -> polar encode ->
// +-1/sqrt2 per real dimension -> + N(0, no/2) -> logit = -2.sqrt2.y/no.
//
// Replaces System_AWGN_model.forward up to the decoder call (z_sys_model/awgn_model.py:33-40):
// BinarySource (my_sn/trans/binary_source.py:18-19), PolarEncoder, Mapper (mapping.py:136-149: even
// code bits -> real axis, odd -> imaginary, bit 0 -> +), AWGN (awgn.py:19-29, utils.py:2-17) and the
// exact 2-point log-sum-exp Demapper (mapping.py:195-241), whose closed form is -2.sqrt2.y/no
// (SURVEY 3.2 [probe], <= 6e-6 abs).  The reference draws from torch's CPU mt19937; this kernel
// uses counter-based Philox4x32-10, so parity is statistical (BER/BLER inside confidence
// intervals), never bitwise.  One warp per codeword; 4 positions per lane per step (one Philox call
// -> two Box-Muller pairs -> one 128-bit store).  HBM-bound on the [B,n] fp32 logit write.
#include <atomic>

#include "polar_internal.h"
#include "polar_warp.cuh"

namespace polar {

constexpr uint32_t kStreamBits = 0x42495453u;   // "BITS"
constexpr uint32_t kStreamNoise = 0x4E4F4953u;  // "NOIS"

__device__ __forceinline__ float4 noisy_logits(const Philox &ph, uint64_t cw_id, uint32_t group, uint32_t bits4,
                                               float sigma, float scale) {
  const uint4 r = ph((uint32_t)cw_id, (uint32_t)(cw_id >> 32), group, kStreamNoise);
  const float2 z0 = box_muller(r.x, r.y), z1 = box_muller(r.z, r.w);
  const float amp = 0.70710678118654752f;   // QPSK point (+-1 +-1j)/sqrt2 (mapping.py:40)
  float4 o;
  o.x = scale * (((bits4 & 1u) ? -amp : amp) + sigma * z0.x);
  o.y = scale * (((bits4 & 2u) ? -amp : amp) + sigma * z0.y);
  o.z = scale * (((bits4 & 4u) ? -amp : amp) + sigma * z1.x);
  o.w = scale * (((bits4 & 8u) ? -amp : amp) + sigma * z1.y);
  return o;
}

// Binary erasure channel with LLR output (my_sn/trans/channel/discrete_channel.py:79-107, return_llrs=True): logit =
// +-llr_max for bit 1 / 0, erased to 0 with probability pe.  The reference samples the erasure pattern with a
// Gumbel-softmax pair (:53-72), i.e. a Bernoulli(pe) draw; here one Philox word per position is compared with pe.
__device__ __forceinline__ float4 erased_logits(const Philox &ph, uint64_t cw_id, uint32_t group, uint32_t bits4,
                                                float pe, float llr_max) {
  const uint4 r = ph((uint32_t)cw_id, (uint32_t)(cw_id >> 32), group, kStreamNoise);
  const float k = 2.3283064365386963e-10f;     // 2^-32: u in [0,1)
  float4 o;
  o.x = ((float)r.x * k < pe) ? 0.0f : ((bits4 & 1u) ? llr_max : -llr_max);
  o.y = ((float)r.y * k < pe) ? 0.0f : ((bits4 & 2u) ? llr_max : -llr_max);
  o.z = ((float)r.z * k < pe) ? 0.0f : ((bits4 & 4u) ? llr_max : -llr_max);
  o.w = ((float)r.w * k < pe) ? 0.0f : ((bits4 & 8u) ? llr_max : -llr_max);
  return o;
}
template <bool BEC>
__device__ __forceinline__ float4 channel_logits(const Philox &ph, uint64_t cw_id, uint32_t group, uint32_t bits4, float a,
                                                 float b) {
  return BEC ? erased_logits(ph, cw_id, group, bits4, a, b) : noisy_logits(ph, cw_id, group, bits4, a, b);
}

template <int R, bool BEC = false>
__global__ void __launch_bounds__(256) frontend_kernel(uint64_t seed, uint64_t offset, float sigma, float scale,
                                                       const uint32_t *__restrict__ fmask, int n, int m, int64_t B,
                                                       uint32_t *__restrict__ u_out, uint32_t *__restrict__ c_out,
                                                       float *__restrict__ logit) {
  const int lane = threadIdx.x & 31;
  const int nw = n < 32 ? 1 : n >> 5;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const Philox ph(seed);
  const uint32_t tail = n < 32 ? ((1u << n) - 1u) : 0xFFFFFFFFu;
  for (int64_t b = warp0; b < B; b += nwarps) {
    const uint64_t id = (uint64_t)b + offset;
    uint32_t x[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int wd = r * 32 + lane;
      uint32_t w = 0u;
      if (wd < nw) {
        // Bernoulli(1/2) info bits (binary_source.py:19); frozen positions forced to 0 (enc.py:33-35)
        const uint4 rb = ph((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)(wd >> 2), kStreamBits);
        const uint32_t rw = (wd & 3) == 0 ? rb.x : (wd & 3) == 1 ? rb.y : (wd & 3) == 2 ? rb.z : rb.w;
        w = rw & ~__ldg(fmask + wd) & tail;
        if (u_out) u_out[b * nw + wd] = w;
      }
      x[r] = w;
    }
    warp_polar_transform<R>(x, m, nw);
    if (c_out) {
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (r * 32 + lane < nw) c_out[b * nw + r * 32 + lane] = x[r];
    }
    // 4 positions per lane per step: group g covers positions 4g..4g+3, which live in word g>>3
    const int ngroups = n >> 2;
    float *row = logit + b * (int64_t)n;
    if (n >= 4) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        for (int it = 0; it < 8; ++it) {            // 8 steps x 32 lanes x 4 = 1024 positions per register row
          const int g = (r * 8 + it) * 32 + lane;
          const uint32_t w = __shfl_sync(0xFFFFFFFFu, x[r], (it * 32 + lane) >> 3);
          if (g < ngroups) {
            const uint32_t bits4 = (w >> ((4 * g) & 31)) & 0xFu;
            *reinterpret_cast<float4 *>(row + 4 * g) = channel_logits<BEC>(ph, id, (uint32_t)g, bits4, sigma, scale);
          }
        }
      }
    } else {  // n == 2
      const uint32_t w = __shfl_sync(0xFFFFFFFFu, x[0], 0);
      if (lane == 0) {
        const float4 o = channel_logits<BEC>(ph, id, 0u, w & 3u, sigma, scale);
        row[0] = o.x; row[1] = o.y;
      }
    }
  }
}

// 5G NR uplink front end (TS 38.212 5.3.1 / 5.4.1 as built by Polar5GEncoder): payload bits -> CRC -> channel
// allocation -> polar transform -> sub-block interleaver + circular buffer + channel interleaver (one gather index) ->
// QPSK/AWGN -> closed-form demapper.  One warp per codeword, n <= 1024: one 32-bit word per lane.  The codeword is
// staged in 128 B of shared memory per warp so that every channel position can read its bit through rm_idx.
// Random numbers: the payload words are the Philox words of frontend_kernel; the noise of channel group g is that of
// polar_qpsk_awgn_llr for the rate-matched codeword zero-padded to a multiple of 4.
__global__ void __launch_bounds__(256) nr5g_frontend_kernel(uint64_t seed, uint64_t offset, float sigma, float scale,
                                                            const uint32_t *__restrict__ payload_mask,
                                                            const uint32_t *__restrict__ crc_rows,
                                                            const int32_t *__restrict__ crc_pos, int crc_len,
                                                            const int32_t *__restrict__ rm_idx, int n, int m, int e,
                                                            int64_t B, uint32_t *__restrict__ u_out,
                                                            uint32_t *__restrict__ c_out, float *__restrict__ logit) {
  __shared__ uint32_t s_cw[8][32];
  const int lane = threadIdx.x & 31;
  uint32_t *cw = s_cw[threadIdx.x >> 5];
  const int nw = n >> 5, ew = (e + 31) >> 5, ngroups = (e + 3) >> 2;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const Philox ph(seed);
  // parity bit `lane` of the CRC (MSB of the syndrome word = parity bit 0) and the polar position it goes to
  const int my_crc_pos = lane < crc_len ? __ldg(crc_pos + lane) : 0;
  for (int64_t b = warp0; b < B; b += nwarps) {
    const uint64_t id = (uint64_t)b + offset;
    uint32_t w = 0u;
    if (lane < nw) {
      const uint4 rb = ph((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)(lane >> 2), kStreamBits);
      const uint32_t rw = (lane & 3) == 0 ? rb.x : (lane & 3) == 1 ? rb.y : (lane & 3) == 2 ? rb.z : rb.w;
      w = rw & __ldg(payload_mask + lane);
    }
    uint32_t syn = 0u;
    for (uint32_t t = w; t; t &= t - 1u) syn ^= __ldg(crc_rows + lane * 32 + __ffs(t) - 1);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) syn ^= __shfl_xor_sync(0xFFFFFFFFu, syn, d);
    __syncwarp();                                   // the previous codeword's channel reads are done
    cw[lane] = w;
    __syncwarp();
    if (lane < crc_len && ((syn >> (crc_len - 1 - lane)) & 1u)) atomicOr(cw + (my_crc_pos >> 5), 1u << (my_crc_pos & 31));
    __syncwarp();
    uint32_t x[1] = {cw[lane]};
    if (lane < nw) u_out[b * nw + lane] = x[0];
    warp_polar_transform<1>(x, m, nw);
    cw[lane] = x[0];
    __syncwarp();
    float *row = logit + b * (int64_t)e;
    const bool vec = ((uintptr_t)row & 15) == 0;
    for (int g0 = 0; g0 < ngroups; g0 += 32) {
      const int g = g0 + lane;
      uint32_t bits4 = 0u;
      if (g < ngroups) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int p = 4 * g + t;
          if (p < e) {
            const int i = __ldg(rm_idx + p);
            bits4 |= ((cw[i >> 5] >> (i & 31)) & 1u) << t;
          }
        }
        const float4 o = noisy_logits(ph, id, (uint32_t)g, bits4, sigma, scale);
        if (vec && 4 * g + 3 < e) {
          *reinterpret_cast<float4 *>(row + 4 * g) = o;
        } else {
          row[4 * g] = o.x;
          if (4 * g + 1 < e) row[4 * g + 1] = o.y;
          if (4 * g + 2 < e) row[4 * g + 2] = o.z;
          if (4 * g + 3 < e) row[4 * g + 3] = o.w;
        }
      }
      if (c_out) {                                  // 8 consecutive lanes hold the 32 bits of one codeword word
        uint32_t cword = bits4 << (4 * (lane & 7));
        cword |= __shfl_xor_sync(0xFFFFFFFFu, cword, 1);
        cword |= __shfl_xor_sync(0xFFFFFFFFu, cword, 2);
        cword |= __shfl_xor_sync(0xFFFFFFFFu, cword, 4);
        const int wq = g >> 3;
        if ((lane & 7) == 0 && wq < ew) c_out[b * ew + wq] = cword;
      }
    }
  }
}

// channel + demapper for caller-supplied codewords (fp32 0/1)
template <bool BEC = false>
__global__ void __launch_bounds__(256) qpsk_awgn_kernel(uint64_t seed, uint64_t offset, float sigma, float scale,
                                                        const float *__restrict__ c, int n, int64_t B,
                                                        float *__restrict__ logit) {
  const Philox ph(seed);
  const int ngroups = n >> 2;
  const int64_t total = B * (int64_t)ngroups;
  // (row, group) of the flat index, advanced without a division per element (a 64-bit division costs as much as the Philox call)
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, sb = stride / ngroups;
  const int sg = (int)(stride - sb * ngroups);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t b = i / ngroups;
  int g = (int)(i - b * ngroups);
  for (; i < total; i += stride, b += sb, g += sg) {
    if (g >= ngroups) { g -= ngroups; ++b; }
    const float4 v = __ldg(reinterpret_cast<const float4 *>(c + b * (int64_t)n) + g);
    const uint32_t bits4 = (v.x != 0.f) | ((v.y != 0.f) << 1) | ((v.z != 0.f) << 2) | ((v.w != 0.f) << 3);
    *reinterpret_cast<float4 *>(logit + b * (int64_t)n + 4 * g) = channel_logits<BEC>(ph, (uint64_t)b + offset, (uint32_t)g, bits4, sigma, scale);
  }
}

}  // namespace polar

using namespace polar;

// Persistent grid-stride kernels: exactly as many CTAs as are resident at once (the kernel needs 40 registers, so 6 CTAs of
// 256 threads per SM, not 8 -- with 8 x SMs CTAs a third of them ran as a second, mostly empty wave).
template <class K>
static unsigned fe_grid(K kern, int64_t warps_needed) {
  static std::atomic<int> per_sm{0};                     // one value per kernel instantiation (function-local static of a template)
  int r = per_sm.load(std::memory_order_relaxed);
  if (r <= 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&r, kern, 256, 0) != cudaSuccess || r <= 0) { (void)cudaGetLastError(); r = 4; }
    per_sm.store(r, std::memory_order_relaxed);
  }
  int64_t g = (warps_needed + 7) / 8;
  const int64_t cap = (int64_t)device_sm_count() * r;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (unsigned)g;
}

extern "C" int polar_awgn_frontend(uint64_t seed, uint64_t offset, float no, const uint32_t *d_frozen_mask, int n,
                                   int64_t B, uint32_t *d_u_packed_out, uint32_t *d_c_packed_out, float *d_logit_out,
                                   void *stream) {
  if (!is_pow2(n) || n < 2 || n > POLAR_MAX_N) return set_error(POLAR_EINVAL, "frontend: n=%d must be a power of two in [2,%d]", n, POLAR_MAX_N);
  if (B < 0 || !(no > 0.0f)) return set_error(POLAR_EINVAL, "frontend: B < 0 or no <= 0");
  if (B == 0) return POLAR_OK;
  if (!d_frozen_mask || !d_logit_out) return set_error(POLAR_EINVAL, "frontend: null pointer");
  if (n >= 4 && ((uintptr_t)d_logit_out & 15)) return set_error(POLAR_EALIGN, "frontend: logit_out must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int m = ilog2(n);
  const float sigma = sqrtf(no * 0.5f);                   // std per real dimension (utils.py:12-13, awgn.py:27)
  const float scale = -2.0f * 1.41421356237309505f / no;  // closed-form demapper
#define POLAR_FE_LAUNCH(R) frontend_kernel<R><<<fe_grid(frontend_kernel<R>, B), 256, 0, st>>>(seed, offset, sigma, scale, d_frozen_mask, n, m, B, d_u_packed_out, d_c_packed_out, d_logit_out)
  if (n <= 1024) POLAR_FE_LAUNCH(1);
  else if (n == 2048) POLAR_FE_LAUNCH(2);
  else if (n == 4096) POLAR_FE_LAUNCH(4);
  else POLAR_FE_LAUNCH(8);
#undef POLAR_FE_LAUNCH
  count_launch();
  POLAR_CHECK_LAUNCH("frontend");
  return POLAR_OK;
}

extern "C" int polar_nr5g_awgn_frontend(uint64_t seed, uint64_t offset, float no, const uint32_t *d_payload_mask,
                                        const uint32_t *d_crc_rows, const int32_t *d_crc_pos, int crc_len,
                                        const int32_t *d_rm_idx, int n, int e, int64_t B, uint32_t *d_u_packed_out,
                                        uint32_t *d_c_packed_out, float *d_logit_out, void *stream) {
  if (!is_pow2(n) || n < 32 || n > 1024) return set_error(POLAR_EINVAL, "nr5g frontend: n=%d must be a power of two in [32,1024]", n);
  if (e < 1 || e > POLAR_MAX_N) return set_error(POLAR_EINVAL, "nr5g frontend: e=%d outside [1,%d]", e, POLAR_MAX_N);
  if (crc_len < 1 || crc_len > 32) return set_error(POLAR_EINVAL, "nr5g frontend: crc_len=%d outside [1,32]", crc_len);
  if (B < 0 || !(no > 0.0f)) return set_error(POLAR_EINVAL, "nr5g frontend: B < 0 or no <= 0");
  if (!d_payload_mask || !d_crc_rows || !d_crc_pos || !d_rm_idx) return set_error(POLAR_EINVAL, "nr5g frontend: null table pointer");
  if (B == 0) return POLAR_OK;
  if (!d_u_packed_out || !d_logit_out) return set_error(POLAR_EINVAL, "nr5g frontend: null output pointer");
  const float sigma = sqrtf(no * 0.5f), scale = -2.0f * 1.41421356237309505f / no;
  nr5g_frontend_kernel<<<fe_grid(nr5g_frontend_kernel, B), 256, 0, (cudaStream_t)stream>>>(
      seed, offset, sigma, scale, d_payload_mask, d_crc_rows, d_crc_pos, crc_len, d_rm_idx, n, ilog2(n), e, B,
      d_u_packed_out, d_c_packed_out, d_logit_out);
  count_launch();
  POLAR_CHECK_LAUNCH("nr5g_frontend");
  return POLAR_OK;
}

extern "C" int polar_qpsk_awgn_llr(uint64_t seed, uint64_t offset, float no, const float *d_c, int n, int64_t B,
                                   float *d_logit_out, void *stream) {
  if (n < 4 || (n & 3) || B < 0 || !(no > 0.0f)) return set_error(POLAR_EINVAL, "qpsk_awgn: n must be a multiple of 4, B >= 0, no > 0");
  if (B == 0) return POLAR_OK;
  if (!d_c || !d_logit_out) return set_error(POLAR_EINVAL, "qpsk_awgn: null pointer");
  if (((uintptr_t)d_c & 15) || ((uintptr_t)d_logit_out & 15)) return set_error(POLAR_EALIGN, "qpsk_awgn: buffers must be 16-byte aligned");
  const float sigma = sqrtf(no * 0.5f), scale = -2.0f * 1.41421356237309505f / no;
  const int64_t total = B * (int64_t)(n >> 2);
  int64_t g = (total + 255) / 256;
  const int64_t cap = (int64_t)device_sm_count() * 8;
  if (g > cap) g = cap;
  qpsk_awgn_kernel<false><<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(seed, offset, sigma, scale, d_c, n, B, d_logit_out);
  count_launch();
  POLAR_CHECK_LAUNCH("qpsk_awgn");
  return POLAR_OK;
}

// ---- binary erasure channel (SURVEY 8f row N4, channel half) ------------------------------------------------------
extern "C" int polar_bec_frontend(uint64_t seed, uint64_t offset, float pe, float llr_max, const uint32_t *d_frozen_mask,
                                  int n, int64_t B, uint32_t *d_u_packed_out, uint32_t *d_c_packed_out, float *d_logit_out,
                                  void *stream) {
  if (!is_pow2(n) || n < 2 || n > POLAR_MAX_N) return set_error(POLAR_EINVAL, "bec frontend: n=%d must be a power of two in [2,%d]", n, POLAR_MAX_N);
  if (B < 0 || !(pe >= 0.0f && pe <= 1.0f) || !(llr_max >= 0.0f)) return set_error(POLAR_EINVAL, "bec frontend: B < 0, pe outside [0,1] or llr_max < 0");
  if (B == 0) return POLAR_OK;
  if (!d_frozen_mask || !d_logit_out) return set_error(POLAR_EINVAL, "bec frontend: null pointer");
  if (n >= 4 && ((uintptr_t)d_logit_out & 15)) return set_error(POLAR_EALIGN, "bec frontend: logit_out must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int m = ilog2(n);
#define POLAR_FE_LAUNCH(R) frontend_kernel<R, true><<<fe_grid(frontend_kernel<R, true>, B), 256, 0, st>>>(seed, offset, pe, llr_max, d_frozen_mask, n, m, B, d_u_packed_out, d_c_packed_out, d_logit_out)
  if (n <= 1024) POLAR_FE_LAUNCH(1);
  else if (n == 2048) POLAR_FE_LAUNCH(2);
  else if (n == 4096) POLAR_FE_LAUNCH(4);
  else POLAR_FE_LAUNCH(8);
#undef POLAR_FE_LAUNCH
  count_launch();
  POLAR_CHECK_LAUNCH("bec_frontend");
  return POLAR_OK;
}

extern "C" int polar_bec_llr(uint64_t seed, uint64_t offset, float pe, float llr_max, const float *d_c, int n, int64_t B,
                             float *d_logit_out, void *stream) {
  if (n < 4 || (n & 3) || B < 0 || !(pe >= 0.0f && pe <= 1.0f)) return set_error(POLAR_EINVAL, "bec: n must be a multiple of 4, B >= 0, pe in [0,1]");
  if (B == 0) return POLAR_OK;
  if (!d_c || !d_logit_out) return set_error(POLAR_EINVAL, "bec: null pointer");
  if (((uintptr_t)d_c & 15) || ((uintptr_t)d_logit_out & 15)) return set_error(POLAR_EALIGN, "bec: buffers must be 16-byte aligned");
  const int64_t total = B * (int64_t)(n >> 2);
  int64_t g = (total + 255) / 256;
  const int64_t cap = (int64_t)device_sm_count() * 8;
  if (g > cap) g = cap;
  qpsk_awgn_kernel<true><<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(seed, offset, pe, llr_max, d_c, n, B, d_logit_out);
  count_launch();
  POLAR_CHECK_LAUNCH("bec_llr");
  return POLAR_OK;
}
