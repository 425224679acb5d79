// polar_enc.cu -- bit-packed XOR-butterfly polar encoder + bit (un)packing helpers (sm_100a).
//
// Replaces PolarEncoder.forward: x_run_sn_polar/polar/enc.py:30-43 (scatter + dense (c@G)%2) and
// my_sn/fec/polar/enc.py:85-113 (gather/xor stages).  c_j = XOR_{i superset j} u_i.
// One warp per codeword, 32 positions per lane-word; stages below 32 are in-register shifts,
// stages 32..1023 are __shfl_xor, stages above are register-to-register.  HBM-bound.
#include "polar_launch.h"
#include "polar_warp.cuh"

namespace polar {

// ---- packed -> packed ------------------------------------------------------------------------
// n <= 1024: a warp carries 32/nw codewords (lane = cw_local*nw + word).
__global__ void __launch_bounds__(256) enc_packed_small_kernel(const uint32_t *__restrict__ u, int m, int nw,
                                                               int64_t nwords_total, uint32_t *__restrict__ c) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t base = warp0 * 32; base < nwords_total; base += nwarps * 32) {
    const int64_t idx = base + lane;
    uint32_t x = idx < nwords_total ? __ldg(u + idx) : 0u;
    x = ptransform_rt(x, m);
    for (int d = 1; d < nw; d <<= 1) {
      const uint32_t y = __shfl_xor_sync(0xFFFFFFFFu, x, d);
      if (!(lane & d)) x ^= y;
    }
    if (idx < nwords_total) c[idx] = x;
  }
}
// n >= 1024: one codeword per warp, R = n/1024 words per lane.
template <int R>
__global__ void __launch_bounds__(256) enc_packed_kernel(const uint32_t *__restrict__ u, int m, int64_t B,
                                                         uint32_t *__restrict__ c) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp0; b < B; b += nwarps) {
    uint32_t x[R];
#pragma unroll
    for (int r = 0; r < R; ++r) x[r] = __ldg(u + b * (R * 32) + r * 32 + lane);
    warp_polar_transform<R>(x, m, R * 32);
#pragma unroll
    for (int r = 0; r < R; ++r) c[b * (R * 32) + r * 32 + lane] = x[r];
  }
}

// ---- fp32 API tensor in / out: whole PolarEncoder.forward --------------------------------------
template <int R>
__global__ void __launch_bounds__(256) enc_f32_kernel(const float *__restrict__ u, const int32_t *__restrict__ info_rank,
                                                      int n, int m, int k, int64_t B, float *__restrict__ c,
                                                      uint32_t *__restrict__ c_packed) {
  const int lane = threadIdx.x & 31;
  const int nw = n < 32 ? 1 : n >> 5;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp0; b < B; b += nwarps) {
    uint32_t x[R];
#pragma unroll
    for (int r = 0; r < R; ++r) x[r] = 0u;
    // scatter: position p takes u[b, rank(p)] (enc.py:33-35); frozen positions stay 0
    for (int wd = 0; wd < nw; ++wd) {
      const int p = wd * 32 + lane;
      int bit = 0;
      if (p < n) {
        const int rk = __ldg(info_rank + p);
        if (rk >= 0) bit = (__ldg(u + b * (int64_t)k + rk) != 0.0f);
      }
      const uint32_t w = __ballot_sync(0xFFFFFFFFu, bit);
      if (lane == (wd & 31)) x[R == 1 ? 0 : (wd >> 5)] = w;
    }
    warp_polar_transform<R>(x, m, nw);
    if (c_packed) {
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (r * 32 + lane < nw) c_packed[b * nw + r * 32 + lane] = x[r];
    }
    float *row = c + b * (int64_t)n;
    if (n >= 128 && (reinterpret_cast<uintptr_t>(row) & 15) == 0) {
      // 128 positions per round: lane l writes positions 4l .. 4l+3 of the round as one float4; they sit in word l/8 of it
      for (int g = 0; g < (n >> 7); ++g) {
        const int wd = 4 * g + (lane >> 3);
        const uint32_t w = __shfl_sync(0xFFFFFFFFu, x[R == 1 ? 0 : (wd >> 5)], wd & 31) >> ((4 * lane) & 31);
        float4 o;
        o.x = (float)(w & 1u); o.y = (float)((w >> 1) & 1u); o.z = (float)((w >> 2) & 1u); o.w = (float)((w >> 3) & 1u);
        __stcs(reinterpret_cast<float4 *>(row + 128 * g) + lane, o);
      }
    } else {
      for (int wd = 0; wd < nw; ++wd) {
        const uint32_t w = __shfl_sync(0xFFFFFFFFu, x[R == 1 ? 0 : (wd >> 5)], wd & 31);
        const int p = wd * 32 + lane;
        if (p < n) row[p] = (float)((w >> lane) & 1u);
      }
    }
  }
}

// ---- helpers ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_bits_kernel(const float *__restrict__ x, int n, int64_t B,
                                                        uint32_t *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int nw = n < 32 ? 1 : n >> 5;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = warp0; row < B * nw; row += nwarps) {
    const int64_t b = row / nw;
    const int wd = (int)(row - b * nw);
    const int p = wd * 32 + lane;
    const int bit = (p < n) ? (__ldg(x + b * (int64_t)n + p) != 0.0f) : 0;
    const uint32_t w = __ballot_sync(0xFFFFFFFFu, bit);
    if (lane == 0) out[row] = w;
  }
}
// n a multiple of 128 and 16-byte aligned rows: the tensor is one flat stream of 128-position chunks; a lane loads four
// positions as one float4, eight lanes assemble a word
__global__ void __launch_bounds__(256) pack_bits_vec_kernel(const float4 *__restrict__ x, int64_t chunks, uint32_t *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t c = warp0; c < chunks; c += nwarps) {
    const float4 v = __ldcs(x + c * 32 + lane);
    uint32_t w = ((v.x != 0.0f) | ((v.y != 0.0f) << 1) | ((v.z != 0.0f) << 2) | ((v.w != 0.0f) << 3)) << (4 * (lane & 7));
    w |= __shfl_xor_sync(0xFFFFFFFFu, w, 1);
    w |= __shfl_xor_sync(0xFFFFFFFFu, w, 2);
    w |= __shfl_xor_sync(0xFFFFFFFFu, w, 4);
    if ((lane & 7) == 0) out[c * 4 + (lane >> 3)] = w;
  }
}
// [B, nw] packed words -> [B, k] fp32 0./1. at the positions pos[0..k-1] (polar_sc.py:127-133).  One warp per row and
// pass, a float4 per lane and round (128-bit streaming stores: the 4k bytes per row written are the kernel's only real
// traffic); VEC = false is the element-wise fallback for k % 4 != 0 or unaligned buffers.
template <bool VEC>
__global__ void __launch_bounds__(256) unpack_info_kernel(const uint32_t *__restrict__ packed, const int32_t *__restrict__ pos,
                                                          int nw, int k, int64_t B, float *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp0; b < B; b += nwarps) {
    const uint32_t *w = packed + b * nw;
    float *row = out + b * (int64_t)k;
    if (VEC) {
      const int4 *ip = reinterpret_cast<const int4 *>(pos);
      for (int t4 = lane; t4 < (k >> 2); t4 += 32) {
        const int4 p = __ldg(ip + t4);
        float4 o;
        o.x = (float)((__ldg(w + (p.x >> 5)) >> (p.x & 31)) & 1u);
        o.y = (float)((__ldg(w + (p.y >> 5)) >> (p.y & 31)) & 1u);
        o.z = (float)((__ldg(w + (p.z >> 5)) >> (p.z & 31)) & 1u);
        o.w = (float)((__ldg(w + (p.w >> 5)) >> (p.w & 31)) & 1u);
        __stcs(reinterpret_cast<float4 *>(row) + t4, o);
      }
    } else {
      for (int t = lane; t < k; t += 32) {
        const int p = __ldg(pos + t);
        row[t] = (float)((__ldg(w + (p >> 5)) >> (p & 31)) & 1u);
      }
    }
  }
}

}  // namespace polar

using namespace polar;

extern "C" int polar_encode_packed(const uint32_t *d_u, int n, int64_t B, uint32_t *d_c, void *stream) {
  if (const int rc = check_pow2_n("encode", n, 2, POLAR_MAX_N)) return rc;
  if (B < 0) return set_error(POLAR_EINVAL, "encode: B < 0");
  if (B == 0) return POLAR_OK;
  if (!d_u || !d_c) return set_error(POLAR_EINVAL, "encode: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int m = ilog2(n), nw = POLAR_WORDS(n);
  if (n <= 1024) {
    const int64_t total = B * nw;
    return launch("enc_packed", enc_packed_small_kernel, grid_for((total + 31) / 32, 8, 8), 256, 0, st, d_u, m, nw, total, d_c);
  }
  const auto kern = n == 2048 ? enc_packed_kernel<2> : n == 4096 ? enc_packed_kernel<4> : enc_packed_kernel<8>;
  return launch("enc_packed", kern, grid_for(B, 8, 8), 256, 0, st, d_u, m, B, d_c);
}

extern "C" int polar_encode_f32(const float *d_u, const int32_t *d_info_rank, int n, int k, int64_t B, float *d_c,
                                uint32_t *d_c_packed, void *stream) {
  if (const int rc = check_pow2_n("encode", n, 2, POLAR_MAX_N)) return rc;
  if (B < 0 || k < 0 || k > n) return set_error(POLAR_EINVAL, "encode: bad B/k");
  if (B == 0) return POLAR_OK;
  if (!d_u || !d_info_rank || !d_c) return set_error(POLAR_EINVAL, "encode: null pointer");
  const auto kern = n <= 1024 ? enc_f32_kernel<1> : n == 2048 ? enc_f32_kernel<2> : n == 4096 ? enc_f32_kernel<4> : enc_f32_kernel<8>;
  return launch("enc_f32", kern, grid_for(B, 8, 8), 256, 0, (cudaStream_t)stream, d_u, d_info_rank, n, ilog2(n), k, B, d_c,
                d_c_packed);
}

extern "C" int polar_pack_bits_f32(const float *d_x, int n, int64_t B, uint32_t *d_packed, void *stream) {
  if (n < 1 || B < 0 || (n > 32 && (n & 31))) return set_error(POLAR_EINVAL, "pack: n must be <= 32 or a multiple of 32");
  if (B == 0) return POLAR_OK;
  if (!d_x || !d_packed) return set_error(POLAR_EINVAL, "pack: null pointer");
  const cudaStream_t st = (cudaStream_t)stream;
  if ((n & 127) == 0 && ((uintptr_t)d_x & 15) == 0) {
    const int64_t chunks = B * (int64_t)(n >> 7);
    return launch("pack_bits", pack_bits_vec_kernel, grid_for(chunks, 8, 8), 256, 0, st, reinterpret_cast<const float4 *>(d_x),
                  chunks, d_packed);
  }
  return launch("pack_bits", pack_bits_kernel, grid_for(B * POLAR_WORDS(n), 8, 8), 256, 0, st, d_x, n, B, d_packed);
}

extern "C" int polar_unpack_info_f32(const uint32_t *d_packed, const int32_t *d_pos, int n, int k, int64_t B,
                                     float *d_out, void *stream) {
  if (n < 1 || k < 0 || B < 0) return set_error(POLAR_EINVAL, "unpack: bad sizes");
  if (B == 0 || k == 0) return POLAR_OK;
  if (!d_packed || !d_pos || !d_out) return set_error(POLAR_EINVAL, "unpack: null pointer");
  const bool vec = (k & 3) == 0 && (((uintptr_t)d_pos | (uintptr_t)d_out) & 15) == 0;
  const auto kern = vec ? unpack_info_kernel<true> : unpack_info_kernel<false>;
  return launch("unpack_info", kern, grid_for(B, 8, 8), 256, 0, (cudaStream_t)stream,   // one warp per row, 8 warps per CTA
                d_packed, d_pos, POLAR_WORDS(n), k, B, d_out);
}


// ---- 5G rate matching / recovery (SURVEY 8f row N3) -------------------------------------------------------------
// Polar5GEncoder.forward (my_sn/fec/polar/enc.py:378-381): sub-block interleaver, circular-buffer selection and channel
// interleaver are ONE gather c_matched[b, e] = c[b, idx[e]].  Polar5GDecoder.forward (my_sn/fec/polar/dec.py:607-634):
// channel de-interleaver, de-puncturing (logit 0), de-shortening (logit -100), repetition combining (sum) and the
// sub-block de-interleaver are ONE pass out[b, j] = fill[j] + x[b, src0[j]] + x[b, src1[j]] (negative index = absent).
namespace polar {
// one warp per row and pass (no 64-bit division per element; consecutive lanes write consecutive floats of a row)
__global__ void __launch_bounds__(256) gather_cols_kernel(const float *__restrict__ x, const int32_t *__restrict__ idx, int n_in,
                                                          int n_out, int64_t B, float *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp0; b < B; b += nwarps) {
    const float *xr = x + b * (int64_t)n_in;
    float *o = out + b * (int64_t)n_out;
    for (int e = lane; e < n_out; e += 32) o[e] = __ldg(xr + __ldg(idx + e));
  }
}
__global__ void __launch_bounds__(256) rate_recover_kernel(const float *__restrict__ x, const int32_t *__restrict__ src0,
                                                           const int32_t *__restrict__ src1, const float *__restrict__ fill,
                                                           int n_in, int n_out, int64_t B, float *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t b = warp0; b < B; b += nwarps) {
    const float *xr = x + b * (int64_t)n_in;
    float *o = out + b * (int64_t)n_out;
    for (int j = lane; j < n_out; j += 32) {
      const int s0 = __ldg(src0 + j), s1 = __ldg(src1 + j);
      float v = __ldg(fill + j);
      if (s0 >= 0) v = __ldg(xr + s0);                    // received position (fill is 0 there)
      if (s1 >= 0) v = v + __ldg(xr + s1);                // repetition: llr_1 + llr_3 (dec.py:617-620)
      o[j] = v;
    }
  }
}
}  // namespace polar

extern "C" int polar_gather_cols_f32(const float *d_x, const int32_t *d_idx, int n_in, int n_out, int64_t B, float *d_out,
                                     void *stream) {
  using namespace polar;
  if (n_in < 1 || n_out < 1 || B < 0) return set_error(POLAR_EINVAL, "gather: bad sizes");
  if (B == 0) return POLAR_OK;
  if (!d_x || !d_idx || !d_out) return set_error(POLAR_EINVAL, "gather: null pointer");
  return launch("gather_cols", gather_cols_kernel, grid_for(B, 8, 16), 256, 0, (cudaStream_t)stream, d_x, d_idx, n_in, n_out,
                B, d_out);
}

extern "C" int polar_rate_recover_f32(const float *d_x, const int32_t *d_src0, const int32_t *d_src1, const float *d_fill,
                                      int n_in, int n_out, int64_t B, float *d_out, void *stream) {
  using namespace polar;
  if (n_in < 1 || n_out < 1 || B < 0) return set_error(POLAR_EINVAL, "rate_recover: bad sizes");
  if (B == 0) return POLAR_OK;
  if (!d_x || !d_src0 || !d_src1 || !d_fill || !d_out) return set_error(POLAR_EINVAL, "rate_recover: null pointer");
  return launch("rate_recover", rate_recover_kernel, grid_for(B, 8, 16), 256, 0, (cudaStream_t)stream, d_x, d_src0, d_src1,
                d_fill, n_in, n_out, B, d_out);
}
