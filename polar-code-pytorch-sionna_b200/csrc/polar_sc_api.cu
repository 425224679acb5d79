// polar_sc_api.cu -- the C entry points of the SC decoder (include/polar_b200.h, polar_sc_decode_f32 and
// polar_sc_decode_boxplus_f32), its argument check, and the choice of mapping, by the code length alone:
//   n <= 64           one thread per codeword, the whole tree in registers (polar_sc.cu);
//   128 <= n <= 512   a warp per 32 codewords, everything on chip: shared memory / tensor memory / registers (polar_sc4.cu);
//   n >= 1024         the same with TMA-staged fused descents through the top stages and a global scratch hierarchy for
//                     the stages that do not fit on chip (polar_sc5.cu).
// Every mapping runs in the arithmetic of the call: min-sum from namespace polar, exact boxplus from namespace polar_bp.
#include "polar_sc.h"

namespace polar {

int check_sc_args(const char *who, int n, int64_t B, const float *logit, const uint32_t *fmask, bool has_output,
                  const float *u_info, const int32_t *info_pos, int k) {
  if (const int rc = check_pow2_n(who, n, 2, POLAR_MAX_N)) return rc;
  if (B < 0) return set_error(POLAR_EINVAL, "%s: B=%lld < 0", who, (long long)B);
  if (B == 0) return POLAR_OK;
  if (!logit || !fmask) return set_error(POLAR_EINVAL, "%s: null logit / frozen_mask", who);
  if (!has_output) return set_error(POLAR_EINVAL, "%s: no output buffer", who);
  if (u_info && (!info_pos || k < 0 || k > n)) return set_error(POLAR_EINVAL, "%s: u_info requested without valid info_pos/k", who);
  return POLAR_OK;
}

int sc_decode(Arith arith, const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
              const int32_t *info_pos, int k, void *stream) {
  const int rc = check_sc_args("sc", n, B, logit, fmask, u_packed || u_info, u_info, info_pos, k);
  if (rc != POLAR_OK || B == 0) return rc;
  if (n >= 4 && ((uintptr_t)logit & 15)) return set_error(POLAR_EALIGN, "sc: logit must be 16-byte aligned");
  const bool minsum = arith == Arith::minsum;
  const cudaStream_t st = (cudaStream_t)stream;
  if (n <= 64)
    return (minsum ? launch_sc_small : polar_bp::launch_sc_small)(logit, fmask, n, B, u_packed, u_info, info_pos, k, st);
  const int warps = env_int("POLAR_SC_WARPS_SM", 0);      // autonomous warps per SM (0 = as many as the on-chip storage holds)
  if (n <= 512) return (minsum ? launch_sc4 : polar_bp::launch_sc4)(logit, fmask, n, B, u_packed, u_info, info_pos, k, warps, st);
  return (minsum ? launch_sc5 : polar_bp::launch_sc5)(logit, fmask, n, B, u_packed, u_info, info_pos, k, warps, st);
}

}  // namespace polar

extern "C" int polar_sc_decode_f32(const float *d_logit, const uint32_t *d_frozen_mask, int n, int64_t B,
                                   uint32_t *d_u_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k, void *stream) {
  return polar::sc_decode(polar::Arith::minsum, d_logit, d_frozen_mask, n, B, d_u_packed, d_u_info_f32, d_info_pos, k, stream);
}

extern "C" int polar_sc_decode_boxplus_f32(const float *d_logit, const uint32_t *d_frozen_mask, int n, int64_t B,
                                           uint32_t *d_u_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                                           void *stream) {
  return polar::sc_decode(polar::Arith::boxplus, d_logit, d_frozen_mask, n, B, d_u_packed, d_u_info_f32, d_info_pos, k, stream);
}
