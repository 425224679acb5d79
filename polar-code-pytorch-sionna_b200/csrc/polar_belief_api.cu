// polar_belief_api.cu -- the C entry point of the belief-propagation decoder (include/polar_b200.h,
// polar_belief_decode_f32): argument check, then the kernel of the chosen arithmetic (polar_belief.cu: launch_belief,
// in namespace polar with min-sum and in namespace polar_bp, compiled through polar_bp_wrap.cu, with exact boxplus).
#include "polar_launch.h"
#include "polar_belief.h"

using namespace polar;

extern "C" int polar_belief_decode_f32(const float *d_logit, const uint32_t *d_frozen_mask, int n, int64_t B, int num_iter,
                                       int cn_mode, uint32_t *d_u_packed, float *d_u_info_f32, float *d_llr_info_f32,
                                       const int32_t *d_info_pos, int k, void *stream) {
  if (const int rc = check_pow2_n("belief", n, 2, POLAR_BP_MAX_N)) return rc;
  if (num_iter < 1) return set_error(POLAR_EINVAL, "belief: num_iter=%d must be >= 1", num_iter);
  if (cn_mode != 0 && cn_mode != 1) return set_error(POLAR_EINVAL, "belief: cn_mode=%d must be 0 (min-sum) or 1 (boxplus)", cn_mode);
  if (B < 0) return set_error(POLAR_EINVAL, "belief: B=%lld < 0", (long long)B);
  if (B == 0) return POLAR_OK;
  if (!d_logit || !d_frozen_mask) return set_error(POLAR_EINVAL, "belief: null logit / frozen_mask");
  if (!d_u_packed && !d_u_info_f32 && !d_llr_info_f32) return set_error(POLAR_EINVAL, "belief: no output buffer");
  if ((d_u_info_f32 || d_llr_info_f32) && (!d_info_pos || k < 0 || k > n))
    return set_error(POLAR_EINVAL, "belief: a [B, k] output needs info_pos and k in [0,%d], got k=%d", n, k);
  if (n >= 4 && ((uintptr_t)d_logit & 15)) return set_error(POLAR_EALIGN, "belief: logit must be 16-byte aligned");
  BeliefParams P;
  P.logit = d_logit; P.fmask = d_frozen_mask; P.n = n; P.B = B; P.iters = num_iter;
  P.u_packed = d_u_packed; P.u_info = d_u_info_f32; P.llr_info = d_llr_info_f32; P.info_pos = d_info_pos; P.k = k;
  const cudaStream_t st = (cudaStream_t)stream;
  return (Arith)cn_mode == Arith::minsum ? launch_belief(P, st) : polar_bp::launch_belief(P, st);
}
