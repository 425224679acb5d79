// polar_belief.h -- internal declarations of the belief-propagation decoder: the kernel parameters shared by
// polar_belief.cu (belief_kernel and its launcher) and polar_belief_api.cu (argument check and C entry point).
//
// polar_belief.cu is compiled twice (min-sum into namespace polar, exact boxplus into namespace polar_bp through
// polar_bp_wrap.cu).  polar_bp_wrap.cu includes this header before it renames the namespace, so both builds share the
// parameter type and define the launcher declared here in both namespaces.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace polar {

struct BeliefParams {
  const float *logit; const uint32_t *fmask; int n; int64_t B; int iters;
  uint32_t *u_packed; float *u_info; float *llr_info; const int32_t *info_pos; int k;   // any output may be null
};

// polar_belief.cu: belief_kernel over P, with the min-sum f here and the exact boxplus f in polar_bp
int launch_belief(const BeliefParams &P, cudaStream_t st);

}  // namespace polar

namespace polar_bp {
int launch_belief(const polar::BeliefParams &P, cudaStream_t st);
}
