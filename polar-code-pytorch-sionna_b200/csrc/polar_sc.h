// polar_sc.h -- internal declarations of the SC decoder: the launchers of its three mappings, in both arithmetics, and
// the argument check and dispatch of polar_sc_api.cu.
//
// polar_sc.cu, polar_sc4.cu and polar_sc5.cu are compiled twice (min-sum into namespace polar, exact boxplus into
// namespace polar_bp through polar_bp_wrap.cu).  polar_internal.h declares the ::polar launch_sc4 / launch_sc5.
#pragma once
#include "polar_launch.h"

namespace polar {

// polar_sc.cu: n in [2, 64], one thread per codeword
int launch_sc_small(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
                    const int32_t *info_pos, int k, cudaStream_t st);

// polar_sc_api.cu.  check_sc_args: the checks an SC decode on device or host buffers shares; a call with B == 0 passes
// once n and B are valid, whatever its buffers.  sc_decode: one SC decode on device buffers, checked, of any n.
int check_sc_args(const char *who, int n, int64_t B, const float *logit, const uint32_t *fmask, bool has_output,
                  const float *u_info, const int32_t *info_pos, int k);
int sc_decode(Arith arith, const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
              const int32_t *info_pos, int k, void *stream);

}  // namespace polar

namespace polar_bp {

int launch_sc_small(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
                    const int32_t *info_pos, int k, cudaStream_t st);
int launch_sc4(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
               const int32_t *info_pos, int k, int warps, cudaStream_t st);
int launch_sc5(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
               const int32_t *info_pos, int k, int warps, cudaStream_t st);

}  // namespace polar_bp
