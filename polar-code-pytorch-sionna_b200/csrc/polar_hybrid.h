// polar_hybrid.h -- internal declarations of the hybrid SC -> SCL decoder (polar_hybrid.cu).
//
// polar_scl.cu is compiled twice (min-sum into namespace polar, boxplus into namespace polar_bp through polar_bp_wrap.cu);
// both builds export the row-indexed scl2 launcher declared here.  Under polar_bp_wrap.cu `polar` is a macro for
// `polar_bp`, so the first block below declares the boxplus copies there; the second block gives polar_hybrid.cu the
// boxplus names directly.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#define POLAR_HYBRID_DECLS                                                                                            \
  /* bytes of the workspace of scl2_kernel<L> planned for B codewords (persistent grid, never shrunk) */             \
  size_t scl2_rows_workspace_bytes(int n, int L, int64_t B);                                                          \
  /* scl2_kernel<L> over the rows rows[0 .. min(*n_rows, B)-1] of logit / best / u_info (device pointers); the grid   \
     is planned from the upper bound B, ws must hold scl2_rows_workspace_bytes(n, L, B); fast: boxplus build only */  \
  int launch_scl2_rows(const float *logit, const uint32_t *fmask, int n, int L, int64_t B, const int32_t *rows,       \
                       const int32_t *n_rows, uint32_t *best, float *u_info, const int32_t *info_pos, int k,          \
                       const uint32_t *crc_rows, int crc_len, void *ws, int fast, cudaStream_t st);

namespace polar { POLAR_HYBRID_DECLS }
namespace polar_bp { POLAR_HYBRID_DECLS }
