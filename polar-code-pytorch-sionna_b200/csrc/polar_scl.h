// polar_scl.h -- internal declarations of the list decoder: the kernel parameters and plan shared by polar_scl.cu
// (scl2_kernel<L>), polar_scl_api.cu (argument check, plan and C entry points) and polar_host.cu.
//
// polar_scl.cu is compiled twice (min-sum into namespace polar, exact boxplus into namespace polar_bp through
// polar_bp_wrap.cu).  polar_bp_wrap.cu includes this header before it renames the namespace, so both builds share the
// types below and define the launcher declared here in both namespaces.
#pragma once
#include "polar_launch.h"

namespace polar {

struct SclParams {
  const float *logit; const uint32_t *fmask; int n, m; int64_t B;
  uint32_t *best; float *u_info; const int32_t *info_pos; int k;
  double *pm_out; uint32_t *list; const uint32_t *crc_rows; int crc_len;
  double *ws; size_t ws_doubles_per_warp; int s_glob;   // LLR stages >= s_glob live in ws
  size_t smem_per_warp;
  int words_global;                                     // scl2: partial-sum words live in ws (after the LLR stages)
  int fast;                                             // boxplus build only: node-level path-metric updates (use_fast_scl)
  // row-indexed decode (the hybrid's list stage): when rows != nullptr, codeword j = 0 .. min(*n_rows, B)-1 is logit
  // row rows[j] and its outputs go to row rows[j]; no other output row is written.  B is then the host-side upper bound
  // of *n_rows.
  const int32_t *rows; const int32_t *n_rows;
};

// How one list decode runs (scl_plan).
struct SclPlan {
  bool scl3;                  // scl3_kernel (polar_scl3.cu) runs; otherwise scl2_kernel<L>
  int64_t grid;               // persistent grid, in warps (scl2_kernel<L> runs one warp per CTA)
  size_t ws_bytes_per_warp;
  size_t ws_bytes;            // the workspace to allocate for the call (see scl_plan)
  int s_glob; size_t smem_per_warp; int words_global;   // scl2_kernel<L>: SclParams fields of the same names
};

// LLR stages 0 .. s_glob-1 of scl2_kernel<L> in shared memory: [2^s elements][32 slots] doubles per stage s
__host__ __device__ inline size_t scl2_llr_smem_doubles(int s_glob) { return (size_t)32 * ((1u << s_glob) - 1u); }

// polar_scl_api.cu.  check_scl_shape: n, L and B of any list-decoder call.  scl_plan: the mapping, grid and workspace
// of a decode of B rows; scl3_rows says whether the rows suit scl3 (16-byte aligned, decoded in order).
int check_scl_shape(const char *who, int n, int L, int64_t B);
SclPlan scl_plan(int n, int L, int64_t B, Arith arith, bool scl3_rows);

// polar_scl.cu: scl2_kernel<L> over P on pl.grid one-warp CTAs, with the min-sum f here and the exact boxplus f in polar_bp
int launch_scl2(const SclParams &P, const SclPlan &pl, int L, cudaStream_t st);

}  // namespace polar

namespace polar_bp {
int launch_scl2(const polar::SclParams &P, const polar::SclPlan &pl, int L, cudaStream_t st);
}
