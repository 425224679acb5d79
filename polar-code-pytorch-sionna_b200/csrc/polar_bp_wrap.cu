// polar_bp_wrap.cu -- compiles one SC translation unit a second time with the exact-boxplus f
// (my_sn/fec/polar/dec.py:33-46) instead of min-sum: every kernel, launcher and device symbol of the unit lands
// in namespace polar_bp; the SC C entry point is renamed polar_sc_decode_boxplus_f32 (SURVEY 8f row N2), the list
// kernel's launcher launch_scl2_boxplus and the belief-propagation kernel's launcher launch_belief_boxplus.
//   nvcc ... -DPOLAR_BP_SRC=\"polar_sc4.cu\" -c polar_bp_wrap.cu -o polar_sc4_bp.o
#include "polar_internal.h"      // host plumbing stays in ::polar (set_error, env_int, device queries ...)
#include "polar_scl.h"           // so do the list decoder's parameter and plan types
#include "polar_belief.h"        // and the belief-propagation decoder's parameters
namespace polar_bp { using namespace polar; }
#define POLAR_F_BOXPLUS 1
#define polar polar_bp
#define polar_sc_decode_f32 polar_sc_decode_boxplus_f32
#define polar_sc4_debug_read polar_sc4_bp_debug_read
#define polar_sc5_debug_read polar_sc5_bp_debug_read
#define launch_scl2 launch_scl2_boxplus
#define launch_belief launch_belief_boxplus
namespace polar {                // the launchers the units call across files, redeclared in the boxplus namespace
int launch_sc5(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
               const int32_t *info_pos, int k, int warps, cudaStream_t st);
int launch_sc4(const float *logit, const uint32_t *fmask, int n, int64_t B, uint32_t *u_packed, float *u_info,
               const int32_t *info_pos, int k, int warps, cudaStream_t st);
}
#include POLAR_BP_SRC
