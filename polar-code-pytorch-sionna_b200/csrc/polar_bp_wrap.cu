// polar_bp_wrap.cu -- compiles one decoder translation unit a second time with the exact-boxplus f
// (my_sn/fec/polar/dec.py:33-46) instead of min-sum (SURVEY 8f row N2): every kernel, launcher and device symbol of the
// unit lands in namespace polar_bp, so the boxplus launchers are the min-sum ones' namesakes, polar_bp::launch_sc4,
// polar_bp::launch_scl2, polar_bp::launch_belief and so on.
//   nvcc ... -DPOLAR_BP_SRC=\"polar_sc4.cu\" -c polar_bp_wrap.cu -o polar_sc4_bp.o
// Every internal header (*.h) that a unit compiled here includes must be included below, before `polar` is renamed:
// otherwise its #pragma once declarations land in namespace polar_bp.  The device headers (*.cuh) are left to the unit,
// so that they are compiled with the boxplus f.
#include "polar_internal.h"      // host plumbing stays in ::polar (set_error, env_int, device queries ...)
#include "polar_launch.h"        // so do the launch helpers and the Arith enum
#include "polar_sc.h"            // and the declarations of the launchers in both namespaces
#include "polar_scl.h"
#include "polar_belief.h"
namespace polar_bp { using namespace polar; }
#define POLAR_F_BOXPLUS 1
#define polar polar_bp
// the debug hooks are extern "C", outside any namespace: a second copy needs its own name
#define polar_sc4_debug_read polar_sc4_bp_debug_read
#define polar_sc5_debug_read polar_sc5_bp_debug_read
#include POLAR_BP_SRC
