// FAST64 depth-1 kernels, lean scenes (rtrb::Lean: one light of radius 0, no textures, exponent 2).  -fmad=false.
#include "rtrb_trace_fast_launch.cuh"
namespace rtrb_fast_lean { const FastKernels d1 = kernels<1>(); }
