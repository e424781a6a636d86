// FAST64 depth-1 kernels (trace_depth <= 1, stackless; config 2's kernel lives here), generic scenes.  -fmad=false.
#include "rtrb_trace_fast_launch.cuh"
namespace rtrb_fast { const FastKernels d1 = kernels<1>(); }
