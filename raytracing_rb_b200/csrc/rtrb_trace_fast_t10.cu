// FAST64 ray-tree kernels with a work stack of up to 10 items, generic scenes.  -fmad=false.
#include "rtrb_trace_fast_launch.cuh"
namespace rtrb_fast { const FastKernels t10 = kernels<10>(); }
