// FAST64 ray-tree kernels (work stack <= 32 items), one-light scenes (rtrb::OneLight).  -fmad=false.
#include "rtrb_trace_fast_launch.cuh"
namespace rtrb_fast_l1 { const FastKernels t32 = kernels<32>(); }
