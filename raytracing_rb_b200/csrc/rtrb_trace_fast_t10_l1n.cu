// FAST64 ray-tree kernels (work stack <= 10 items), one-light scenes in frames without Monte-Carlo rays
// (rtrb::OneLightNoMc).  -fmad=false.
#include "rtrb_trace_fast_launch.cuh"
namespace rtrb_fast_l1n { const FastKernels t10 = kernels<10>(); }
