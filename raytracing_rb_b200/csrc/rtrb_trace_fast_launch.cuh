// rtrb_trace_fast_launch.cuh — the FAST64 kernels of every class build (rtrb_trace.cuh, "build policies").  The
// kernels carry their class as a namespace: rtrb_fast (generic), rtrb_fast_lean, rtrb_fast_l1 (one light) and
// rtrb_fast_l1n (one light, no Monte-Carlo rays).  Each rtrb_trace_fast_*.cu translation unit instantiates one
// (class, work-stack capacity) pair, so `make -j` compiles them in parallel; rtrb_trace_fast.cu launches them.
#pragma once
#include "rtrb_launch.h"
#include "rtrb_trace_fast.cuh"

// Launch shape per kernel family (16 warps per SM at 128 registers either way; measured on B200, profiles/README.md):
//   depth-1 kernels (MAXS == 1): 128 threads x Policy::d1_min_blocks CTAs per SM.  The extra-sample kernels keep 4
//                                CTAs (config 1: 0.707 vs 0.735 ms)
//   ray-tree kernels (MAXS > 1): lockstep item loop, so the CTA is the unit that shares the instruction caches:
//                                512 threads x 1 CTA per SM on frames of more than a few waves (config 4: 4.44 / 3.78 /
//                                3.57 ms and config 5: 5.13 / 4.61 / 4.24 ms with 128 / 256 / 512 threads; config 3:
//                                3.87 / 3.44 / 3.52), RTRB_TREE_MIN_BLOCK threads on small frames
constexpr int kFastBlock = 128, kExtraMinBlocks = 4, kTreeBlock = 512;

// One class build's kernels for one work-stack capacity (1: the stackless depth-1 kernels), indexed
// [count_detail][use_bvh], and the class they were compiled for.
struct FastKernels {
  bool one_light, lean, no_mc;
  int capacity;
  TraceKernel pre[2][2], extra[2][2];
};

namespace rtrb_fast {
using Pol = rtrb::Generic;
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kFastBlock, Pol::d1_min_blocks) trace_pre_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_body<Pol::at<MAXS>, MAXS, DETAIL, BVH>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kTreeBlock, 1) trace_pre_tree_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_tree_body<Pol::at<MAXS>, MAXS, BVH, DETAIL>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kFastBlock, kExtraMinBlocks) trace_extra_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_extra_body<Pol::at<MAXS>, MAXS, DETAIL, BVH>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
TraceKernel pre_kernel() {
  if constexpr (MAXS == 1) return trace_pre_fast_kernel<1, DETAIL, BVH>;
  else return trace_pre_tree_kernel<MAXS, DETAIL, BVH>;
}
template <int MAXS>
FastKernels kernels() {
  return {Pol::one_light, Pol::lean, Pol::no_mc, MAXS,
          {{pre_kernel<MAXS, false, false>(), pre_kernel<MAXS, false, true>()},
           {pre_kernel<MAXS, true, false>(), pre_kernel<MAXS, true, true>()}},
          {{trace_extra_fast_kernel<MAXS, false, false>, trace_extra_fast_kernel<MAXS, false, true>},
           {trace_extra_fast_kernel<MAXS, true, false>, trace_extra_fast_kernel<MAXS, true, true>}}};
}
}  // namespace rtrb_fast

// depth-1 kernels only
namespace rtrb_fast_lean {
using Pol = rtrb::Lean;
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kFastBlock, Pol::d1_min_blocks) trace_pre_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_body<Pol::at<MAXS>, MAXS, DETAIL, BVH>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kFastBlock, kExtraMinBlocks) trace_extra_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_extra_body<Pol::at<MAXS>, MAXS, DETAIL, BVH>(P);
}
template <int MAXS>
FastKernels kernels() {
  return {Pol::one_light, Pol::lean, Pol::no_mc, MAXS,
          {{trace_pre_fast_kernel<MAXS, false, false>, trace_pre_fast_kernel<MAXS, false, true>},
           {trace_pre_fast_kernel<MAXS, true, false>, trace_pre_fast_kernel<MAXS, true, true>}},
          {{trace_extra_fast_kernel<MAXS, false, false>, trace_extra_fast_kernel<MAXS, false, true>},
           {trace_extra_fast_kernel<MAXS, true, false>, trace_extra_fast_kernel<MAXS, true, true>}}};
}
}  // namespace rtrb_fast_lean

// ray-tree kernels only (the depth-1 frames of these classes run the generic build)
namespace rtrb_fast_l1 {
using Pol = rtrb::OneLight;
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kTreeBlock, 1) trace_pre_tree_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_tree_body<Pol, MAXS, BVH, DETAIL>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kFastBlock, kExtraMinBlocks) trace_extra_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_extra_body<Pol, MAXS, DETAIL, BVH>(P);
}
template <int MAXS>
FastKernels kernels() {
  return {Pol::one_light, Pol::lean, Pol::no_mc, MAXS,
          {{trace_pre_tree_kernel<MAXS, false, false>, trace_pre_tree_kernel<MAXS, false, true>},
           {trace_pre_tree_kernel<MAXS, true, false>, trace_pre_tree_kernel<MAXS, true, true>}},
          {{trace_extra_fast_kernel<MAXS, false, false>, trace_extra_fast_kernel<MAXS, false, true>},
           {trace_extra_fast_kernel<MAXS, true, false>, trace_extra_fast_kernel<MAXS, true, true>}}};
}
}  // namespace rtrb_fast_l1

namespace rtrb_fast_l1n {
using Pol = rtrb::OneLightNoMc;
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kTreeBlock, 1) trace_pre_tree_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_tree_body<Pol, MAXS, BVH, DETAIL>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kFastBlock, kExtraMinBlocks) trace_extra_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_extra_body<Pol, MAXS, DETAIL, BVH>(P);
}
template <int MAXS>
FastKernels kernels() {
  return {Pol::one_light, Pol::lean, Pol::no_mc, MAXS,
          {{trace_pre_tree_kernel<MAXS, false, false>, trace_pre_tree_kernel<MAXS, false, true>},
           {trace_pre_tree_kernel<MAXS, true, false>, trace_pre_tree_kernel<MAXS, true, true>}},
          {{trace_extra_fast_kernel<MAXS, false, false>, trace_extra_fast_kernel<MAXS, false, true>},
           {trace_extra_fast_kernel<MAXS, true, false>, trace_extra_fast_kernel<MAXS, true, true>}}};
}
}  // namespace rtrb_fast_l1n

// The builds, one object each (rtrb_trace_fast_{d1,d1lean,t10,t10_l1,t10_l1n,t32,t32_l1,t32_l1n,t128}.cu).
namespace rtrb_fast { extern const FastKernels d1, t10, t32, t128; }
namespace rtrb_fast_lean { extern const FastKernels d1; }
namespace rtrb_fast_l1 { extern const FastKernels t10, t32; }
namespace rtrb_fast_l1n { extern const FastKernels t10, t32; }
