// rtrb_trace_fast_build.cuh — the kernels of one FAST64 class build.  Included once inside the namespace of each build,
// after `using Pol = <the build's policy>;` (rtrb_trace_fast_launch.cuh), hence no include guard.  A fragment rather
// than a macro, so that -lineinfo maps each kernel wrapper to its own lines.  Each build's translation units
// instantiate kernels<MAXS>() for the capacities it exists for (rtrb_trace_fast_*.cu).
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kBlock, Pol::d1_min_blocks) trace_pre_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_body<Pol::at<MAXS>, MAXS, DETAIL, BVH>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kTreeBlock, 1) trace_pre_tree_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_tree_body<Pol::at<MAXS>, MAXS, BVH, DETAIL>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kBlock, kExtraMinBlocks) trace_extra_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_extra_body<Pol::at<MAXS>, MAXS, DETAIL, BVH>(P);
}
// progressive frames: the pre kernels' pass variants (same launch shape)
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kBlock, Pol::d1_min_blocks) trace_pass_fast_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_body<Pol::at<MAXS>, MAXS, DETAIL, BVH, true>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kTreeBlock, 1) trace_pass_tree_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_tree_body<Pol::at<MAXS>, MAXS, BVH, DETAIL, true>(P);
}
template <int MAXS, bool DETAIL, bool BVH>
TraceKernel pre_kernel() {
  if constexpr (MAXS == 1) return trace_pre_fast_kernel<1, DETAIL, BVH>;
  else return trace_pre_tree_kernel<MAXS, DETAIL, BVH>;
}
// Only the generic build has pass kernels (the class builds give the same bits; each instantiation costs compile time).
template <int MAXS, bool DETAIL, bool BVH>
TraceKernel pass_kernel() {
  if constexpr (!std::is_same<Pol, rtrb::Generic>::value) return nullptr;
  else if constexpr (MAXS == 1) return trace_pass_fast_kernel<1, DETAIL, BVH>;
  else return trace_pass_tree_kernel<MAXS, DETAIL, BVH>;
}
template <int MAXS>
FastKernels kernels() {
  return {Pol::one_light, Pol::lean, Pol::no_mc, MAXS,
          {{pre_kernel<MAXS, false, false>(), pre_kernel<MAXS, false, true>()},
           {pre_kernel<MAXS, true, false>(), pre_kernel<MAXS, true, true>()}},
          {{trace_extra_fast_kernel<MAXS, false, false>, trace_extra_fast_kernel<MAXS, false, true>},
           {trace_extra_fast_kernel<MAXS, true, false>, trace_extra_fast_kernel<MAXS, true, true>}},
          {{pass_kernel<MAXS, false, false>(), pass_kernel<MAXS, false, true>()},
           {pass_kernel<MAXS, true, false>(), pass_kernel<MAXS, true, true>()}}};
}
