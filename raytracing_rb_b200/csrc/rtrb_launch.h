// rtrb_launch.h — host-callable launchers of the trace kernels.  Each arithmetic mode lives in its
// own translation units, all compiled -fmad=false (the exact FP64 parts must round like the reference's scalar code;
// the FP32 filter of FAST64 uses explicit fmaf()):
//   rtrb_trace_strict.cu                          RTRB_PREC_STRICT
//   rtrb_trace_fast.cu + rtrb_trace_fast_*.cu     RTRB_PREC_FAST64 (dispatch + one TU per class build and work-stack
//                                                 capacity, rtrb_trace_fast_launch.cuh)
#pragma once
#include <cuda_runtime.h>

#include "rtrb_types.h"

// Work-stack capacities the ray-tree kernels are compiled for: the smallest one that holds stack_need items
// (0: none does).  The FAST64 depth-1 kernels are stackless.
constexpr int kMaxStack = 128;
constexpr int stack_capacity(int stack_need) {
  return stack_need <= 10 ? 10 : stack_need <= 32 ? 32 : stack_need <= kMaxStack ? kMaxStack : 0;
}
inline int rtrb_max_stack_supported(void) { return kMaxStack; }

inline int sm_count() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}
// CTAs of `block` threads that cover `threads` threads: 0 when there is nothing to launch, -1 when the grid is too large.
inline long long grid_size(unsigned long long threads, int block) {
  const unsigned long long blocks = (threads + block - 1) / block;
  return blocks > 0x7fffffffull ? -1 : (long long)blocks;
}
// Threads of a pre-sample launch: one per (tile pixel, sample < pre).
inline unsigned long long pre_threads(const FrameParams& P) {
  return (unsigned long long)P.n_tiles * RTRB_SUPER_PIXELS * (unsigned long long)P.pre;
}
// Grid of the persistent grid-stride extra-sample kernels: 8 CTAs per SM.
inline unsigned extra_grid() { return (unsigned)sm_count() * 8u; }

using TraceKernel = void (*)(FrameParams);

// stack_need = deepest work stack the frame can reach (trace_depth * (1 + mc) + 1).
cudaError_t rtrb_launch_trace_pre_strict(const FrameParams& P, int stack_need, cudaStream_t s);
cudaError_t rtrb_launch_trace_extra_strict(const FrameParams& P, int stack_need, cudaStream_t s);
// overlap: launch with programmatic stream serialization (depth-1 frames only; rtrb_api.cu, render_impl)
cudaError_t rtrb_launch_trace_pre_fast(const FrameParams& P, int stack_need, cudaStream_t s, bool overlap = false);
cudaError_t rtrb_launch_trace_extra_fast(const FrameParams& P, int stack_need, cudaStream_t s);
cudaError_t rtrb_launch_trace_mt_strict(const FrameParams& P, int stack_need, cudaStream_t s);  // RTRB_RNG_MT
