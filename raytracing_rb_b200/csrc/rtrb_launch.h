// rtrb_launch.h — which trace kernel a frame or ray batch runs, its launch shape, and the host-callable launchers.
// Each arithmetic mode lives in its own translation units, all compiled -fmad=false (the exact FP64 parts must round
// like the reference's scalar code; the FP32 filter of FAST64 uses explicit fmaf()):
//   rtrb_trace_strict.cu                          RTRB_PREC_STRICT
//   rtrb_trace_fast.cu + rtrb_trace_fast_*.cu     RTRB_PREC_FAST64 (dispatch + one TU per class build and work-stack
//                                                 capacity, rtrb_trace_fast_launch.cuh)
//   rtrb_rays.cu                                  the ray-level kernels of both modes (rtrb_rays.h)
#pragma once
#include <cuda_runtime.h>

#include "rtrb_types.h"

// Work-stack capacity of the kernels that trace a frame or ray batch: a trace of depth trace_depth with mc Monte-Carlo
// rays per hit can hold trace_depth * (1 + mc) + 1 items on its work stack, and runs the kernels of the smallest
// capacity (10, 32, kMaxStack) that holds them.  The FAST64 kernels of depth <= 1 are stackless: capacity 1.  0: no
// kernel holds the stack.
constexpr int kMaxStack = 128;
constexpr int trace_capacity(bool strict, int trace_depth, int mc) {
  const long long need = (long long)trace_depth * (1 + (long long)mc) + 1;
  if (need > kMaxStack) return 0;
  if (!strict && trace_depth <= 1) return 1;
  return need <= 10 ? 10 : need <= 32 ? 32 : kMaxStack;
}

// Launch shape (16 warps per SM at 128 registers either way; measured on B200, profiles/README.md):
//   kBlock           threads per CTA of the trace and ray kernels, except the FAST64 ray-tree pre kernels: the
//                    depth-1 kernels run 128 x Policy::d1_min_blocks CTAs per SM (rtrb_trace.cuh; config 2: 256 x 2
//                    is slower)
//   kExtraMinBlocks  CTAs per SM of the free-running FAST64 kernels that are not depth-1 pre kernels: the
//                    extra-sample kernels (config 1: 0.707 vs 0.735 ms) and the ray-tree trace_rays kernels
//   kTreeBlock       the FAST64 ray-tree pre kernels run a lockstep item loop, so the CTA is the unit that shares the
//                    instruction caches: 512 threads x 1 CTA per SM on frames of more than a few waves (config 4:
//                    4.44 / 3.78 / 3.57 ms and config 5: 5.13 / 4.61 / 4.24 ms with 128 / 256 / 512 threads;
//                    config 3: 3.87 / 3.44 / 3.52), RTRB_TREE_MIN_BLOCK threads on small frames
constexpr int kBlock = 128, kExtraMinBlocks = 4, kTreeBlock = 512;

inline int sm_count() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}
// Threads of a pre-sample launch: one per (tile pixel, sample < pre).
inline unsigned long long pre_threads(const FrameParams& P) {
  return (unsigned long long)P.n_tiles * RTRB_SUPER_PIXELS * (unsigned long long)P.pre;
}
// Threads of a progressive frame's pass: one per (tile pixel, sample in [pass_begin, pass_end)).
inline unsigned long long pass_threads(const FrameParams& P) {
  return (unsigned long long)P.n_tiles * RTRB_SUPER_PIXELS * (unsigned long long)(P.pass_end - P.pass_begin);
}
// Grid of the persistent grid-stride extra-sample kernels: 8 CTAs per SM.
inline unsigned extra_grid() { return (unsigned)sm_count() * 8u; }

// Launches `k(args...)` with one thread for each of `threads`, in CTAs of `block` threads with `smem` bytes of dynamic
// shared memory: nothing when there are no threads, cudaErrorInvalidConfiguration when the grid would be too large.
// overlap: with programmatic stream serialization, so the kernel may start under the tail of the previous kernel on the
// stream (trace_pre_body).
template <class... Params, class... Args>
cudaError_t launch_cover(void (*k)(Params...), unsigned long long threads, int block, size_t smem, bool overlap,
                         cudaStream_t s, const Args&... args) {
  const unsigned long long blocks = (threads + block - 1) / block;
  if (blocks == 0) return cudaSuccess;
  if (blocks > 0x7fffffffull) return cudaErrorInvalidConfiguration;
  if (!overlap) {
    k<<<(unsigned)blocks, block, smem, s>>>(args...);
    return cudaGetLastError();
  }
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)blocks);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k, args...);
}

using TraceKernel = void (*)(FrameParams);

// capacity: trace_capacity() of the frame, never 0.
cudaError_t rtrb_launch_trace_pre_strict(const FrameParams& P, int capacity, cudaStream_t s);
cudaError_t rtrb_launch_trace_extra_strict(const FrameParams& P, int capacity, cudaStream_t s);
// overlap: launch with programmatic stream serialization (depth-1 frames only; rtrb_api.cu, render_impl)
cudaError_t rtrb_launch_trace_pre_fast(const FrameParams& P, int capacity, cudaStream_t s, bool overlap = false);
cudaError_t rtrb_launch_trace_extra_fast(const FrameParams& P, int capacity, cudaStream_t s);
// progressive frames (rtrb_api.cu, rtrb_progressive_pass): samples [P.pass_begin, P.pass_end) into the sample buffer
cudaError_t rtrb_launch_trace_pass_strict(const FrameParams& P, int capacity, cudaStream_t s);
cudaError_t rtrb_launch_trace_pass_fast(const FrameParams& P, int capacity, cudaStream_t s);
cudaError_t rtrb_launch_trace_mt_strict(const FrameParams& P, int capacity, cudaStream_t s);  // RTRB_RNG_MT
