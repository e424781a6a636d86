// rtrb_trace_strict.cu — RTRB_PREC_STRICT instantiation of the trace kernels.
// MUST be compiled with -fmad=false: see the arithmetic contract in rtrb_trace.cuh.
#include "rtrb_launch.h"
#include "rtrb_trace.cuh"

namespace {

template <int MAXS, bool DETAIL>
__global__ void __launch_bounds__(kBlock) trace_pre_strict_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_body<rtrb::Strict, MAXS, DETAIL>(P);
}
template <int MAXS, bool DETAIL>
__global__ void __launch_bounds__(kBlock) trace_extra_strict_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_extra_body<rtrb::Strict, MAXS, DETAIL>(P);
}
template <int MAXS, bool DETAIL>
__global__ void __launch_bounds__(kBlock) trace_pass_strict_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_pre_body<rtrb::Strict, MAXS, DETAIL, false, true>(P);
}
template <int MAXS, bool DETAIL>
__global__ void __launch_bounds__(kBlock) trace_mt_strict_kernel(const __grid_constant__ FrameParams P) {
  rtrb::trace_mt_body<rtrb::Strict, MAXS, DETAIL>(P);
}

struct StrictKernels {
  TraceKernel pre, extra, mt, pass;
};
template <int MAXS, bool DETAIL>
const StrictKernels kKernels = {trace_pre_strict_kernel<MAXS, DETAIL>, trace_extra_strict_kernel<MAXS, DETAIL>,
                                trace_mt_strict_kernel<MAXS, DETAIL>, trace_pass_strict_kernel<MAXS, DETAIL>};

// the kernels of `capacity`, with or without the detailed counters
const StrictKernels& kernels(const FrameParams& P, int capacity) {
  const bool det = P.count_detail != 0;
  switch (capacity) {
    case 10: return det ? kKernels<10, true> : kKernels<10, false>;
    case 32: return det ? kKernels<32, true> : kKernels<32, false>;
    default: return det ? kKernels<128, true> : kKernels<128, false>;
  }
}

}  // namespace

cudaError_t rtrb_launch_trace_pre_strict(const FrameParams& P, int capacity, cudaStream_t s) {
  return launch_cover(kernels(P, capacity).pre, pre_threads(P), kBlock, 0, false, s, P);
}
cudaError_t rtrb_launch_trace_extra_strict(const FrameParams& P, int capacity, cudaStream_t s) {
  const TraceKernel k = kernels(P, capacity).extra;
  k<<<extra_grid(), kBlock, 0, s>>>(P);
  return cudaGetLastError();
}
cudaError_t rtrb_launch_trace_mt_strict(const FrameParams& P, int capacity, cudaStream_t s) {
  // one thread per PIXEL
  return launch_cover(kernels(P, capacity).mt, (unsigned long long)P.n_tiles * RTRB_SUPER_PIXELS, kBlock, 0, false, s, P);
}
cudaError_t rtrb_launch_trace_pass_strict(const FrameParams& P, int capacity, cudaStream_t s) {
  return launch_cover(kernels(P, capacity).pass, pass_threads(P), kBlock, 0, false, s, P);
}
