// rtrb_rays.cu — the ray-level kernels behind rtrb_trace_rays, rtrb_intersect_rays and rtrb_camera_rays: one thread per
// caller-supplied ray (or per camera sample), running the same device functions as the frame kernels.
//   trace_rays      RayTracer#trace_sync (ray_tracer.rb:16-46): trace_sample (STRICT) / trace_sample_fast (FAST64,
//                   generic build), free-running, instantiated over the frame kernels' axes (stack capacity, detailed
//                   counters with the Box code, BVH or linear filter)
//   intersect_rays  World#intersect (world.rb:37-59): the literal scan (STRICT) / filter + exact test (FAST64)
//   camera_rays     Camera#lens_func (camera.rb:129-151) with the frames' aperture draw
// The FrameParams these kernels get never carry a valid camera apex table (cam_tab_valid = 0): that table only bounds
// rays that start at the camera.  MUST be compiled with -fmad=false, like every trace translation unit.
#include "rtrb_launch.h"
#include "rtrb_rays.h"
#include "rtrb_trace_fast.cuh"

namespace {

using namespace rtrb;

// One thread per ray; the status of ray i is reported as pixel (i, 0) of a frame of height 1.
template <class Pol, int MAXS, bool DETAIL, bool BVH>
__device__ __forceinline__ void trace_rays_body(const FrameParams& P, const RayBatch& B) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  ThreadCtx ctx;
  init_ctx(ctx, DETAIL);
  const bool active = i < (unsigned long long)B.n;
  if (active) {
    const double* q = B.rays + i * 6ull;
    const d3 ro = mk(q[0], q[1], q[2]), rd = mk(q[3], q[4], q[5]);
    uint32_t pixel = (uint32_t)i, sample = 0u;
    if (B.keys) { pixel = B.keys[2ull * i]; sample = B.keys[2ull * i + 1ull]; }
    int ph;
    const d3 col = trace_dispatch<Pol, MAXS, BVH, DETAIL>(P, ro, rd, pixel, sample, ctx, &ph);
    RTRB_COUNT(ctx, RTRB_CNT_SAMPLES);
    double* out = B.rgb + i * 3ull;
    out[0] = col.x; out[1] = col.y; out[2] = col.z;
    if (B.hit) B.hit[i] = ph;
  }
  flush_ctx(P, ctx, (int)i, 0, active);
}

// Launch bounds as the frame kernels that run the same per-sample code free-running: the STRICT kernels, the generic
// depth-1 kernel (Policy::d1_min_blocks) and the extra-sample kernels (kExtraMinBlocks).
template <int MAXS, bool DETAIL>
__global__ void __launch_bounds__(kBlock) trace_rays_strict_kernel(const __grid_constant__ FrameParams P, const RayBatch B) {
  trace_rays_body<Strict, MAXS, DETAIL, false>(P, B);
}
template <int MAXS, bool DETAIL, bool BVH>
__global__ void __launch_bounds__(kBlock, MAXS == 1 ? Generic::d1_min_blocks : kExtraMinBlocks)
    trace_rays_fast_kernel(const __grid_constant__ FrameParams P, const RayBatch B) {
  trace_rays_body<Generic::at<MAXS>, MAXS, DETAIL, BVH>(P, B);
}

using RayKernel = void (*)(FrameParams, RayBatch);

template <int MAXS>
RayKernel strict_trace(bool detail) {
  return detail ? trace_rays_strict_kernel<MAXS, true> : trace_rays_strict_kernel<MAXS, false>;
}
template <int MAXS>
RayKernel fast_trace(bool detail, bool bvh) {
  if (detail) return bvh ? trace_rays_fast_kernel<MAXS, true, true> : trace_rays_fast_kernel<MAXS, true, false>;
  return bvh ? trace_rays_fast_kernel<MAXS, false, true> : trace_rays_fast_kernel<MAXS, false, false>;
}

// World#intersect for one ray into the ABI record, with intersect_parameters' delta.
template <bool STRICT, bool BVH>
__global__ void __launch_bounds__(kBlock) intersect_rays_kernel(const __grid_constant__ FrameParams P, const RayBatch B) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (unsigned long long)B.n) return;
  const double* q = B.rays + i * 6ull;
  const d3 o = mk(q[0], q[1], q[2]), d = mk(q[3], q[4], q[5]);
  ThreadCtx ctx;
  init_ctx(ctx, false);
  HitRec bh;
  bh.p = mk(0, 0, 0); bh.dir_in = false; bh.face = 0;
  int best_i;
  if constexpr (STRICT) {
    best_i = closest_hit_scan<Strict, true>(P, o, d, bh, ctx);
  } else {
    const CullRay r = make_cull_ray(P, o, d);
    best_i = closest_hit_fast<Generic, BVH, true, !BVH>(P, o, d, r, bh, ctx, false);
  }
  rtrb_ray_hit h = {};
  h.object = best_i;
  h.face = -1;
  if (best_i >= 0) {
    const DevGeom g = P.geom[best_i];
    const d3 delta = intersect_parameters<true>(P, g, P.mat[best_i], bh, d).delta;
    if (g.type == RTRB_OBJ_BOX) h.face = bh.face;
    h.direction = bh.dir_in ? 1 : 0;
    h.distance = norm(o - bh.p);  // the expression World#intersect compared
    h.intersection[0] = bh.p.x; h.intersection[1] = bh.p.y; h.intersection[2] = bh.p.z;
    h.delta[0] = delta.x; h.delta[1] = delta.y; h.delta[2] = delta.z;
  }
  B.hits[i] = h;
}

// Camera#lens_func for (window pixel, sample j): the frame kernels' camera_ray.
__global__ void __launch_bounds__(kBlock) camera_rays_kernel(const __grid_constant__ FrameParams P, const RayBatch B) {
  const unsigned long long w = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= (unsigned long long)B.n) return;
  const unsigned long long S = (unsigned long long)(B.sample_end - B.sample_begin);
  const unsigned long long px = w / S;
  const uint32_t j = (uint32_t)B.sample_begin + (uint32_t)(w - px * S);
  const unsigned long long wx = (unsigned long long)(P.x1 - P.x0);
  const int y = P.y0 + (int)(px / wx), x = P.x0 + (int)(px % wx);
  const uint32_t pixel = (uint32_t)y * (uint32_t)P.width + (uint32_t)x;
  d3 ro, rd;
  camera_ray<Generic>(P, x, y, pixel, j, ro, rd);
  double* out = B.rays_out + w * 6ull;
  out[0] = ro.x; out[1] = ro.y; out[2] = ro.z;
  out[3] = rd.x; out[4] = rd.y; out[5] = rd.z;
  if (B.keys_out) { B.keys_out[2ull * w] = pixel; B.keys_out[2ull * w + 1ull] = j; }
}

}  // namespace

cudaError_t rtrb_launch_trace_rays(const FrameParams& P, const RayBatch& B, bool strict, int capacity, cudaStream_t s) {
  const bool det = P.count_detail != 0, bvh = P.use_bvh != 0;
  RayKernel k = nullptr;
  switch (capacity) {
    case 1: k = fast_trace<1>(det, bvh); break;
    case 10: k = strict ? strict_trace<10>(det) : fast_trace<10>(det, bvh); break;
    case 32: k = strict ? strict_trace<32>(det) : fast_trace<32>(det, bvh); break;
    case kMaxStack: k = strict ? strict_trace<kMaxStack>(det) : fast_trace<kMaxStack>(det, bvh); break;
    default: return cudaErrorInvalidValue;
  }
  return launch_cover(k, (unsigned long long)B.n, kBlock, 0, false, s, P, B);
}

cudaError_t rtrb_launch_intersect_rays(const FrameParams& P, const RayBatch& B, bool strict, cudaStream_t s) {
  RayKernel k = strict ? intersect_rays_kernel<true, false>
                       : (P.use_bvh ? intersect_rays_kernel<false, true> : intersect_rays_kernel<false, false>);
  return launch_cover(k, (unsigned long long)B.n, kBlock, 0, false, s, P, B);
}

cudaError_t rtrb_launch_camera_rays(const FrameParams& P, const RayBatch& B, cudaStream_t s) {
  return launch_cover(camera_rays_kernel, (unsigned long long)B.n, kBlock, 0, false, s, P, B);
}
