// rtrb_rays.h — launchers of the ray-level kernels (rtrb_rays.cu): RayTracer#trace_sync and World#intersect on rays
// the caller supplies, and Camera#lens_func for a window of pixels.  rtrb_api.cu validates the arguments, fills the
// FrameParams (scene part as for frames, cam_tab_valid = 0) and owns the buffers.
#pragma once
#include <cuda_runtime.h>

#include "../../include/rtrb_b200.h"
#include "rtrb_types.h"

// The per-call arrays of a ray kernel (device pointers).  A ray is six doubles, position then front (rtrb_ray).
struct RayBatch {
  const double* rays;      // [n][6] trace_rays / intersect_rays input
  const uint32_t* keys;    // [n][2] (pixel, sample) RNG keys of trace_rays, or nullptr: ray i is keyed (i, 0)
  double* rgb;             // [n][3] trace_rays: rt_reduce's unclamped colour
  int32_t* hit;            // [n] trace_rays: the root ray's World#intersect winner (-1 miss, -2 highlight), or nullptr
  rtrb_ray_hit* hits;      // [n] intersect_rays
  double* rays_out;        // [n][6] camera_rays
  uint32_t* keys_out;      // [n][2] camera_rays, or nullptr
  long long n;             // rays
  int32_t sample_begin, sample_end;  // camera_rays: samples j in [sample_begin, sample_end) of every window pixel
};

// capacity = trace_capacity() of the batch (rtrb_launch.h), as for frames.  P.count_detail selects the kernels with the
// full counters (and the Box code); P.use_bvh the sphere filter.
cudaError_t rtrb_launch_trace_rays(const FrameParams& P, const RayBatch& B, bool strict, int capacity, cudaStream_t s);
cudaError_t rtrb_launch_intersect_rays(const FrameParams& P, const RayBatch& B, bool strict, cudaStream_t s);
// one thread per (window pixel, sample); P holds the baked camera, the window and the lens tables
cudaError_t rtrb_launch_camera_rays(const FrameParams& P, const RayBatch& B, cudaStream_t s);
