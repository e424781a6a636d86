// rtrb_trace_fast.cu — RTRB_PREC_FAST64 dispatch (FP32 filter + exact FP64 refine).  The kernels of each class build
// and work-stack capacity are instantiated in their own translation unit (rtrb_trace_fast_launch.cuh).
#include "rtrb_trace_fast_launch.cuh"

// A persistent-THREAD variant (single lanes refetch a new sample when their stack empties) was measured in round 1
// and rejected: it mixed unrelated rays into one warp (22.9 instead of 29.1 of 32 lanes active on config 3).  Round 2
// measured warp-granular refill as well (profiles/README.md): also rejected.

namespace {

// Every build that exists, the most specialised class first within each capacity: a frame runs the first build of
// its capacity whose class it belongs to.
const FastKernels* const kBuilds[] = {
    &rtrb_fast_lean::d1, &rtrb_fast::d1,
    &rtrb_fast_l1n::t10, &rtrb_fast_l1::t10, &rtrb_fast::t10,
    &rtrb_fast_l1n::t32, &rtrb_fast_l1::t32, &rtrb_fast::t32,
    &rtrb_fast::t128,
};

const FastKernels* build_for(const FrameParams& P, int capacity) {
  const bool one_light = (P.scene_class & RTRB_SCENE_CLASS_ONE_LIGHT) != 0;
  const bool lean = (P.scene_class & RTRB_SCENE_CLASS_LEAN) != 0;
  for (const FastKernels* k : kBuilds)
    if (k->capacity == capacity && (one_light || !k->one_light) && (lean || !k->lean) && (P.mc == 0 || !k->no_mc)) return k;
  return nullptr;
}

}  // namespace

cudaError_t rtrb_launch_trace_pre_fast(const FrameParams& P, int capacity, cudaStream_t s, bool overlap) {
  const FastKernels* k = build_for(P, capacity);
  if (!k) return cudaErrorInvalidValue;
  if (overlap && k->capacity != 1) return cudaErrorInvalidValue;  // only the depth-1 kernels wait before their writes
  // one thread per (pixel, sample); the ray-tree kernels run lockstep CTAs (rtrb_trace_fast.cuh, trace_pre_tree_body),
  // more and smaller ones on small frames
  unsigned long long threads = pre_threads(P);
  // sky-fill frames (FrameParams::sky_fill_tiles): the traced tiles' pixels, then the CTAs that store the sky runs
  if (P.sky_fill_tiles != 0u)
    threads = ((unsigned long long)P.sky_fill_traced * (RTRB_SUPER_PIXELS / kBlock) +
               (P.sky_fill_tiles + RTRB_SKY_FILL_TILES - 1) / RTRB_SKY_FILL_TILES) * kBlock;
  int block = kBlock;
  if (k->capacity > 1) block = threads < 4ull * (unsigned long long)sm_count() * kTreeBlock ? RTRB_TREE_MIN_BLOCK : kTreeBlock;
  // in-CTA resolve (ray-tree frames only): the host only selects it for sample counts that divide both CTA sizes
  const bool in_cta = P.fuse_resolve == RTRB_RESOLVE_IN_CTA;
  if (in_cta && (block % P.pre) != 0) return cudaErrorInvalidConfiguration;
  const size_t smem = in_cta ? (size_t)block * 3u * sizeof(double) : 0u;
  return launch_cover(k->pre[P.count_detail != 0][P.use_bvh != 0], threads, block, smem, overlap, s, P);
}

cudaError_t rtrb_launch_trace_extra_fast(const FrameParams& P, int capacity, cudaStream_t s) {
  const FastKernels* k = build_for(P, capacity);
  if (!k) return cudaErrorInvalidValue;
  const TraceKernel kernel = k->extra[P.count_detail != 0][P.use_bvh != 0];
  kernel<<<extra_grid(), kBlock, 0, s>>>(P);
  return cudaGetLastError();
}

cudaError_t rtrb_launch_trace_pass_fast(const FrameParams& P, int capacity, cudaStream_t s) {
  const FastKernels* k = nullptr;
  for (const FastKernels* g : {&rtrb_fast::d1, &rtrb_fast::t10, &rtrb_fast::t32, &rtrb_fast::t128})
    if (g->capacity == capacity) k = g;
  if (!k) return cudaErrorInvalidValue;
  // the pre kernels' launch shape for the pass's samples (the lockstep CTAs of the ray-tree kernels included)
  const unsigned long long threads = pass_threads(P);
  int block = kBlock;
  if (k->capacity > 1) block = threads < 4ull * (unsigned long long)sm_count() * kTreeBlock ? RTRB_TREE_MIN_BLOCK : kTreeBlock;
  return launch_cover(k->pass[P.count_detail != 0][P.use_bvh != 0], threads, block, 0, false, s, P);
}
