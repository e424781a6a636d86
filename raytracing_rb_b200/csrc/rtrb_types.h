// rtrb_types.h — device-side data layout shared by the host API (rtrb_api.cu) and the kernels.
//
// Scene data is baked ONCE at rtrb_renderer_create into flat arrays (DESIGN.md "Data layout"):
//   geom[]  : one 64-byte record per world object, in world.yml order, read by every lane of a warp
//             at the same index (broadcast) while scanning objects (World#intersect world.rb:44-57,
//             World#lit_area world.rb:64-67);
//   mat[]   : one record per object, read only for the object a ray actually hit;
//   lights[]: one record per light;
//   textures: 8-bit RGB rows, texel = v8/256.0 (texture.rb:19).
#pragma once
#include <stdint.h>

#include "rtrb_bvh.h"
#include "rtrb_cull_tables.h"

#define RTRB_MAX_LIGHTS 64
#define RTRB_SUPER 32                 // super-tile edge in pixels (tile partition unit across GPUs)
#define RTRB_SUPER_PIXELS (RTRB_SUPER * RTRB_SUPER)
#define RTRB_APEX_MAX 32              // linear-filter scenes (<= 32 spheres) get apex tables, see FrameParams
#define RTRB_K_PLANES 8               // ... have at most this many planes
#define RTRB_K_LIGHTS 2               // ... and at most this many lights (anything larger runs the BVH kernels)
#define RTRB_SCENE_CLASS_ONE_LIGHT 1
#define RTRB_SCENE_CLASS_LEAN 2
#define RTRB_TREE_MIN_BLOCK 128        // smallest CTA the ray-tree kernels are launched with (the largest is 512): a
                                      // pre_sample_times that divides it has every sample of a pixel in one CTA
#define RTRB_SKY_FILL_TILES 4         // sky tiles one fill CTA of a sky-fill frame stores (FrameParams::sky_fill_tiles)

struct DevGeom {      // 64 B
  double px, py, pz;  // sphere centre / plane point
  double radius;      // sphere radius (0 for planes)
  double nx, ny, nz;  // plane front (unnormalised, as the reference keeps it)
  int32_t type;       // RTRB_OBJ_*
  int32_t aux;        // box: index into FrameParams::boxes
};

// One bounded face of a Box (box.rb:22-73): a Plane.create_from_scratch with front / up / point / units
// assigned, `left` from Plane#reinit (plane.rb:21-23), and the two unit vectors Plane#get_uv forms.
struct DevBoxFace {   // 112 B
  double px, py, pz;  // point
  double nx, ny, nz;  // front (unnormalised)
  double lx, ly, lz;  // normalize(normalize(front x up))   plane.rb:22,82
  double ux, uy, uz;  // normalize(up)                      plane.rb:83
  double u_unit, v_unit;
};
struct DevBox { DevBoxFace f[6]; };  // up, bottom, front, back, left, right (box.rb:60-65)

struct DevMat {
  double diffuse[3], refl[3], refr[3], ambient[3];
  double refractive_rate;
  // texture frame: sphere (sphere.rb:111-120): e0 = greenwich^, e1 = ninety_degree_east^, e2 = north^
  //                plane  (plane.rb:81-85):    e0 = left^ (normalised twice, as upstream), e1 = up^
  double e0[3], e1[3], e2[3];
  double u_unit, v_unit;
  double hscale, vscale, uoff, voff;
  double plane_nn[3];   // plane only: normalize(front); normalize(-front) is its exact negation
  const uint8_t* tex;   // device pointer to rows of RGB8, or nullptr
  int32_t tex_w, tex_h;
  int32_t has_refraction;
  int32_t plane_nn_valid;  // 0 when front is the zero vector: the runtime normalize must run (and flag)
};

struct DevLight {
  double px, py, pz;
  double color[3];
  double color_hl[3];   // color * high_light_rate (world.rb:94)
  double radius;
  double hl_threshold;  // high_light_angle / 180.0 * PI (world.rb:92)
};

typedef RtrbLightF DevLightF;  // FP32 view of a light for the highlight filter (rtrb_trace_fast.cuh)

// Per-frame constants: thin-lens camera baked on the host in the reference's evaluation order
// (camera.rb:129-151) + sampling + tiling.  Passed by value as a __grid_constant__ kernel parameter.
struct FrameParams {
  // camera
  double pos[3];
  double front[3];          // as given (focal-plane normal, camera.rb:144)
  double left[3];           // normalize(up x front)            camera.rb:130
  double left_n[3];         // normalize(left)                  camera.rb:136
  double up_n[3];           // normalize(up)
  double retina_center[3];  // pos - front^ * image_distance    camera.rb:131
  double focal_point[3];    // pos + front^ * object_distance   camera.rb:143
  double retina_width, retina_height, aperture_radius;
  double variant_threshold;
  int32_t width, height;
  int32_t pre, max_samples;
  int32_t trace_depth, mc;
  // world
  double max_distance, soft_shadow_exponent;
  int32_t n_objects, n_lights;
  const DevGeom* geom;
  const DevMat* mat;
  const DevLight* lights;
  const DevBox* boxes;         // [n_boxes], indexed by DevGeom::aux
  // FP32 filter view (FAST64): spheres and planes split by type, original indices kept
  const float4* cull_sph;      // [n_sph] (cx, cy, cz, R); sign bit of R set = bounding sphere of a box:
                               //         the line test applies, "certain hit" conclusions do not
  const int32_t* sph_index;    // [n_sph] index in world_objects
  const float4* cull_pl;       // [2*n_pl] (nx, ny, nz, |n|_1), (px, py, pz, |P|_inf)
  const int32_t* pl_index;     // [n_pl]
  const DevLightF* lights_f;   // [n_lights]
  const struct BvhNode* bvh;   // sphere BVH over cull_sph[] (rtrb_bvh.h); node 0 = root
  int32_t n_sph, n_pl;
  int32_t use_bvh;             // > RTRB_BVH_MIN_SPHERES spheres: BVH kernels; else the linear-scan kernels
  int32_t scene_class;         // what is known about the scene (rtrb_trace.cuh, "build policies"):
                               // bit 0 = exactly one light and soft_shadow_exponent == 2; bit 1 = that and: the
                               // light's radius is exactly 0 and no object is textured.  Selects kernel builds
                               // without the code the class cannot reach; results are the generic kernels' bit for bit
  // Apex tables (linear-filter scenes only): rays that pass through a known point A — primary rays
  // through the lens centre (within aperture_radius), shadow probes through their light — test sphere k
  // with b = v.u, survive unless b*b < Kq, where (v, Kq) = (C - A, |v|^2 - (R + margins)^2 - slack)
  // is precomputed per (apex, sphere).  cam_tab lives in the kernel parameters (constant bank).
  float4 cam_tab[RTRB_APEX_MAX];
  const float4* light_tab;     // [n_lights][n_sph] or nullptr
  int32_t cam_tab_valid, pad_tab;
  float m_scene;               // max over spheres of |C|_inf + R  (error-bound scale)
  float max_distance_f;        // max_distance rounded up to float
  // rng
  uint32_t key0, key1;
  // work domain
  int32_t x0, y0, x1, y1;      // window
  int32_t n_tiles;             // super-tiles assigned to this renderer for this frame
  int32_t stx_count;           // super-tiles per row of the full image
  const int32_t* tiles;        // [n_tiles] super-tile coordinates packed as tx | ty << 16
  const double* lens_sx;       // [width]  2.0 * (x.to_f / width - 0.5) * retina_width    camera.rb:133
  const double* lens_sy;       // [height] 2 * (y.to_f / height - 0.5) * retina_height    camera.rb:134
  // outputs / scratch
  double* samples;             // [n_tiles * 1024 * S][3] per-sample colours of the current pass
  double* rgb;                 // [H][W][3] or nullptr
  int32_t* hit;                // [H][W] or nullptr
  uint8_t* rgba;               // [H][W][4] (may be a peer mapping)
  unsigned long long* counters;// RTRB_CNT_* u64 counters
  uint32_t* status;            // [0] status bits, [1] max stack
  unsigned long long* first_bad;// max over flagged pixels of ~(x*H + y)  (0 = none)
  // adaptive pass
  uint32_t* extra_count;       // number of pixels taking the extra-sample branch
  uint32_t* extra_list;        // [n_tiles*1024] pixel slots (tile k * 1024 + q)
  double* extra_samples;       // [extra][max-pre][3]
  double* pre_avg;             // [extra][3] mean of the pre samples of the queued pixels, stored by the kernel that
                               // queued them (rtrb_trace.cuh, queue_adaptive)
  unsigned long long* work_counter;  // [2] spare work-claim counters (zeroed with the control block)
  int32_t count_detail;
  int32_t fuse_resolve;        // RTRB_RESOLVE_*: who finishes render_at
  int32_t pixel_format;        // RTRB_FMT_*: 4 (RGBA8) or 3 (RGB8) bytes per pixel in `rgba`
  // whole frame on one renderer: tile k is (k % stx_count, k / stx_count), no table load at kernel start;
  // k / stx_count == __umulhi(k, tiles_magic), verified on the host for every k < n_tiles
  uint32_t tiles_magic;        // 0 = use tiles[]
  unsigned long long* hot;     // [RTRB_HOT_SLICES][2] sliced (rays, shadow queries) counters
  // frame overlap (rtrb_api.cu, render_impl): the control block of the next frame on this stream, zeroed by CTA 0 of
  // a depth-1 FAST64 kernel once the frame before it has completed, instead of a memset between the two launches
  unsigned long long* ctl_next;  // [ctl_next_words] or nullptr
  uint32_t ctl_next_words, pad_next;
  // RTRB_RNG_MT (stream-exact validation mode): the reference's MT19937 doubles, generated on the host, and
  // for every pixel of the window in the reference's order (x outer, y inner) where its draws start
  const double* mt_stream;     // [mt_len] genrand_res53 values after init_genrand(seed)
  const uint32_t* mt_offset;   // [window pixels] first draw of pixel (x - x0) * (y1 - y0) + (y - y0)
  uint32_t* mt_count;          // [window pixels] out: draws the pixel consumed (0xFFFFFFFF = ran past mt_len)
  uint32_t mt_len, pad_mt;
  // SMALL-SCENE TABLES IN THE CONSTANT BANK.  The linear-filter kernels only run scenes with <= RTRB_APEX_MAX
  // spheres (+ boxes), <= RTRB_K_PLANES planes and <= RTRB_K_LIGHTS lights, and read every per-ray table from
  // here instead of global memory: uniform LDC/LDCU instead of LDG (L1 is cold at every launch boundary, and a
  // frame is one ~0.1 ms launch).  The BVH kernels ignore these fields.
  float4 k_cull_sph[RTRB_APEX_MAX];                  // = cull_sph[]
  float4 k_cull_pl[2 * RTRB_K_PLANES];               // = cull_pl[]
  DevLight k_lights[RTRB_K_LIGHTS];                  // = lights[]
  DevLightF k_lights_f[RTRB_K_LIGHTS];               // = lights_f[]
  int32_t k_pl_index[RTRB_K_PLANES];                 // = pl_index[]
  int32_t k_has_light_tab, pad_k;
  // progressive frames (rtrb_progressive_pass): the pass kernels trace samples j in [pass_begin, pass_end) of every
  // slot into samples[slot * pre + j]; `pre` stays the frame's pre_sample_times (the buffer's stride)
  int32_t pass_begin, pass_end;
  // Candidate masks of the depth-1 linear-filter kernels (rtrb_cull_tables.h): camera rays of super-tile (tx, ty) need
  // the apex test only for the spheres in k_cam_tx[tx] & k_cam_ty[ty] (tiles beyond the last entry share it), shadow
  // probes of light l only for those in light_cand's bins of their direction.  Every set bit is a sphere < n_sph.
  uint32_t k_cam_tx[RTRB_CAM_TX], k_cam_ty[RTRB_CAM_TY];  // valid with cam_tab_valid (all spheres: aperture frames)
  const uint32_t* light_cand;  // [n_lights][3 axes][2 ratios][RTRB_LIGHT_BINS], valid with k_has_light_tab
  // Tile certificates of the same kernels (rtrb_tile_rows): for super-tile column tx < RTRB_CAM_TX, the camera rays of
  // every super-tile row ty in [x, y) certainly meet no plane and no highlight cone, and those of rows [z, w) no
  // highlight cone.  A tile of the first kind whose candidate mask is empty is sky: its pixels are black, hit id -1.
  // All zero (no rows) for aperture frames and where the bounds do not hold; columns past the table share nothing.
  uchar4 k_tile_rows[RTRB_CAM_TX];
  // Ground certificates (rtrb_ground_rows; scenes with exactly one plane): in rows [x, y) of column tx, a tile whose
  // candidate mask is empty sends its camera rays to the exact test of plane 0 alone, with no highlight.  All zero =
  // nothing.
  uchar2 k_ground_rows[RTRB_CAM_TX];
  // Sky fill (rtrb_sky_fill; depth-1 FAST64 linear-filter frames resolved in the thread, whole frame on one renderer,
  // pinhole camera): the grid is 8 CTAs for each of the sky_fill_traced tiles outside the sky runs k_sky_run (one run of
  // columns per super-tile row), in row-major order (k_trace_before[r]: those of the rows < r), then
  // ceil(sky_fill_tiles / RTRB_SKY_FILL_TILES) CTAs that store the runs' tiles without tracing.  sky_fill_tiles == 0:
  // the one-thread-per-pixel grid over every tile, as for every other frame.
  uchar2 k_sky_run[RTRB_CAM_TY];
  uint16_t k_trace_before[RTRB_CAM_TY];
  uint32_t sky_fill_tiles, sky_fill_traced;
};

static_assert(sizeof(FrameParams) <= 4096, "FrameParams must fit the 4 KB kernel-parameter space");

// FrameParams::fuse_resolve: who finishes render_at (camera.rb:79-98) after the first sample loop
enum {
  RTRB_RESOLVE_SAMPLE_BUFFER = 0,  // resolve_kernel, from the per-sample buffer
  RTRB_RESOLVE_IN_THREAD = 1,      // the trace kernel: one sample per pixel and a positive threshold, so the mean is
                                   // the sample and the variance 0 can never take the extra-sample branch
  RTRB_RESOLVE_IN_CTA = 2,         // the ray-tree kernels, in the CTA that traced the pixel's samples (ordered mean
                                   // and variance test from shared memory)
};

#define RTRB_HOT_SLICES 64     // one atomic per warp lands on one of 64 address pairs (no L2 atomic hot spot)

enum {
  RTRB_CNT_SAMPLES = 0, RTRB_CNT_RAYS, RTRB_CNT_SHADOW, RTRB_CNT_HIGHLIGHT, RTRB_CNT_HITS, RTRB_CNT_LOCAL,
  RTRB_CNT_LIT, RTRB_CNT_MC, RTRB_CNT_REFR, RTRB_CNT_TEXEL, RTRB_CNT_SPH_TEST, RTRB_CNT_SPH_ACC,
  RTRB_CNT_PL_TEST, RTRB_CNT_PL_ACC, RTRB_CNT_COV_SPH, RTRB_CNT_COV_SPH_FULL, RTRB_CNT_COV_SPH_PEN,
  RTRB_CNT_COV_PL, RTRB_CNT_COV_PL_ACC, RTRB_CNT_ADAPTIVE, RTRB_CNT_EXACT,
  RTRB_CNT_BOX_TEST, RTRB_CNT_BOX_ACC, RTRB_CNT_COV_BOX, RTRB_CNT_COV_BOX_ACC, RTRB_CNT_N
};

// Morton decode of the 10-bit in-super-tile index q: even bits -> x, odd bits -> y, so that 32
// consecutive q cover an 8x4 pixel block (warp-coherent tile ordering).
__host__ __device__ inline void rtrb_morton_decode(uint32_t q, int* qx, int* qy) {
  uint32_t x = q & 0x155u, y = (q >> 1) & 0x155u;
  x = (x | (x >> 1)) & 0x133u; x = (x | (x >> 2)) & 0x10Fu; x = (x | (x >> 4)) & 0x1Fu;
  y = (y | (y >> 1)) & 0x133u; y = (y | (y >> 2)) & 0x10Fu; y = (y | (y >> 4)) & 0x1Fu;
  *qx = (int)x; *qy = (int)y;
}
__host__ __device__ inline uint32_t rtrb_morton_encode(int qx, int qy) {
  uint32_t x = (uint32_t)qx & 0x1Fu, y = (uint32_t)qy & 0x1Fu;
  x = (x | (x << 4)) & 0x10Fu; x = (x | (x << 2)) & 0x133u; x = (x | (x << 1)) & 0x155u;
  y = (y | (y << 4)) & 0x10Fu; y = (y | (y << 2)) & 0x133u; y = (y | (y << 1)) & 0x155u;
  return x | (y << 1);
}
