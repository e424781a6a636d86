/*
 * rtrb_b200.h — C ABI of the B200 tracing core for raytracing_rb's per-pixel hot path.
 *
 * One call per FRAME replaces the reference's per-pixel loop
 *   Camera#render_sync / render_fork -> Camera#render_at -> RayTracer#trace_sync
 *   (reference src/camera.rb:41-110, src/ray_tracer.rb:16-164, src/world.rb:37-98,
 *    src/objects/{world_object,sphere,plane,texture}.rb, ext/fast_4d_matrix/fast_4d_matrix.c:57-305).
 *
 * The reference has no FFI for this path; its only native-extension convention is
 * ext/fast_4d_matrix (extconf.rb:5,16 + fast_4d_matrix.c:29 `Init_fast_4d_matrix`).  The Ruby
 * shim that follows the same convention and binds exactly these entry points is in
 * ext/rtrb_b200/rtrb_b200.c; INTEGRATION.md shows how Camera/World hand their ivars over.
 *
 * Conventions (mirroring fast_4d_matrix.c's rb_raise style at :124,:220,:291):
 *   - every function returns an int status, 0 = RTRB_OK; rtrb_last_error() gives the message
 *     for the calling thread.
 *   - plain pointers and sizes only; the caller owns every output buffer.
 *   - all scene numbers are FP64 because the reference is FP64 end to end.
 *   - there is NO CPU fallback: every entry point that computes fails with RTRB_ERR_CUDA when
 *     no CUDA device is usable.
 */
#ifndef RTRB_B200_H
#define RTRB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTRB_ABI_VERSION 4

/* ---- status codes ------------------------------------------------------------------------- */
enum {
  RTRB_OK = 0,
  RTRB_ERR_INVALID = 1,   /* bad argument / scene the reference itself would reject (TypeError etc.) */
  RTRB_ERR_CUDA = 2,      /* CUDA runtime failure or no device */
  RTRB_ERR_RAISED = 3,    /* frame finished, but the reference would have raised (see rtrb_stats.status) */
  RTRB_ERR_UNSUPPORTED = 4
};

/* ---- per-frame status word: the reference's raise sites, one bit each ---------------------- */
enum {
  RTRB_ST_COLOR_GT_1 = 1u << 0,   /* ray_tracer.rb:294-296 'color greater than 1' */
  RTRB_ST_ZERO_VECTOR = 1u << 1,  /* fast_4d_matrix.c:123-124,290-291 and world_object.rb:106 */
  RTRB_ST_MATH_DOMAIN = 1u << 2,  /* Math.sqrt / Math.acos / Math.asin outside their domain */
  RTRB_ST_STACK_OVERFLOW = 1u << 3, /* device bounce stack exceeded (not a reference condition) */
  RTRB_ST_NAN_TO_INT = 1u << 4    /* texture.rb:24-25 Float#to_i on NaN/Infinity (FloatDomainError) */
};

/* ---- object kinds (world.yml `type:`; world.rb:28-34) -------------------------------------- */
enum { RTRB_OBJ_PLANE = 0, RTRB_OBJ_SPHERE = 1, RTRB_OBJ_BOX = 2 };

/* ---- RNG modes ----------------------------------------------------------------------------- */
enum {
  RTRB_RNG_CTR = 0,  /* Philox4x32-10 keyed by (seed; pixel, sample, ray path, purpose); device + oracle */
  RTRB_RNG_MT = 1    /* MT19937 genrand_res53 in the reference's consumption order (Random.srand(seed), main.rb:10;
                        one draw per lens_func, camera.rb:135, two per Monte-Carlo ray, world_object.rb:84; pixels x
                        outer / y inner, rays LIFO).  Stream-exact VALIDATION mode: blocking calls only, one GPU,
                        STRICT arithmetic, one thread per pixel, iterated to the fixed point of the per-pixel
                        stream offsets (the draw counts are data dependent).  Seeds must fit 32 bits. */
};

/* ---- rtrb_render_opts.pixel_format: layout of the 8-bit frame -------------------------------- */
enum {
  RTRB_FMT_RGBA8 = 0, /* H*W*4 bytes, alpha = 255: what array_to_color builds (camera.rb:153-156) */
  RTRB_FMT_RGB8 = 1,  /* H*W*3 bytes: alpha is the constant 255, so it need not cross PCIe; the caller
                         (Camera#render_cuda) re-inserts it when it fills the PNG canvas */
  RTRB_FMT_PNG_RGB8 = 2 /* H rows of 1 + 3*W bytes: the PNG filter-type byte 0 ("None") followed by the row's RGB8
                         pixels, i.e. exactly the byte stream a PNG encoder deflates into IDAT for an 8-bit RGB image
                         (what Camera#save_image, camera.rb:36-39, produces through the png gem): the host only runs
                         zlib over the buffer and frames the chunks */
};
/* bytes of one 8-bit frame in `format` */
#define RTRB_FRAME_BYTES(width, height, format) \
  ((format) == RTRB_FMT_RGBA8 ? (size_t)(width) * (height) * 4 : (format) == RTRB_FMT_RGB8 ? (size_t)(width) * (height) * 3 \
                                                               : (size_t)(height) * ((size_t)(width) * 3 + 1))

/* ---- rtrb_render_opts.skip_outputs ----------------------------------------------------------- */
enum { RTRB_SKIP_RGB = 1, RTRB_SKIP_HIT = 2 };

/* ---- arithmetic modes of the device path ---------------------------------------------------- */
enum {
  RTRB_PREC_STRICT = 0,   /* FP64, no FMA contraction, every div/sqrt as the reference writes it */
  RTRB_PREC_FAST64 = 1,   /* FP64 decisions identical to STRICT (FP32 cull + exact FP64 refine) */
  RTRB_PREC_DEFAULT = 1
};

/* One entry of world.yml `world_objects` (plane.rb:9-15, sphere.rb:8-14, box.rb:10-14), order preserved:
 * World#intersect's strict `<` (world.rb:48) makes the lowest index win distance ties. */
typedef struct rtrb_object_desc {
  int32_t type;            /* RTRB_OBJ_* */
  int32_t texture;         /* index into rtrb_scene_desc.textures, -1 = untextured */
  int32_t has_refraction;  /* plane / box: refractive_rate key present (plane.rb:57); sphere: must be 1 */
  int32_t reserved0;
  double point[3];         /* sphere: center ; plane: point ; box: point (its centre) */
  double radius;           /* sphere only */
  double front[3];         /* plane normal / box front axis, NOT normalised by the reference */
  double up[3];            /* plane / box `up` */
  double u_unit, v_unit;   /* plane uv units (plane.rb:81-85) */
  double greenwich_vec[3]; /* sphere texture frame (sphere.rb:111-120) */
  double north_pole_vec[3];
  double texture_horizontal_scale, texture_vertical_scale;
  double texture_u_offset, texture_v_offset; /* 0.0 when absent (texture.rb:15-16) */
  double refractive_rate;
  double diffuse_rate[3];
  double reflective_attenuation[3];
  double refractive_attenuation[3];
  double ambient[3];
  /* box only (box.rb:10,22-58): extents along front / up / normalize(front x up).  The six bounded
   * faces are derived by the library exactly as Box#initialize does.  A box ignores `texture`
   * (Box never overrides local_lighting, world_object.rb:51-74 runs without a colour filter). */
  double width_front, width_up, width_left;
} rtrb_object_desc;

/* One entry of world.yml `lights` (lights/light.rb:3-4, spot_light.rb:5). */
typedef struct rtrb_light_desc {
  double position[3];
  double color[3];
  double radius;
  double high_light_rate;
  double high_light_angle; /* degrees */
} rtrb_light_desc;

/* Decoded texture (texture.rb:12-20): 8-bit RGB rows, texel = v8/256.0, alpha ignored. */
typedef struct rtrb_texture_desc {
  int32_t width, height;   /* columns, rows */
  const uint8_t* rgb8;     /* height*width*3, row-major */
} rtrb_texture_desc;

typedef struct rtrb_scene_desc {
  double max_distance;          /* world.yml:1  */
  double soft_shadow_exponent;  /* world.yml:2  */
  int32_t n_objects, n_lights, n_textures, reserved0;
  const rtrb_object_desc* objects;
  const rtrb_light_desc* lights;
  const rtrb_texture_desc* textures;
} rtrb_scene_desc;

/* camera.yml (camera.rb:17-24). retina_* are HALF extents (camera.rb:133-134). */
typedef struct rtrb_camera_desc {
  double position[3], up[3], front[3];
  double retina_width, retina_height;
  double aperture_radius, image_distance, focal_distance;
  double variant_threshold;
  int32_t width, height;
  int32_t pre_sample_times, max_sample_times;
  int32_t trace_depth, monte_carlo_diffusion_times;
} rtrb_camera_desc;

typedef struct rtrb_render_opts {
  int32_t rng_mode;     /* RTRB_RNG_* */
  int32_t precision;    /* RTRB_PREC_* */
  uint64_t seed;        /* main.rb:10 uses Random.srand(1) */
  /* window of pixels to render, x in [x0,x1), y in [y0,y1); all zero = whole frame.
   * A column strip is exactly render_fork's child_work (camera.rb:53-65). */
  int32_t x0, y0, x1, y1;
  /* image-tile partition (replaces fork_jobs row farming): this call renders the 32x32-pixel
   * super-tiles number tile_rank, tile_rank + tile_world, ... of the window (row-major order; see
   * rtrb_tile_partition). tile_world <= 1 = everything. */
  int32_t tile_rank, tile_world;
  int32_t count_detail; /* 1 = fill every rtrb_stats counter (slower); 0 = rays/shadow/samples only */
  int32_t skip_outputs; /* rtrb_render_device only: RTRB_SKIP_RGB | RTRB_SKIP_HIT drop the optional float RGB
                           (24 B/pixel) / hit-id (4 B/pixel) frames; 0 keeps both for rtrb_download */
  void* stream;         /* cudaStream_t to launch on; NULL = the renderer's own stream */
  void* rgba_device_out;/* rtrb_render_device / rtrb_submit only: device pointer (possibly a peer mapping) the 8-bit
                           frame is written to; NULL = the renderer's own framebuffer.  The host-buffer calls
                           (rtrb_render, rtrb_render_multi) reject it with RTRB_ERR_INVALID, and rtrb_download refuses
                           to fetch an 8-bit frame that went elsewhere */
  int32_t pixel_format; /* RTRB_FMT_*: layout of the 8-bit frame (device buffer and host copies alike) */
  int32_t reserved0;
} rtrb_render_opts;

typedef struct rtrb_stats {
  uint64_t samples;           /* trace_sync calls (camera.rb:75,91) */
  uint64_t rays;              /* work-stack items passing the cut at ray_tracer.rb:52 */
  uint64_t shadow_queries;    /* lit_area calls made from local_lights (world.rb:75) */
  uint64_t highlight_hits;    /* items terminated by the highlight test (ray_tracer.rb:60-75) */
  uint64_t hits;              /* items whose World#intersect found an object */
  uint64_t local_shaded;      /* local_lighting evaluations (ray_tracer.rb:152) */
  uint64_t lit_lights;        /* lights kept by local_lights (area > 0) */
  uint64_t mc_rays;           /* path_tracing rays spawned (world_object.rb:76-90) */
  uint64_t refractions;       /* refraction children created */
  uint64_t texel_fetches;     /* Texture#color calls */
  uint64_t sphere_tests, sphere_accepts;      /* Sphere#intersect from World#intersect */
  uint64_t plane_tests, plane_accepts;        /* Plane#intersect from World#intersect */
  uint64_t cover_sphere, cover_sphere_full, cover_sphere_penumbra; /* Sphere#cover_area by branch */
  uint64_t cover_plane, cover_plane_accepts;  /* WorldObject#cover_area on planes */
  uint64_t adaptive_pixels;   /* pixels taking the extra-sample branch (camera.rb:87-93) */
  uint64_t exact_tests;       /* FAST64 only: objects re-evaluated in strict FP64 after the FP32 cull */
  uint64_t box_tests, box_accepts;            /* Box#intersect from World#intersect (box.rb:78-97) */
  uint64_t cover_box, cover_box_accepts;      /* WorldObject#cover_area on boxes */
  uint32_t status;            /* RTRB_ST_* bits */
  int32_t first_bad_x, first_bad_y; /* lowest (y*W+x) pixel that set a status bit, -1 if none */
  uint32_t max_stack;         /* deepest work stack seen */
  float device_ms;            /* CUDA-event time of the frame's kernels on the launch stream (0 for rtrb_submit frames) */
  float trace_ms;             /* CUDA-event time of the dominant kernel alone (trace over the pre samples); 0 likewise */
} rtrb_stats;

typedef struct rtrb_renderer rtrb_renderer; /* opaque: scene SoA + scratch + framebuffers on ONE device */

/* -- lifecycle ------------------------------------------------------------------------------- */
int rtrb_abi_version(void);
const char* rtrb_last_error(void);
int rtrb_device_count(int* count_out);

/* Bakes the scene (derived vectors plane `left`, sphere `ninety_degree_east_vec`, unit frames) into
 * flat SoA device buffers once; replaces World#initialize's object graph (world.rb:15-34). */
int rtrb_renderer_create(const rtrb_scene_desc* scene, int device, rtrb_renderer** out);
int rtrb_renderer_destroy(rtrb_renderer* r);

/* Replaces the renderer's baked scene with `scene` (same description, rules and errors as rtrb_renderer_create), for
 * scenes that change between frames (World edits, animation).  Ordered on `stream` (NULL = the renderer's own):
 *   - every frame, rtrb_submit frame or ray call queued before the update, on any stream this renderer has launched
 *     on, sees the old scene; everything issued after it sees the new one (the first such launch on each stream
 *     waits for the update's copies, and a depth-1 frame does not overlap the kernel before it);
 *   - a stream that such a call used should outlive the next update; if it was destroyed meanwhile, that update
 *     waits for the whole device instead (the work the stream had queued still runs);
 *   - a rejected scene (RTRB_ERR_INVALID / RTRB_ERR_UNSUPPORTED) leaves the old one fully in force;
 *   - a scene whose bake equals the current one queues nothing;
 *   - framebuffers (and exported device pointers / IPC handles), pipeline slots and tickets are not touched.
 * The scene is copied from pinned staging memory: the call returns without waiting for the device, except for the
 * previous update's copies, and for its device to go idle when that update had to grow a scene buffer. */
int rtrb_scene_update(rtrb_renderer* r, const rtrb_scene_desc* scene, void* stream);

/* -- the hot path ---------------------------------------------------------------------------- */
/* Renders one frame into DEVICE buffers (async on opts->stream unless stats_out != NULL, which
 * synchronises).  Replaces the pixel loops camera.rb:59-63 and :102-106.
 * Consecutive depth-1, 1-spp FAST64 frames on one stream overlap on the device: a frame's kernel traces under the
 * tail of the previous one and stores only after it has completed (results unchanged).  RTRB_FRAME_OVERLAP=0 in the
 * environment when the renderer is created turns this off. */
int rtrb_render_device(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts,
                       rtrb_stats* stats_out);

/* Copies the last frame to HOST buffers. rgba: RTRB_FRAME_BYTES(W, H, pixel_format) bytes (H*W*4 for the default
 * RTRB_FMT_RGBA8), row = y, column = x (camera.rb:98,105);
 * rgb_or_null: H*W*3 doubles = render_at's unclamped `color`; hit_or_null: H*W int32 primary hit
 * ids (index in world_objects, -1 miss, -2 highlight-terminated, -3 pixel not rendered). */
int rtrb_download(rtrb_renderer* r, uint8_t* rgba, double* rgb_or_null, int32_t* hit_or_null);

/* render_device + download in one blocking call with HOST buffers: what Camera#render_cuda binds. */
int rtrb_render(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts,
                uint8_t* rgba, double* rgb_or_null, int32_t* hit_or_null, rtrb_stats* stats_out);

/* Pipelined form of rtrb_render for frame sequences: rtrb_submit launches the frame and queues its
 * device->host copy into rgba_host (pinned memory recommended) on a separate copy stream, then
 * returns; rtrb_wait blocks until that frame's bytes and stats are in host memory.  Up to four frames
 * may be in flight per renderer (tickets are consecutive integers; wait for them in order), so
 * later frames render while earlier ones cross PCIe.  8-bit frame only (opts->pixel_format).  rtrb_wait fails with
 * RTRB_ERR_INVALID for a ticket that is not the one occupying its slot (stale or duplicate). */
int rtrb_submit(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts, uint8_t* rgba_host,
                int* ticket_out);
int rtrb_wait(rtrb_renderer* r, int ticket, rtrb_stats* stats_out);

/* -- PNG files encoded on the device (ABI 4) ------------------------------------------------------ */
/* The encoder writes 8-bit RGB PNG files (colour type 2, no interlace; alpha is not stored because it is always 255).
 * Every row takes the PNG filter (None, Sub, Up, Average, Paeth) with the smallest sum of |signed byte|, ties to the
 * lowest type.  The filtered stream is cut into segments of RTRB_PNG_SEGMENT_BYTES that are deflated independently on
 * the device, each into the smallest of a stored, fixed-Huffman or dynamic-Huffman block (matches may reach 32 KiB
 * back into earlier segments) and one IDAT chunk; the zlib header and the Adler-32 trailer are IDAT chunks of their
 * own.  The same image always gives the same bytes. */
#define RTRB_PNG_SEGMENT_BYTES 32768

/* bytes that always suffice for a device-encoded PNG of width x height (stored-block worst case; pure host) */
int rtrb_png_max_bytes(int width, int height, size_t* bytes_out);

/* Encodes a width x height image in `pixel_format` that is in device memory: `src_device` or, if NULL, the start of
 * the renderer's framebuffer (its last frame, or a frame that tile ranks gathered there).  Ordered after the work on
 * `stream` (NULL = the renderer's own).  Blocks until exactly *bytes_out bytes of PNG file are in png_host. */
int rtrb_encode_png(rtrb_renderer* r, const void* src_device, int width, int height, int pixel_format, void* stream,
                    uint8_t* png_host, size_t capacity, size_t* bytes_out);

/* Pipelined form (the rtrb_submit slots and tickets; completed by the unchanged rtrb_wait, which also stores the
 * byte count into *png_bytes_out).  png_host must be page-locked and device-mapped.  Only the encoded bytes cross
 * PCIe: device stores through the mapped alias, as publish_ctl_kernel already does for the control block.
 * opts->pixel_format is RTRB_FMT_RGBA8 or RTRB_FMT_RGB8; opts->rgba_device_out is rejected.  The frame is encoded on
 * the renderer's copy stream, so the next frame renders meanwhile.  A frame that raises still yields its PNG. */
int rtrb_submit_png(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts, uint8_t* png_host,
                    size_t capacity, size_t* png_bytes_out, int* ticket_out);

/* -- progressive frames --------------------------------------------------------------------------- */
/* One camera plus render options whose pre_sample_times samples are traced in passes the caller chooses, with a
 * well-defined image after every pass (interactive previews, renders that stop when a time budget is spent):
 *   - Preview: after a pass that brings the frame to e < pre_sample_times samples, its outputs (the 8-bit frame in
 *     opts->pixel_format, the float RGB, the hit ids) and stats equal bit for bit those of rtrb_render_device for the
 *     same camera with pre_sample_times = max_sample_times = e, including render_at's variance test and its rescale of
 *     the adaptive pixels.
 *   - Final: the pass that reaches pre_sample_times finishes render_at as the one-shot frame does (variance test and,
 *     when max_sample_times > pre_sample_times, the extra samples of the adaptive pixels, traced whole in that pass);
 *     outputs and stats then equal rtrb_render_device of the camera as given.
 *   - Stats: a pass reports the stats of the frame its outputs equal.  Counters, status, first_bad_x/y and max_stack
 *     accumulate over the passes so far; device_ms / trace_ms cover this pass only.
 * Arguments and buffers:
 *   - opts follow the rules of rtrb_render_device: window, tile_rank / tile_world, the three pixel formats,
 *     skip_outputs, rgba_device_out and stream.  RTRB_RNG_MT returns RTRB_ERR_UNSUPPORTED.
 *   - the handle owns its scratch (the per-sample buffer [slots][pre][3] FP64, the extra-sample buffers, a control
 *     block, its tile list and lens table) and its outputs: the float RGB, the hit ids and, unless opts->rgba_device_out
 *     is given, the 8-bit frame.  Pixels outside the window or the rank's tiles read 0 and hit id -3.
 *   - frames, rtrb_submit frames, ray calls and other progressive frames on the same renderer may run between passes:
 *     they do not disturb it, and it does not disturb them.
 *   - rtrb_progressive_create fails with RTRB_ERR_UNSUPPORTED when the sample buffer exceeds the per-frame memory
 *     budget of rtrb_render_device, and with RTRB_ERR_CUDA when no CUDA device is usable.
 * Passes:
 *   - rtrb_progressive_pass traces samples [done, sample_end) of every pixel, done being the samples of the passes
 *     before it; sample_end must be in (done, pre_sample_times].  A pass after the final one returns RTRB_ERR_INVALID.
 *   - passes are ordered on opts->stream (NULL = the renderer's own) and synchronise only when stats_out != NULL,
 *     like rtrb_render_device.  They read the scene, so rtrb_scene_update orders them as it orders frames.
 *   - when rtrb_scene_update has replaced the scene since create, the next pass returns RTRB_ERR_INVALID ("scene
 *     changed"): one pixel mixing two scenes would be neither frame.  An update whose scene equals the current one
 *     does not count.
 *   - RTRB_ERR_RAISED when the frame the outputs equal would have raised (every output is written).
 * A progressive frame must be destroyed before its renderer. */
typedef struct rtrb_progressive rtrb_progressive;
int rtrb_progressive_create(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts,
                            rtrb_progressive** out);
/* samples [done, sample_end) */
int rtrb_progressive_pass(rtrb_progressive* p, int sample_end, rtrb_stats* stats_out);
/* Copies the outputs of the passes so far to HOST buffers (layouts of rtrb_download; each pointer may be NULL).
 * Blocking.  RTRB_ERR_INVALID before the first pass, for an 8-bit frame that went to rgba_device_out, and for an
 * output that skip_outputs dropped. */
int rtrb_progressive_download(rtrb_progressive* p, uint8_t* frame, double* rgb_or_null, int32_t* hit_or_null);
/* Device pointer of the 8-bit frame (its own buffer, or rgba_device_out), e.g. for rtrb_encode_png. */
int rtrb_progressive_frame_ptr(rtrb_progressive* p, void** ptr_out);
/* Waits for the device and frees the frame's buffers.  NULL is a no-op. */
int rtrb_progressive_destroy(rtrb_progressive* p);

/* -- ray-level queries on caller-supplied rays ---------------------------------------------------- */
/* The layers below the camera, for callers with their own rays (other projections, picking, probes of one ray):
 * RayTracer#trace_sync (ray_tracer.rb:16-46) and World#intersect (world.rb:37-59) on a batch of rays, one device
 * thread per ray, and Camera#lens_func (camera.rb:129-151) for a window of pixels.  Same kernels' arithmetic as the
 * frames: STRICT and FAST64 give the same bits.  The calls never touch the renderer's framebuffers, its last frame or
 * its rtrb_submit slots (they have a control block and scratch of their own); they are not pipelined and draw their
 * Monte-Carlo rays from the counter RNG only.  Every call fails with RTRB_ERR_CUDA when no CUDA device is usable. */

/* Ray(front, position) of the reference (algebra.rb); `front` is NOT normalised, as the reference keeps it. */
typedef struct rtrb_ray {
  double position[3];
  double front[3];
} rtrb_ray;

/* World#intersect's answer for one ray.  A miss has object -1, face -1 and zeros elsewhere. */
typedef struct rtrb_ray_hit {
  int32_t object;          /* index in world_objects, -1 = miss */
  int32_t direction;       /* 1 = :in, 0 = :out */
  int32_t face;            /* box: Box#intersect's data[:index] (box.rb:89: 0 up, 1 bottom, 2 front, 3 back, 4 left,
                              5 right); -1 otherwise */
  int32_t reserved0;
  double distance;         /* Ray#distance(intersection) (algebra.rb:10-12) */
  double intersection[3];
  double delta[3];         /* sphere.rb:84 / plane.rb:50 (a box: the winning face's plane) */
} rtrb_ray_hit;

/* bytes of device scratch a host-buffer ray call may use (inputs and outputs staged on the device) */
#define RTRB_RAY_SCRATCH_BUDGET ((size_t)16 << 30)

typedef struct rtrb_ray_opts {
  int32_t precision;       /* RTRB_PREC_* */
  int32_t device_buffers;  /* 0: host pointers, blocking.  1: device pointers on the renderer's device, ordered on
                              `stream`; synchronises only when stats_out != NULL (like rtrb_render_device) */
  uint64_t seed;           /* Philox key, as rtrb_render_opts.seed */
  int32_t trace_depth, monte_carlo_diffusion_times;  /* rtrb_trace_rays: the root item's depth, MC rays per bounce */
  int32_t count_detail;    /* rtrb_trace_rays: 1 = fill every rtrb_stats counter */
  int32_t x0, y0, x1, y1;  /* rtrb_camera_rays: window of pixels, x in [x0,x1), y in [y0,y1); all zero = whole frame */
  int32_t reserved0;
  void* stream;            /* cudaStream_t; NULL = the renderer's own stream */
} rtrb_ray_opts;

/* RayTracer#trace_sync on n rays: the root item has depth opts->trace_depth and attenuation (1, 1, 1).  Ray i draws its
 * Monte-Carlo rays from the Philox counter (keys[2i], keys[2i+1], path, 1), keys_or_null = NULL meaning (i, 0); a
 * frame's sample j of pixel (x, y) is keyed (y * W + x, j), so rays from rtrb_camera_rays traced with its keys reproduce
 * the frame's samples bit for bit.  rgb_out: n x 3 doubles, the unclamped rt_reduce sum; hit_or_null: n root-ray
 * World#intersect winners (-1 miss, -2 highlight-terminated).  stats_out: counters and status as for a frame of height
 * 1, so first_bad_x is the lowest offending ray index and first_bad_y is 0.  RTRB_ERR_RAISED when a ray would have
 * raised in the reference (every output is written); RTRB_ERR_UNSUPPORTED when trace_depth * (1 + mc) + 1 exceeds the
 * device work stack (128 items, as for frames) or the host-buffer scratch exceeds RTRB_RAY_SCRATCH_BUDGET. */
int rtrb_trace_rays(rtrb_renderer* r, const rtrb_ray_opts* opts, int n, const rtrb_ray* rays, const uint32_t* keys_or_null,
                    double* rgb_out, int32_t* hit_or_null, rtrb_stats* stats_out);
/* World#intersect on n rays (opts: precision, device_buffers, stream). */
int rtrb_intersect_rays(rtrb_renderer* r, const rtrb_ray_opts* opts, int n, const rtrb_ray* rays, rtrb_ray_hit* hits_out);
/* Camera#lens_func for every pixel (x, y) of the window and every sample j in [sample_begin, sample_end), with the
 * aperture angle the frame draws for that sample (Philox counter (y * W + x, j, 0, 0)).  Ray (x, y, j) is at index
 * ((y - y0) * (x1 - x0) + (x - x0)) * (sample_end - sample_begin) + (j - sample_begin); keys_or_null receives its
 * (y * W + x, j) key.  The camera's sampling and tracing fields are not used. */
int rtrb_camera_rays(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_ray_opts* opts, int sample_begin,
                     int sample_end, rtrb_ray* rays_out, uint32_t* keys_or_null);

/* -- multi-GPU tile gather without a collective ----------------------------------------------- */
/* Device pointer of the renderer's RGBA8 framebuffer for (width,height) (allocates it if needed).  From this
 * call (or rtrb_framebuffer_ipc_export) on the framebuffer is PINNED: a later frame or request that needs a larger
 * one fails with RTRB_ERR_INVALID instead of reallocating memory that peers may still be writing to. */
int rtrb_framebuffer_device_ptr(rtrb_renderer* r, int width, int height, void** ptr_out);
/* Copies width*height*4 bytes of that framebuffer to host memory (blocking).  With a framebuffer
 * allocated for (width, height * n) this fetches n frames that were rendered into consecutive slots
 * through rgba_device_out. */
int rtrb_framebuffer_download(rtrb_renderer* r, int width, int height, uint8_t* rgba_host);
/* Queues a copy of the first `bytes` bytes of that framebuffer to host memory on `stream` (NULL = the renderer's own)
 * and returns without synchronising: the last step of a multi-process tile gather, ordered on the caller's stream
 * behind whatever tells rank 0 that every rank's tiles have landed (render_fork's parent, camera.rb:42-52). */
int rtrb_framebuffer_copy_async(rtrb_renderer* r, size_t bytes, uint8_t* host, void* stream);
/* CUDA IPC handle (64 bytes) of that framebuffer, to hand to the other per-GPU processes. */
int rtrb_framebuffer_ipc_export(rtrb_renderer* r, int width, int height, uint8_t handle_out[64]);
/* Maps a peer process's framebuffer into this process; pass the result as rgba_device_out. */
int rtrb_ipc_open(int device, const uint8_t handle[64], void** ptr_out);
int rtrb_ipc_close(int device, void* ptr);
/* In-process variant: renders tile_world = n renderers (one per GPU, one host thread each) into
 * renderers[0]'s framebuffer through peer mappings, then downloads from renderers[0]. */
int rtrb_render_multi(rtrb_renderer* const* renderers, int n, const rtrb_camera_desc* cam,
                      const rtrb_render_opts* opts, uint8_t* rgba, double* rgb_or_null,
                      int32_t* hit_or_null, rtrb_stats* stats_out);

/* Copy-engine form of the gather (whole frames dealt to ranks, see DESIGN.md 8): queues a
 * device-to-device copy of `bytes` from `src` (a buffer of this renderer's device) to `dst_peer` (a
 * peer mapping, e.g. a frame slot of rank 0's framebuffer) on the renderer's copy stream, ordered
 * after everything queued so far on `after_stream` (NULL = the renderer's own stream).  The render
 * stream does not wait: the next frame renders while this one crosses NVLink. */
int rtrb_peer_push(rtrb_renderer* r, const void* src, void* dst_peer, size_t bytes, void* after_stream);
/* Makes `stream` (NULL = the renderer's own) wait for every rtrb_peer_push queued so far. */
int rtrb_peer_push_join(rtrb_renderer* r, void* stream);

/* Pure host helper (no GPU): the 32x32-pixel super-tiles of a width x height frame (optionally
 * clipped to window {x0,y0,x1,y1}, NULL = whole frame) that tile_rank renders out of tile_world,
 * as global ids ty * ceil(width/32) + tx in ascending order.  count_out receives the number of
 * tiles even when it exceeds capacity.  This is the partition rtrb_render_device applies. */
int rtrb_tile_partition(int width, int height, const int32_t* window_or_null, int tile_rank, int tile_world,
                        int32_t* tiles_out, int capacity, int* count_out);

/* -- measurement helpers ---------------------------------------------------------------------- */
/* Dependent-free FMA issue microbenchmark on `device`: the roofline denominator SURVEY.md 8d asks
 * for. which: 0 = FP32 FFMA, 1 = FP64 DFMA. Result in TFLOP/s (2 flops per FMA). */
int rtrb_measure_fma_peak(int device, int which, double* tflops_out);
/* Passes the last RTRB_RNG_MT frame of this renderer needed to reach its fixed point (0 if none yet). */
int rtrb_last_mt_passes(rtrb_renderer* r);
/* Number of kernel launches issued by this library in this process so far. */
uint64_t rtrb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* RTRB_B200_H */
