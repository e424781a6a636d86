/*
 * rtrb_b200.c — Ruby C extension: the thin shim between the reference's Ruby classes and the CUDA
 * tracing core (include/rtrb_b200.h).  Same shape as the reference's only native component
 * (ext/fast_4d_matrix/fast_4d_matrix.c): `Init_<name>` registers methods on a module; objects are
 * wrapped C pointers (Data_Wrap_Struct with a dfree hook, fast_4d_matrix.c:68); errors surface as
 * rb_raise(rb_eRuntimeError, ...) (fast_4d_matrix.c:124).
 *
 * It only FLATTENS: it reads World's @world_objects / @lights / scalars and Camera's accessors
 * (camera.rb:17-24), turns every Vec3 into three doubles through #to_a (fast_4d_matrix.c:86-96) and
 * calls the C ABI.  No tracing arithmetic lives here.  NOT compiled in this repository's image (no
 * ruby.h); INTEGRATION.md lists the build steps for a machine with Ruby.
 *
 *   Rtrb::Renderer.new(world)                      -> bakes the scene on GPU 0 (rtrb_renderer_create)
 *   renderer.update(world)                         -> re-bakes the world's current objects and lights in place
 *                                                     (rtrb_scene_update; nothing is queued when they did not change)
 *   renderer.render(camera, seed = 1, precision = 1) -> String of H*W*3 RGB8 bytes, row = y, col = x
 *                                                     (RTRB_FMT_RGB8: alpha is always 255, camera.rb:155)
 *   renderer.render_png(camera, seed = 1, precision = 1) -> binary String: the frame as an 8-bit RGB PNG file,
 *                                                     encoded on the GPU (only the file crosses PCIe)
 *   renderer.render_progressive(camera, schedule, seed = 1) { |rgb8, samples_done| ... }
 *                                                  -> the frame in passes (rtrb_progressive_*): after the pass to each
 *                                                     entry of `schedule` (increasing sample counts, the last one
 *                                                     pre_sample_times) yields the preview as render's RGB8 String;
 *                                                     raises as render does when the final frame raised
 *   renderer.render_progressive_png(camera, schedule, seed = 1) { |png, samples_done| ... }
 *                                                  -> the same, each preview as render_png's PNG file
 *   renderer.stats                                 -> Hash of the last frame's (or ray batch's) counters
 *   renderer.trace_rays(packed_rays, trace_depth, mc, seed = 1) -> [rgb, hits]: RayTracer#trace_sync on n rays given as
 *                                                     n*6 doubles (position, front; Array#pack("d*")); rgb = n*3 doubles,
 *                                                     hits = n int32 root-ray winners (unpack("d*") / unpack("l*"))
 *   renderer.intersect_rays(packed_rays)           -> String of n rtrb_ray_hit records (unpack("l4d7") each):
 *                                                     World#intersect's object, :in?, box face, distance, point, delta
 */
#include <ruby.h>
#include <ruby/thread.h>
#include <stdlib.h>
#include <string.h>

#include "rtrb_b200.h"

static VALUE mRtrb, cRenderer;

typedef struct {
  rtrb_renderer* r;
  rtrb_stats last;
} shim_renderer;

static void shim_free(void* p) {
  shim_renderer* s = (shim_renderer*)p;
  if (s->r) rtrb_renderer_destroy(s->r);
  free(s);
}

static void vec3_into(VALUE v, double out[3], const char* what) {
  if (NIL_P(v)) rb_raise(rb_eTypeError, "%s is nil", what);
  VALUE a = rb_funcall(v, rb_intern("to_a"), 0);
  for (int i = 0; i < 3; ++i) out[i] = NUM2DBL(rb_ary_entry(a, i));
}
static VALUE ivar(VALUE obj, const char* name) { return rb_iv_get(obj, name); }
static double ivar_f(VALUE obj, const char* name, const char* what) {
  VALUE v = rb_iv_get(obj, name);
  if (NIL_P(v)) rb_raise(rb_eTypeError, "%s is nil", what);
  return NUM2DBL(v);
}
static int is_a(VALUE obj, const char* klass_path) { return RTEST(rb_obj_is_kind_of(obj, rb_path2class(klass_path))); }

/* Texture -> 8-bit RGB rows: Texture#to_a holds rows of Vec3(v8/256.0) (texture.rb:12-20,34-36).  Converted once per
 * Texture object: `cache` (an identity Hash held by the renderer) keeps the bytes as a String, so Renderer#update, which
 * runs before every frame, does not walk the texels again.  A Texture is never edited after it was decoded
 * (texture.rb:12-20). */
static void texture_bytes(VALUE tex, VALUE cache, rtrb_texture_desc* td) {
  const int w = NUM2INT(rb_funcall(tex, rb_intern("width"), 0));
  const int h = NUM2INT(rb_funcall(tex, rb_intern("height"), 0));
  VALUE bytes = rb_hash_aref(cache, tex);
  if (NIL_P(bytes)) {
    VALUE rows = rb_funcall(tex, rb_intern("to_a"), 0);
    bytes = rb_str_new(NULL, (long)w * h * 3);
    uint8_t* px = (uint8_t*)RSTRING_PTR(bytes);
    for (int y = 0; y < h; ++y) {
      VALUE row = rb_ary_entry(rows, y);
      for (int x = 0; x < w; ++x) {
        double c[3];
        vec3_into(rb_ary_entry(row, x), c, "texel");
        for (int k = 0; k < 3; ++k) px[((size_t)y * w + x) * 3 + k] = (uint8_t)(c[k] * 256.0 + 0.5);
      }
    }
    rb_hash_aset(cache, tex, bytes);  /* only once complete */
  }
  td->rgb8 = (const uint8_t*)RSTRING_PTR(bytes); td->width = w; td->height = h;
}

/* Flattening World -> rtrb_scene_desc can raise half way (a nil ivar, a non-numeric value: vec3_into / ivar_f call
 * rb_raise).  The scratch arrays therefore live in a struct that rb_ensure frees whether the body returns or raises
 * (texture bytes belong to the renderer's cache). */
typedef struct {
  VALUE self, world, texture_cache;
  rtrb_object_desc* od;
  rtrb_light_desc* ld;
  rtrb_texture_desc* td;
  int n_tex;
} init_call;

static VALUE init_cleanup(VALUE p) {
  init_call* c = (init_call*)p;
  free(c->od); free(c->ld); free(c->td);
  return Qnil;
}

/* World -> rtrb_scene_desc: what Renderer.new and Renderer#update hand to the library.  The scratch arrays stay in `c`
 * until its rb_ensure cleanup runs. */
static void flatten_world(init_call* c, rtrb_scene_desc* sd) {
  VALUE world = c->world;
  VALUE objs = ivar(world, "@world_objects"), lights = ivar(world, "@lights");
  long n_obj = RARRAY_LEN(objs), n_li = RARRAY_LEN(lights);
  rtrb_object_desc* od = c->od = (rtrb_object_desc*)calloc(n_obj > 0 ? n_obj : 1, sizeof(*od));
  rtrb_light_desc* ld = c->ld = (rtrb_light_desc*)calloc(n_li > 0 ? n_li : 1, sizeof(*ld));
  rtrb_texture_desc* td = c->td = (rtrb_texture_desc*)calloc(n_obj > 0 ? n_obj : 1, sizeof(*td));
  if (!od || !ld || !td) rb_raise(rb_eNoMemError, "rtrb_b200: scene scratch");
  for (long i = 0; i < n_obj; ++i) {
    VALUE o = rb_ary_entry(objs, i);
    rtrb_object_desc* d = &od[i];
    d->texture = -1;
    VALUE tex = ivar(o, "@texture");
    if (!NIL_P(tex)) {
      d->texture = c->n_tex++;
      texture_bytes(tex, c->texture_cache, &td[d->texture]);
      /* what Texture#color really uses (texture.rb:9-10,15-16,24-25): the Texture object's own scales and offsets.
       * Sphere passes its texture_u/v_offset on (sphere.rb:25); Plane and Box do not (plane.rb:35, box.rb:76), so
       * their textures keep 0.0 whatever the YAML says. */
      d->texture_horizontal_scale = ivar_f(tex, "@horizontal_scale", "texture horizontal_scale");
      d->texture_vertical_scale = ivar_f(tex, "@vertical_scale", "texture vertical_scale");
      d->texture_u_offset = ivar_f(tex, "@u_off", "texture u_off");
      d->texture_v_offset = ivar_f(tex, "@v_off", "texture v_off");
    }
    if (is_a(o, "Alex::Objects::Sphere")) {
      d->type = RTRB_OBJ_SPHERE;
      d->has_refraction = 1;
      vec3_into(ivar(o, "@center"), d->point, "center");
      d->radius = ivar_f(o, "@radius", "radius");
      d->refractive_rate = ivar_f(o, "@refractive_rate", "refractive_rate");   /* sphere.rb:93 */
      if (d->texture >= 0) {
        vec3_into(ivar(o, "@greenwich_vec"), d->greenwich_vec, "greenwich_vec");
        vec3_into(ivar(o, "@north_pole_vec"), d->north_pole_vec, "north_pole_vec");
      }
    } else if (is_a(o, "Alex::Objects::Plane")) {
      d->type = RTRB_OBJ_PLANE;
      vec3_into(ivar(o, "@point"), d->point, "point");
      vec3_into(ivar(o, "@front"), d->front, "front");
      vec3_into(ivar(o, "@up"), d->up, "up");
      VALUE uu = ivar(o, "@u_unit"), vu = ivar(o, "@v_unit"), rr = ivar(o, "@refractive_rate");
      d->u_unit = NIL_P(uu) ? 1.0 : NUM2DBL(uu);
      d->v_unit = NIL_P(vu) ? 1.0 : NUM2DBL(vu);
      d->has_refraction = RTEST(rr) ? 1 : 0;                                    /* plane.rb:57 */
      if (d->has_refraction) d->refractive_rate = NUM2DBL(rr);
    } else if (is_a(o, "Alex::Objects::Box")) {
      /* box.rb:10: the library derives the six faces exactly as Box#initialize does (box.rb:22-73) */
      d->type = RTRB_OBJ_BOX;
      d->texture = -1;                                                          /* Box never samples its texture */
      vec3_into(ivar(o, "@point"), d->point, "point");
      vec3_into(ivar(o, "@front"), d->front, "front");
      vec3_into(ivar(o, "@up"), d->up, "up");
      d->width_front = ivar_f(o, "@width_front", "width_front");
      d->width_up = ivar_f(o, "@width_up", "width_up");
      d->width_left = ivar_f(o, "@width_left", "width_left");
      VALUE rr = ivar(o, "@refractive_rate");
      d->has_refraction = RTEST(rr) ? 1 : 0;                                    /* plane.rb:57 on every face */
      if (d->has_refraction) d->refractive_rate = NUM2DBL(rr);
    } else {
      rb_raise(rb_eNotImpError, "object %ld: only Sphere, Plane and Box run on the GPU path", i);
    }
    vec3_into(ivar(o, "@diffuse_rate"), d->diffuse_rate, "diffuse_rate");
    vec3_into(ivar(o, "@reflective_attenuation"), d->reflective_attenuation, "reflective_attenuation");
    vec3_into(ivar(o, "@ambient"), d->ambient, "ambient");
    if (!NIL_P(ivar(o, "@refractive_attenuation")))
      vec3_into(ivar(o, "@refractive_attenuation"), d->refractive_attenuation, "refractive_attenuation");
  }
  for (long i = 0; i < n_li; ++i) {
    VALUE l = rb_ary_entry(lights, i);
    vec3_into(ivar(l, "@position"), ld[i].position, "light position");
    vec3_into(ivar(l, "@color"), ld[i].color, "light color");
    ld[i].radius = ivar_f(l, "@radius", "radius");
    ld[i].high_light_rate = ivar_f(l, "@high_light_rate", "high_light_rate");
    ld[i].high_light_angle = ivar_f(l, "@high_light_angle", "high_light_angle");
  }
  memset(sd, 0, sizeof(*sd));
  sd->max_distance = ivar_f(world, "@max_distance", "max_distance");
  sd->soft_shadow_exponent = ivar_f(world, "@soft_shadow_exponent", "soft_shadow_exponent");
  sd->n_objects = (int32_t)n_obj; sd->n_lights = (int32_t)n_li; sd->n_textures = c->n_tex;
  sd->objects = od; sd->lights = ld; sd->textures = td;
}

static VALUE init_body(VALUE p) {
  init_call* c = (init_call*)p;
  rtrb_scene_desc sd;
  flatten_world(c, &sd);
  shim_renderer* s;
  Data_Get_Struct(c->self, shim_renderer, s);
  int rc = rtrb_renderer_create(&sd, 0, &s->r);
  if (rc != RTRB_OK) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());
  return c->self;
}

/* The library compares the new bake with the current one: an unchanged world queues nothing. */
static VALUE update_body(VALUE p) {
  init_call* c = (init_call*)p;
  rtrb_scene_desc sd;
  flatten_world(c, &sd);
  shim_renderer* s;
  Data_Get_Struct(c->self, shim_renderer, s);
  int rc = rtrb_scene_update(s->r, &sd, NULL);
  if (rc != RTRB_OK) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());
  return c->self;
}

/* The renderer's Texture -> bytes cache (texture_bytes), made on first use. */
static VALUE texture_cache(VALUE self) {
  VALUE cache = rb_iv_get(self, "@texture_bytes");
  if (NIL_P(cache)) {
    cache = rb_hash_new();
    rb_funcall(cache, rb_intern("compare_by_identity"), 0);
    rb_iv_set(self, "@texture_bytes", cache);
  }
  return cache;
}

static VALUE renderer_initialize(VALUE self, VALUE world) {
  init_call c;
  memset(&c, 0, sizeof(c));
  c.self = self; c.world = world; c.texture_cache = texture_cache(self);
  return rb_ensure(init_body, (VALUE)&c, init_cleanup, (VALUE)&c);
}

static VALUE renderer_update(VALUE self, VALUE world) {
  init_call c;
  memset(&c, 0, sizeof(c));
  c.self = self; c.world = world; c.texture_cache = texture_cache(self);
  return rb_ensure(update_body, (VALUE)&c, init_cleanup, (VALUE)&c);
}

static VALUE renderer_alloc(VALUE klass) {
  shim_renderer* s = (shim_renderer*)calloc(1, sizeof(*s));
  return Data_Wrap_Struct(klass, 0, shim_free, s);
}

typedef struct {
  shim_renderer* s;
  rtrb_camera_desc cam;
  rtrb_render_opts opts;
  uint8_t* rgba;
  int rc;
  size_t capacity, png_bytes;  /* render_png */
} render_call;

static void* render_without_gvl(void* p) {   /* one blocking call per frame; the GVL is released */
  render_call* c = (render_call*)p;
  c->rc = rtrb_render(c->s->r, &c->cam, &c->opts, c->rgba, NULL, NULL, &c->s->last);
  return NULL;
}

static void* render_png_without_gvl(void* p) {  /* render into device memory, encode there, fetch the file */
  render_call* c = (render_call*)p;
  c->rc = rtrb_render_device(c->s->r, &c->cam, &c->opts, &c->s->last);
  if (c->rc != RTRB_OK && c->rc != RTRB_ERR_RAISED) return NULL;
  const int raised = c->rc == RTRB_ERR_RAISED;
  c->rc = rtrb_encode_png(c->s->r, NULL, c->cam.width, c->cam.height, c->opts.pixel_format, NULL, c->rgba, c->capacity,
                          &c->png_bytes);
  if (c->rc == RTRB_OK && raised) c->rc = RTRB_ERR_RAISED;
  return NULL;
}

/* (camera, seed = 1, precision = 1) -> the frame call's camera and options (RTRB_FMT_RGB8) */
static void frame_call(int argc, VALUE* argv, VALUE self, render_call* cp) {
  VALUE camera, seed, precision;
  rb_scan_args(argc, argv, "12", &camera, &seed, &precision);
  shim_renderer* s;
  Data_Get_Struct(self, shim_renderer, s);
  render_call c;
  memset(&c, 0, sizeof(c));
  c.s = s;
  vec3_into(rb_funcall(camera, rb_intern("position"), 0), c.cam.position, "position");
  vec3_into(rb_funcall(camera, rb_intern("up"), 0), c.cam.up, "up");
  vec3_into(rb_funcall(camera, rb_intern("front"), 0), c.cam.front, "front");
#define CAMF(field) c.cam.field = NUM2DBL(rb_funcall(camera, rb_intern(#field), 0))
#define CAMI(field) c.cam.field = NUM2INT(rb_funcall(camera, rb_intern(#field), 0))
  CAMF(retina_width); CAMF(retina_height); CAMF(aperture_radius); CAMF(image_distance); CAMF(focal_distance);
  CAMF(variant_threshold);
  CAMI(width); CAMI(height); CAMI(pre_sample_times); CAMI(max_sample_times); CAMI(trace_depth);
  CAMI(monte_carlo_diffusion_times);
  c.opts.rng_mode = RTRB_RNG_CTR;
  c.opts.seed = NIL_P(seed) ? 1 : NUM2ULL(seed);                 /* main.rb:10 Random.srand(1) */
  c.opts.precision = NIL_P(precision) ? RTRB_PREC_DEFAULT : NUM2INT(precision);
  c.opts.pixel_format = RTRB_FMT_RGB8;                           /* alpha = 255 never crosses PCIe */
  *cp = c;
}

static VALUE renderer_render(int argc, VALUE* argv, VALUE self) {
  render_call c;
  frame_call(argc, argv, self, &c);
  size_t bytes = (size_t)c.cam.width * c.cam.height * 3;
  VALUE out = rb_str_new(NULL, (long)bytes);
  c.rgba = (uint8_t*)RSTRING_PTR(out);
  rb_thread_call_without_gvl(render_without_gvl, &c, RUBY_UBF_IO, NULL);
  if (c.rc == RTRB_ERR_RAISED) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());  /* ray_tracer.rb:295 et al. */
  if (c.rc != RTRB_OK) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());
  return out;
}

static VALUE renderer_render_png(int argc, VALUE* argv, VALUE self) {
  render_call c;
  frame_call(argc, argv, self, &c);
  c.opts.skip_outputs = RTRB_SKIP_RGB | RTRB_SKIP_HIT;           /* only the 8-bit frame is needed */
  if (rtrb_png_max_bytes(c.cam.width, c.cam.height, &c.capacity) != RTRB_OK) rb_raise(rb_eArgError, "%s", rtrb_last_error());
  VALUE out = rb_str_new(NULL, (long)c.capacity);
  c.rgba = (uint8_t*)RSTRING_PTR(out);
  rb_thread_call_without_gvl(render_png_without_gvl, &c, RUBY_UBF_IO, NULL);
  if (c.rc != RTRB_OK) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());  /* RTRB_ERR_RAISED included, as render */
  rb_str_set_len(out, (long)c.png_bytes);  /* rb_str_new strings are binary (ASCII-8BIT) */
  return out;
}

/* ---- progressive frames: one pass per schedule entry, the GVL released around each pass and its download / encode */
typedef struct {
  render_call* c;
  rtrb_progressive* p;
  VALUE schedule;
  int png;
} progressive_run;

typedef struct {
  render_call* c;
  rtrb_progressive* p;
  int sample_end, png;
} pass_call;

static void* pass_without_gvl(void* q) {
  pass_call* pc = (pass_call*)q;
  render_call* c = pc->c;
  c->rc = rtrb_progressive_pass(pc->p, pc->sample_end, &c->s->last);
  if (c->rc != RTRB_OK && c->rc != RTRB_ERR_RAISED) return NULL;
  const int raised = c->rc == RTRB_ERR_RAISED;
  if (pc->png) {
    void* src = NULL;
    c->rc = rtrb_progressive_frame_ptr(pc->p, &src);
    if (c->rc == RTRB_OK)
      c->rc = rtrb_encode_png(c->s->r, src, c->cam.width, c->cam.height, c->opts.pixel_format, NULL, c->rgba, c->capacity,
                              &c->png_bytes);
  } else {
    c->rc = rtrb_progressive_download(pc->p, c->rgba, NULL, NULL);
  }
  if (c->rc == RTRB_OK && raised) c->rc = RTRB_ERR_RAISED;
  return NULL;
}

static VALUE progressive_body(VALUE q) {
  progressive_run* run = (progressive_run*)q;
  render_call* c = run->c;
  const long n = RARRAY_LEN(run->schedule);
  for (long i = 0; i < n; ++i) {
    pass_call pc = {c, run->p, NUM2INT(rb_ary_entry(run->schedule, i)), run->png};
    const size_t bytes = run->png ? c->capacity : (size_t)c->cam.width * c->cam.height * 3;
    VALUE out = rb_str_new(NULL, (long)bytes);
    c->rgba = (uint8_t*)RSTRING_PTR(out);
    rb_thread_call_without_gvl(pass_without_gvl, &pc, RUBY_UBF_IO, NULL);
    const int final = pc.sample_end == c->cam.pre_sample_times;
    if (c->rc != RTRB_OK && c->rc != RTRB_ERR_RAISED) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());
    if (run->png) rb_str_set_len(out, (long)c->png_bytes);
    rb_yield_values(2, out, INT2NUM(pc.sample_end));
    if (final && c->rc == RTRB_ERR_RAISED) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());  /* as render */
  }
  return Qnil;
}

static VALUE progressive_cleanup(VALUE q) {
  rtrb_progressive_destroy(((progressive_run*)q)->p);
  return Qnil;
}

static VALUE renderer_progressive(int argc, VALUE* argv, VALUE self, int png) {
  VALUE camera, schedule, seed;
  rb_scan_args(argc, argv, "21", &camera, &schedule, &seed);
  Check_Type(schedule, T_ARRAY);
  rb_need_block();
  VALUE args[2] = {camera, seed};
  render_call c;
  frame_call(2, args, self, &c);
  c.opts.skip_outputs = RTRB_SKIP_RGB | RTRB_SKIP_HIT;           /* only the 8-bit frame is needed */
  if (png && rtrb_png_max_bytes(c.cam.width, c.cam.height, &c.capacity) != RTRB_OK)
    rb_raise(rb_eArgError, "%s", rtrb_last_error());
  progressive_run run = {&c, NULL, schedule, png};
  if (rtrb_progressive_create(c.s->r, &c.cam, &c.opts, &run.p) != RTRB_OK) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());
  return rb_ensure(progressive_body, (VALUE)&run, progressive_cleanup, (VALUE)&run);
}

static VALUE renderer_render_progressive(int argc, VALUE* argv, VALUE self) { return renderer_progressive(argc, argv, self, 0); }
static VALUE renderer_render_progressive_png(int argc, VALUE* argv, VALUE self) { return renderer_progressive(argc, argv, self, 1); }

typedef struct {
  shim_renderer* s;
  rtrb_ray_opts opts;
  int n;
  const rtrb_ray* rays;
  double* rgb;
  int32_t* hit;
  rtrb_ray_hit* hits;
  int rc;
} ray_call;

static void* trace_rays_without_gvl(void* p) {   /* one blocking call per batch; the GVL is released */
  ray_call* c = (ray_call*)p;
  c->rc = rtrb_trace_rays(c->s->r, &c->opts, c->n, c->rays, NULL, c->rgb, c->hit, &c->s->last);
  return NULL;
}

static void* intersect_rays_without_gvl(void* p) {
  ray_call* c = (ray_call*)p;
  c->rc = rtrb_intersect_rays(c->s->r, &c->opts, c->n, c->rays, c->hits);
  return NULL;
}

/* packed_rays: a String of n * 6 doubles -> the call's rays (the String must stay referenced while the call runs) */
static void ray_call_init(VALUE self, VALUE packed_rays, ray_call* c) {
  StringValue(packed_rays);
  if (RSTRING_LEN(packed_rays) % (long)sizeof(rtrb_ray) != 0)
    rb_raise(rb_eArgError, "packed rays must be a multiple of 48 bytes (6 doubles: position, front)");
  memset(c, 0, sizeof(*c));
  Data_Get_Struct(self, shim_renderer, c->s);
  c->n = (int)(RSTRING_LEN(packed_rays) / (long)sizeof(rtrb_ray));
  c->rays = (const rtrb_ray*)RSTRING_PTR(packed_rays);
  c->opts.precision = RTRB_PREC_DEFAULT;
}

static VALUE renderer_trace_rays(int argc, VALUE* argv, VALUE self) {
  VALUE packed, depth, mc, seed;
  rb_scan_args(argc, argv, "31", &packed, &depth, &mc, &seed);
  ray_call c;
  ray_call_init(self, packed, &c);
  c.opts.trace_depth = NUM2INT(depth);
  c.opts.monte_carlo_diffusion_times = NUM2INT(mc);
  c.opts.seed = NIL_P(seed) ? 1 : NUM2ULL(seed);
  VALUE rgb = rb_str_new(NULL, (long)c.n * 3 * (long)sizeof(double));
  VALUE hit = rb_str_new(NULL, (long)c.n * (long)sizeof(int32_t));
  c.rgb = (double*)RSTRING_PTR(rgb);
  c.hit = (int32_t*)RSTRING_PTR(hit);
  rb_thread_call_without_gvl(trace_rays_without_gvl, &c, RUBY_UBF_IO, NULL);
  RB_GC_GUARD(packed);
  if (c.rc != RTRB_OK) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());  /* RTRB_ERR_RAISED included, as render */
  return rb_ary_new_from_args(2, rgb, hit);
}

static VALUE renderer_intersect_rays(VALUE self, VALUE packed) {
  ray_call c;
  ray_call_init(self, packed, &c);
  VALUE out = rb_str_new(NULL, (long)c.n * (long)sizeof(rtrb_ray_hit));
  c.hits = (rtrb_ray_hit*)RSTRING_PTR(out);
  rb_thread_call_without_gvl(intersect_rays_without_gvl, &c, RUBY_UBF_IO, NULL);
  RB_GC_GUARD(packed);
  if (c.rc != RTRB_OK) rb_raise(rb_eRuntimeError, "%s", rtrb_last_error());
  return out;
}

static VALUE renderer_stats(VALUE self) {
  shim_renderer* s;
  Data_Get_Struct(self, shim_renderer, s);
  VALUE h = rb_hash_new();
#define PUT(k) rb_hash_aset(h, ID2SYM(rb_intern(#k)), ULL2NUM(s->last.k))
  PUT(samples); PUT(rays); PUT(shadow_queries); PUT(highlight_hits); PUT(hits); PUT(local_shaded); PUT(texel_fetches);
  PUT(adaptive_pixels); PUT(box_tests); PUT(box_accepts);
  rb_hash_aset(h, ID2SYM(rb_intern("device_ms")), DBL2NUM(s->last.device_ms));
  rb_hash_aset(h, ID2SYM(rb_intern("status")), UINT2NUM(s->last.status));
  return h;
}

void Init_rtrb_b200(void) {
  mRtrb = rb_define_module("Rtrb");
  cRenderer = rb_define_class_under(mRtrb, "Renderer", rb_cObject);
  rb_define_alloc_func(cRenderer, renderer_alloc);
  rb_define_method(cRenderer, "initialize", renderer_initialize, 1);
  rb_define_method(cRenderer, "update", renderer_update, 1);
  rb_define_method(cRenderer, "render", renderer_render, -1);
  rb_define_method(cRenderer, "render_png", renderer_render_png, -1);
  rb_define_method(cRenderer, "render_progressive", renderer_render_progressive, -1);
  rb_define_method(cRenderer, "render_progressive_png", renderer_render_progressive_png, -1);
  rb_define_method(cRenderer, "stats", renderer_stats, 0);
  rb_define_method(cRenderer, "trace_rays", renderer_trace_rays, -1);
  rb_define_method(cRenderer, "intersect_rays", renderer_intersect_rays, 1);
  rb_define_const(mRtrb, "ABI_VERSION", INT2NUM(rtrb_abi_version()));
}
