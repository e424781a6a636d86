// oracle_rays.cpp — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// Ray-level entry points of the CPU oracle for the tests of rtrb_trace_rays / rtrb_intersect_rays: the oracle's own
// RayTracer#trace_sync and World#intersect (oracle/rtrb_oracle.cpp, included unchanged) on caller-supplied rays.
// tests/rays_oracle.py compiles this file with the oracle's flags (-ffp-contract=off) into a temporary directory.
#include "../oracle/rtrb_oracle.cpp"

extern "C" {

// RayTracer#trace_sync (ray_tracer.rb:16-46) on n rays, rays = n x (position(3), front(3)).  Ray i draws its
// Monte-Carlo rays from the Philox counter (keys[2i], keys[2i+1], path, 1), or (i, 0, path, 1) without keys, as the
// device does.  rgb: n x 3, hit: n root-ray winners.  Counters and status as for a frame of height 1: the first
// offending ray is first_bad_x.  Returns RTRB_ERR_RAISED when some ray would have raised.
int rtrb_oracle_trace_rays(void* scene, int trace_depth, int mc, uint64_t seed, int n, const double* rays,
                           const uint32_t* keys, double* rgb, int32_t* hit, rtrb_stats* stats) {
  const OracleScene* s = (const OracleScene*)scene;
  Ctx ctx;
  ctx.H = 1;
  g_ctx = &ctx;
  RngState rng;
  rng.mode = RTRB_RNG_CTR;
  rng.k0 = (uint32_t)seed; rng.k1 = (uint32_t)(seed >> 32);
  RayTracer rt{&s->world, trace_depth, mc, &rng};
  for (int i = 0; i < n; ++i) {
    ctx.cur_x = i; ctx.cur_y = 0;
    rng.pixel = keys ? keys[2 * (size_t)i] : (uint32_t)i;
    rng.sample = keys ? keys[2 * (size_t)i + 1] : 0u;
    Ray ray{v3(rays + 6 * (size_t)i + 3), v3(rays + 6 * (size_t)i)};
    int ph = -1;
    V3 c = rt.trace_sync(ray, &ph);
    for (int k = 0; k < 3; ++k) rgb[3 * (size_t)i + k] = c.v[k];
    hit[i] = ph;
  }
  g_ctx = nullptr;
  const Counters& c = ctx.cnt;
  std::memset(stats, 0, sizeof(*stats));
  stats->samples = c.samples; stats->rays = c.rays; stats->shadow_queries = c.shadow_queries;
  stats->highlight_hits = c.highlight_hits; stats->hits = c.hits; stats->local_shaded = c.local_shaded;
  stats->lit_lights = c.lit_lights; stats->mc_rays = c.mc_rays; stats->refractions = c.refractions;
  stats->texel_fetches = c.texel_fetches; stats->sphere_tests = c.sphere_tests; stats->sphere_accepts = c.sphere_accepts;
  stats->plane_tests = c.plane_tests; stats->plane_accepts = c.plane_accepts; stats->cover_sphere = c.cover_sphere;
  stats->cover_sphere_full = c.cover_sphere_full; stats->cover_sphere_penumbra = c.cover_sphere_penumbra;
  stats->cover_plane = c.cover_plane; stats->cover_plane_accepts = c.cover_plane_accepts;
  stats->box_tests = c.box_tests; stats->box_accepts = c.box_accepts;
  stats->cover_box = c.cover_box; stats->cover_box_accepts = c.cover_box_accepts;
  stats->max_stack = c.max_stack;
  stats->status = ctx.status;
  stats->first_bad_x = ctx.first_bad < 0 ? -1 : (int32_t)ctx.first_bad;
  stats->first_bad_y = ctx.first_bad < 0 ? -1 : 0;
  return ctx.status ? RTRB_ERR_RAISED : RTRB_OK;
}

// World#intersect (world.rb:37-59) with everything rtrb_ray_hit reports: the winning object (-1 = miss) and
// out7 = Ray#distance(intersection), intersection(3), delta(3); *dir_in = :in; *face = Box#intersect's data[:index]
// (-1 unless a box won).
int rtrb_oracle_world_intersect_full(void* scene, const double* o, const double* d, double* out7, int* dir_in, int* face) {
  Ctx ctx;
  g_ctx = &ctx;
  const OracleScene* s = (const OracleScene*)scene;
  Ray ray{v3(d), v3(o)};
  Hit h;
  const WorldObject* w = s->world.intersect(ray, &h);
  g_ctx = nullptr;
  *dir_in = 0; *face = -1;
  for (int i = 0; i < 7; ++i) out7[i] = 0.0;
  if (!w) return -1;
  out7[0] = ray.distance(h.intersection);
  for (int i = 0; i < 3; ++i) { out7[1 + i] = h.intersection.v[i]; out7[4 + i] = h.delta.v[i]; }
  *dir_in = h.dir_in ? 1 : 0;
  *face = h.data_index;
  return w->index;
}

}  // extern "C"
