// rtrb_trace_fast.cuh — RTRB_PREC_FAST64: the same ray tree, evaluated "filter then exact".
//
// Every per-object decision of the reference (does object i win World#intersect, does object i
// contribute to lit_area, does a light match the highlight test) is first bounded in FP32 with a
// rigorous error margin; only the objects the filter cannot exclude are re-evaluated with the
// STRICT FP64 functions of rtrb_trace.cuh.  Objects the filter excludes contribute exactly what the
// reference computes for them (no hit / cover 0 / no match), so the frame is bit-identical to
// STRICT; the filter only removes FP64 work (DESIGN.md "FAST64", with the error-bound derivation).
//
// Further exact-preserving economies, each justified where it is made:
//   * FP64 ray normalisation (1 sqrt + 3 div) is deferred until an exact sphere test needs it;
//   * children that cannot survive the cut at ray_tracer.rb:52 are not computed;
//   * divisions by exactly 1.0 (one light) are skipped; the attenuation cut avoids its sqrt
//     outside a narrow band around the threshold.
// What a scene / frame class fixes comes from the build policy (rtrb_trace.cuh, "build policies").
//
// Compiled with -fmad=false as well: the exact parts must not contract; the FP32 filter uses
// explicit fmaf().
#pragma once
#include "rtrb_trace.cuh"

namespace rtrb {

__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// A ray as the FP32 filter sees it: origin, direction normalised IN FP32 (|d| = 1 +- 4 eps), and
// E = 96 * 2^-24 * (M_scene + |O|_inf): an absolute bound on the FP32 error of every length the
// sphere filter forms (DESIGN.md derives <= 45 eps M; 96 leaves slack for the approximate MUFU ops).
struct CullRay {
  float ox, oy, oz, dx, dy, dz, E, mo;
};
__device__ __forceinline__ CullRay make_cull_ray(const FrameParams& P, d3 o, d3 d) {
  CullRay r;
  r.ox = (float)o.x; r.oy = (float)o.y; r.oz = (float)o.z;
  const float fx = (float)d.x, fy = (float)d.y, fz = (float)d.z;
  const float inv = rsqrt_approx(fmaf(fz, fz, fmaf(fy, fy, fx * fx)));
  r.dx = fx * inv; r.dy = fy * inv; r.dz = fz * inv;
  r.mo = fmaxf(fabsf(r.ox), fmaxf(fabsf(r.oy), fabsf(r.oz)));
  r.E = 5.7220459e-6f * (P.m_scene + r.mo);  // 96 * 2^-24
  return r;
}

// Hot reject test of the sphere filter: true when the ray's LINE certainly passes farther than R from
// the centre.  !(m2 > ...) keeps NaNs as survivors.
__device__ __forceinline__ bool sphere_line_misses(const float4 s, const CullRay& r) {
  const float ocx = s.x - r.ox, ocy = s.y - r.oy, ocz = s.z - r.oz;
  const float b = fmaf(ocz, r.dz, fmaf(ocy, r.dy, ocx * r.dx));
  const float qx = fmaf(-b, r.dx, ocx), qy = fmaf(-b, r.dy, ocy), qz = fmaf(-b, r.dz, ocz);
  const float m2 = fmaf(qz, qz, fmaf(qy, qy, qx * qx));
  const float Rp = fabsf(s.w) + r.E;  // sign bit = "bounding sphere of a box"
  return m2 > Rp * Rp;
}

// Full sphere classification (survivors only). 0 = certainly no hit, 1 = possible hit (lo valid),
// 2 = certain hit (lo, hi valid).  lo/hi bound Ray#distance(intersection) of Sphere#intersect.
template <bool BOX = true>
__device__ __forceinline__ int classify_sphere(const float4 s, const CullRay& r, float& lo, float& hi) {
  const float ocx = s.x - r.ox, ocy = s.y - r.oy, ocz = s.z - r.oz;
  const float b = fmaf(ocz, r.dz, fmaf(ocy, r.dy, ocx * r.dx));
  const float qx = fmaf(-b, r.dx, ocx), qy = fmaf(-b, r.dy, ocy), qz = fmaf(-b, r.dz, ocz);
  const float m2 = fmaf(qz, qz, fmaf(qy, qy, qx * qx));
  const bool bound_only = BOX && __float_as_int(s.w) < 0;  // a box's bounding sphere: never a certain hit
  const float R = BOX ? fabsf(s.w) : s.w;
  const float Rp = R + r.E;
  if (m2 > Rp * Rp) return 0;
  const float oc2 = fmaf(ocz, ocz, fmaf(ocy, ocy, ocx * ocx));
  const float Rm = fmaxf(R - r.E, 0.0f);
  const bool outside = oc2 > Rp * Rp;
  const bool inside = oc2 < Rm * Rm;
  if (outside && b < -r.E) return 0;  // centre behind an outside origin: `!from_inner && t < 0`
  const float m = sqrt_approx(m2);
  const float mlo = fmaxf(m - r.E, 0.0f), mhi = m + r.E;
  const float h_hi = sqrt_approx(fmaxf(fmaf(Rp, Rp, -mlo * mlo), 0.0f)) * 1.000001f + r.E;
  const float h_lo = sqrt_approx(fmaxf(fmaf(Rm, Rm, -mhi * mhi), 0.0f)) * 0.999999f;
  int kind;
  if (outside) {
    lo = b - h_hi - r.E;
    hi = b - h_lo + r.E;
    kind = (mhi < Rm && b > r.E) ? 2 : 1;
  } else if (inside) {
    lo = b + h_lo - r.E;
    hi = b + h_hi + r.E;
    kind = 2;
  } else {
    lo = b - h_hi - r.E;  // origin within the margin of the surface: either root is possible
    hi = 0.0f;
    kind = 1;
  }
  lo = fmaxf(lo, 0.0f);
  if (bound_only) {  // whatever is inside the sphere is met no earlier than the sphere's entry point
    kind = 1; hi = 0.0f;
    if (!outside) lo = 0.0f;
  }
  if (!(lo == lo) || !(hi == hi)) { lo = 0.0f; kind = 1; }  // NaN anywhere: leave it to the exact test
  return kind;
}

// Plane filter, same contract; a = (n, |n|_1), p = (P, |P|_inf).  Plane#intersect (plane.rb:38-51).
__device__ __forceinline__ int classify_plane(const float4 a, const float4 p, const CullRay& r, float& lo, float& hi) {
  const float eps = 5.9604645e-8f;  // 2^-24
  const float den = fmaf(a.z, r.dz, fmaf(a.y, r.dy, a.x * r.dx));
  const float rx = p.x - r.ox, ry = p.y - r.oy, rz = p.z - r.oz;
  const float num = fmaf(rz, a.z, fmaf(ry, a.y, rx * a.x));
  const float e_num = 16.0f * eps * a.w * (p.w + r.mo);
  const float e_den = 16.0f * eps * a.w;
  const float aden = fabsf(den);
  lo = 0.0f; hi = 0.0f;
  if (!(aden > 16.0f * e_den)) return 1;  // grazing (or NaN): the exact test decides
  const float inv = rcp_approx(den);
  const float t = num * inv;
  // |den_true| >= 15/16 |den| here, hence the 1.1
  const float e_t = (e_num + fabsf(t) * e_den) * fabsf(inv) * 1.1f + 8.0f * eps * fabsf(t);
  if (t + e_t < 0.0f) return 0;
  lo = fmaxf(t - e_t, 0.0f);
  hi = t + e_t;
  if (!(lo == lo) || !(hi == hi)) { lo = 0.0f; return 1; }
  return (t - e_t > 0.0f) ? 2 : 1;
}

// bh = h; the face byte only exists for kernels that carry the Box code
template <bool BOX>
__device__ __forceinline__ void keep_hit(HitRec& bh, const HitRec& h) {
  bh.p = h.p; bh.dir_in = h.dir_in;
  if constexpr (BOX) bh.face = h.face;
}

// Up to 8 survivor slots of 16 bits each, kept in two registers (no local-memory array).
struct Pack8 {
  unsigned long long a, b;
  int n;
  __device__ __forceinline__ void clear() { a = 0ull; b = 0ull; n = 0; }
  __device__ __forceinline__ void push(uint32_t v) {
    if (n < 4) a |= (unsigned long long)v << (16 * n);
    else if (n < 8) b |= (unsigned long long)v << (16 * (n - 4));
    n++;
  }
  __device__ __forceinline__ bool overflow() const { return n > 8; }
  __device__ __forceinline__ uint32_t get(int i) const {
    return (uint32_t)(((i < 4) ? (a >> (16 * i)) : (b >> (16 * (i - 4)))) & 0xffffull);
  }
};

// The reference's own scan (world.rb:44-57); used when the filter keeps more survivors than fit.
template <class Pol, bool BOX>
static __device__ __noinline__ int closest_hit_scan(const FrameParams& P, d3 o, d3 d, HitRec& bh, ThreadCtx& ctx) {
  const double d_r = norm(d);
  const d3 dn = mk(d.x / d_r, d.y / d_r, d.z / d_r);
  double best = P.max_distance;
  int best_i = -1;
  for (int i = 0; i < P.n_objects; ++i) {
    const DevGeom g = P.geom[i];
    HitRec h;
    bool ok;
    double den;
    if (g.type == RTRB_OBJ_SPHERE) ok = sphere_intersect<Pol>(g, o, d, d_r, dn, h);
    else if (BOX && g.type == RTRB_OBJ_BOX) ok = box_intersect(P.boxes[g.aux], o, d, h);
    else ok = plane_intersect(g, o, d, h, den);
    RTRB_COUNT(ctx, RTRB_CNT_EXACT);
    if (ok) {
      const double new_dis = norm(o - h.p);
      if (new_dis < best) { best = new_dis; best_i = i; keep_hit<BOX>(bh, h); }
    }
  }
  return best_i;
}

// The out-of-line fallbacks get TEMPORARIES for everything they take by reference: a thread's own hit record and
// counter block must never have their address taken, or they live in local memory for the whole kernel (ncu:
// 36 local loads/stores per thread on the config 2 kernel before this) instead of registers.
template <class Pol, bool BOX>
__device__ __forceinline__ int closest_hit_scan_call(const FrameParams& P, d3 o, d3 d, HitRec& bh, ThreadCtx& ctx) {
  HitRec h;
  h.p = mk(0, 0, 0); h.dir_in = false; h.face = 0;
  ThreadCtx t;
  init_ctx(t, ctx.detail);
  const int i = closest_hit_scan<Pol, BOX>(P, o, d, h, t);
  if (i >= 0) keep_hit<BOX>(bh, h);
  merge_ctx(ctx, t);
  return i;
}
template <class Pol, bool BOX>
__device__ __forceinline__ double lit_area_call(const FrameParams& P, d3 target, const DevLight& L, ThreadCtx& ctx) {
  ThreadCtx t;
  init_ctx(t, ctx.detail);
  const double a = lit_area<Pol, BOX>(P, target, L, t);
  merge_ctx(ctx, t);
  return a;
}

// ---- sphere BVH traversal (filter only; see rtrb_bvh.h for why it cannot change a result) ----------
struct BvhRay {
  float ox, oy, oz, ix, iy, iz, E;
};
__device__ __forceinline__ BvhRay make_bvh_ray(const CullRay& r) {
  BvhRay b;
  b.ox = r.ox; b.oy = r.oy; b.oz = r.oz;
  b.ix = rcp_approx(r.dx); b.iy = rcp_approx(r.dy); b.iz = rcp_approx(r.dz);
  b.E = r.E;
  return b;
}
// Slab test of the segment t in [tmin, tmax] against the box fattened by E on every side.
__device__ __forceinline__ bool box_hit(float lx, float ly, float lz, float hx, float hy, float hz, const BvhRay& b,
                                        float tmin, float tmax, float& tn_out) {
  const float t0x = (lx - b.E - b.ox) * b.ix, t1x = (hx + b.E - b.ox) * b.ix;
  const float t0y = (ly - b.E - b.oy) * b.iy, t1y = (hy + b.E - b.oy) * b.iy;
  const float t0z = (lz - b.E - b.oz) * b.iz, t1z = (hz + b.E - b.oz) * b.iz;
  const float tn = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fmaxf(fminf(t0z, t1z), tmin));
  const float tf = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fminf(fmaxf(t0z, t1z), tmax));
  tn_out = tn;
  return tn <= tf;
}

#define RTRB_BVH_STACK 32

// Visits every sphere whose (fattened) bounds the segment [tmin, tmax] of the ray touches, nearest
// subtree first.  `leaf(k)` is called with the sphere's slot in cull_sph[] and may shrink `tmax`.
// Returns false when the traversal stack would overflow (caller falls back to the exact scan).
template <typename Leaf>
__device__ __forceinline__ bool bvh_traverse(const FrameParams& P, const BvhRay& b, float tmin, float& tmax, Leaf leaf) {
  if (P.n_sph == 0) return true;
  int stk[RTRB_BVH_STACK];
  int sp = 0;
  int cur = 0;  // root
  while (true) {
    const float4* np = reinterpret_cast<const float4*>(P.bvh + cur);
    const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2);
    const int4 n3 = __ldg(reinterpret_cast<const int4*>(np + 3));
    float tn0, tn1;
    const bool h0 = box_hit(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, b, tmin, tmax, tn0);
    const bool h1 = box_hit(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, b, tmin, tmax, tn1);
    int first = n3.x, second = n3.y;
    bool hf = h0, hs = h1;
    if (h0 && h1 && tn1 < tn0) { first = n3.y; second = n3.x; }
    if (!h0) { first = n3.y; hf = h1; hs = false; }
    int next = -1;  // internal node to descend into
    if (hf) {
      if (first < 0) {
        const uint32_t v = (uint32_t)(~first);
        const uint32_t f0 = v & 0xFFFFFu, cnt = v >> 20;
        for (uint32_t j = 0; j < cnt; ++j) leaf(f0 + j);
      } else {
        next = first;
      }
    }
    if (hs) {
      if (second < 0) {
        const uint32_t v = (uint32_t)(~second);
        const uint32_t f0 = v & 0xFFFFFu, cnt = v >> 20;
        for (uint32_t j = 0; j < cnt; ++j) leaf(f0 + j);
      } else if (next < 0) {
        next = second;
      } else {
        if (sp >= RTRB_BVH_STACK) return false;
        stk[sp++] = second;
      }
    }
    if (next >= 0) { cur = next; continue; }
    if (sp == 0) break;
    cur = stk[--sp];
  }
  return true;
}

// The probe ray of the filtered lit_area: the CoverRay without lt_r / ltn (cover_ray_unit forms them when an exact sphere
// test first needs them), its CullRay, and `far`: hits farther than the light cannot cover, factor needs
// dot(hit - L, T - L) > 0.
__device__ __forceinline__ CoverRay make_cover_probe(const FrameParams& P, d3 target, const DevLight& L, CullRay& r,
                                                     float& far) {
  CoverRay c;
  c.target = target;
  c.lp = mk(L.px, L.py, L.pz);
  c.lt = c.lp - target;
  c.tl = target - c.lp;
  c.lt_r = 0; c.ltn = mk(0, 0, 0);
  r = make_cull_ray(P, target, c.lt);
  const float lx = (float)c.lt.x, ly = (float)c.lt.y, lz = (float)c.lt.z;
  far = sqrt_approx(fmaf(lz, lz, fmaf(ly, ly, lx * lx))) * 1.00001f + 2.0f * r.E;
  return c;
}

// World#intersect (world.rb:37-59) = FP32 filter (planes + sphere BVH) + exact test of the survivors.
template <class Pol, bool BOX>
__device__ __forceinline__ int closest_hit_bvh(const FrameParams& P, d3 o, d3 d, const CullRay& r, HitRec& bh,
                                                ThreadCtx& ctx) {
  // Pack8 keeps survivor slots in 16 bits: the BVH filter serves scenes of up to 65 536 bounded objects (larger ones
  // take the reference's own scan: correct, but brute force)
  if (P.n_sph > 0x10000 || P.n_pl > 8) return closest_hit_scan_call<Pol, BOX>(P, o, d, bh, ctx);
  // pass 1a: planes bound the search first (nothing at or beyond max_distance can win, world.rb:39)
  float best_hi = P.max_distance_f;
  for (int k = 0; k < P.n_pl; ++k) {
    float lo, hi;
    if (classify_plane(__ldg(&P.cull_pl[2 * k]), __ldg(&P.cull_pl[2 * k + 1]), r, lo, hi) == 2) best_hi = fminf(best_hi, hi);
  }
  // pass 1b: spheres through the BVH; certain hits keep shrinking the search interval
  Pack8 S;
  S.clear();
  {
    const BvhRay b = make_bvh_ray(r);
    float tmax = best_hi + r.E;
    const bool ok = bvh_traverse(P, b, -r.E, tmax, [&](uint32_t k) {
      const float4 s = __ldg(&P.cull_sph[k]);
      float lo, hi;
      const int kind = classify_sphere<BOX>(s, r, lo, hi);
      if (kind != 0 && lo <= best_hi) {
        S.push(k);
        if (kind == 2 && hi < best_hi) { best_hi = hi; tmax = hi + r.E; }
      }
    });
    if (!ok || S.overflow()) return closest_hit_scan_call<Pol, BOX>(P, o, d, bh, ctx);
  }
  // pass 2: exact FP64 evaluation of whatever can still win; (distance, index) lexicographic order
  // reproduces the strict `<` scan in world_objects order.
  double best = P.max_distance;
  int best_i = -1;
  bool have_dn = false;
  double d_r = 0;
  d3 dn = mk(0, 0, 0);
  for (int c = 0; c < S.n; ++c) {
    const uint32_t k = S.get(c);
    float lo, hi;
    const int kind = classify_sphere<BOX>(__ldg(&P.cull_sph[k]), r, lo, hi);
    if (kind == 0 || !(lo <= best_hi)) continue;
    if (!have_dn) { d_r = norm(d); dn = mk(d.x / d_r, d.y / d_r, d.z / d_r); have_dn = true; }
    const int i = P.sph_index[k];
    const DevGeom g = P.geom[i];
    HitRec h;
    RTRB_COUNT(ctx, RTRB_CNT_EXACT);
    if ((BOX && g.type == RTRB_OBJ_BOX) ? box_intersect(P.boxes[g.aux], o, d, h) : sphere_intersect<Pol>(g, o, d, d_r, dn, h)) {
      const double new_dis = norm(o - h.p);
      if (new_dis < best || (new_dis == best && best_i >= 0 && i < best_i)) { best = new_dis; best_i = i; keep_hit<BOX>(bh, h); }
    }
  }
  for (int k = 0; k < P.n_pl; ++k) {
    float lo, hi;
    const int kind = classify_plane(__ldg(&P.cull_pl[2 * k]), __ldg(&P.cull_pl[2 * k + 1]), r, lo, hi);
    if (kind == 0 || !(lo <= best_hi)) continue;
    const int i = P.pl_index[k];
    const DevGeom g = P.geom[i];
    HitRec h;
    double den;
    RTRB_COUNT(ctx, RTRB_CNT_EXACT);
    if (plane_intersect(g, o, d, h, den)) {
      const double new_dis = norm(o - h.p);
      if (new_dis < best || (new_dis == best && best_i >= 0 && i < best_i)) { best = new_dis; best_i = i; keep_hit<BOX>(bh, h); }
    }
  }
  return best_i;
}

// World#lit_area (world.rb:62-69) = filter + exact cover of the survivors, subtracted in index order.
// An object the probe ray certainly misses (or certainly meets beyond the light) has factor 0, hence
// cover exactly 0 (sphere.rb:29,45-53 multiply everything by factor; world_object.rb:43-47), and
// total - 0 == total, so skipping it leaves the running difference bit-identical.
template <class Pol, bool BOX>
__device__ __forceinline__ double lit_area_bvh(const FrameParams& P, d3 target, const DevLight& L, ThreadCtx& ctx) {
  CullRay r;
  float far;
  CoverRay c = make_cover_probe(P, target, L, r, far);
  if (P.n_sph > 0x10000 || P.n_pl > 0xFFFF) return lit_area_call<Pol, BOX>(P, target, L, ctx);
  Pack8 S, Q;
  S.clear();
  Q.clear();
  {
    const BvhRay b = make_bvh_ray(r);
    float tmax = far + r.E;
    const bool ok = bvh_traverse(P, b, -r.E, tmax, [&](uint32_t k) {
      const float4 s = __ldg(&P.cull_sph[k]);
      float lo, hi;
      const int kind = classify_sphere<BOX>(s, r, lo, hi);
      if (kind != 0 && !(lo > far)) S.push(k);
    });
    if (!ok) return lit_area_call<Pol, BOX>(P, target, L, ctx);
  }
  for (int k = 0; k < P.n_pl; ++k) {
    float lo, hi;
    const int kind = classify_plane(__ldg(&P.cull_pl[2 * k]), __ldg(&P.cull_pl[2 * k + 1]), r, lo, hi);
    if (kind != 0 && !(lo > far)) Q.push((uint32_t)k);
  }
  if (S.overflow() || Q.overflow()) return lit_area_call<Pol, BOX>(P, target, L, ctx);
  double total = 1;
  bool have_n = false;
  // visit the survivors in ascending world_objects index (selection over <= 16 entries)
  int last = -1;
  while (true) {
    int best_idx = 0x7fffffff, best_k = -1;
    for (int a = 0; a < S.n; ++a) {
      const int k = (int)S.get(a), i = P.sph_index[k];
      if (i > last && i < best_idx) { best_idx = i; best_k = k; }
    }
    for (int a = 0; a < Q.n; ++a) {
      const int i = P.pl_index[Q.get(a)];
      if (i > last && i < best_idx) { best_idx = i; best_k = -1; }
    }
    if (best_idx == 0x7fffffff) break;
    last = best_idx;
    if (best_k >= 0) {  // sphere: the full classification may still prove factor == 0
      float lo, hi;
      const int kind = classify_sphere<BOX>(__ldg(&P.cull_sph[best_k]), r, lo, hi);
      if (kind == 0 || lo > far) continue;
      if (!have_n) { cover_ray_unit(c); have_n = true; }
    }
    RTRB_COUNT(ctx, RTRB_CNT_EXACT);
    if (best_k >= 0) total -= cover_object_exact<Pol, BOX, 1>(P, P.geom[best_idx], c, L.radius, ctx);
    else total -= cover_object_exact<Pol, BOX, 2>(P, P.geom[best_idx], c, L.radius, ctx);
  }
  return fmax(total, 0.0);
}

// ---- SMALL SCENES: linear FP32 scan, no tree (cull_sph[] stays in world_objects order) -------------
// KT = "constant tables": the depth-1 kernels read the uniformly indexed per-ray tables (plane filter records,
// light apex tables, lights) from the kernel-parameter constant bank (FrameParams::k_*); measured -4 % on config 2.
// The ray-tree kernels (MAXS > 1) keep them in global memory: there the extra 2 KB of constants evict the
// camera table and the FP64 literals from the small constant cache, measured +3 % on configs 3/4.
template <bool KT> __device__ __forceinline__ float4 pl_rec(const FrameParams& P, int j) {
  if constexpr (KT) return P.k_cull_pl[j]; else return __ldg(&P.cull_pl[j]);
}
template <bool KT> __device__ __forceinline__ int pl_world_index(const FrameParams& P, int k) {
  if constexpr (KT) return P.k_pl_index[k]; else return P.pl_index[k];
}
// World#intersect (world.rb:37-59) = FP32 filter over every object + exact test of the survivors.
// Survivors of the linear filter are a 32-bit mask over cull_sph[] (n_sph <= RTRB_APEX_MAX = 32 here),
// bit k = sphere k in world_objects order; the hot loop is branch-free.
template <bool KT>
__device__ __forceinline__ uint32_t line_survivors_generic(const FrameParams& P, const CullRay& r) {
  uint32_t m = 0u;
#pragma unroll 4
  for (int k = 0; k < P.n_sph; ++k) {
    float4 s;
    if constexpr (KT) s = P.k_cull_sph[k]; else s = __ldg(&P.cull_sph[k]);
    m |= (sphere_line_misses(s, r) ? 0u : 1u) << k;
  }
  return m;
}
// Apex-table form: b = v.u, survive unless b*b < Kq (NaN survives).  Padding entries have Kq = +inf.
__device__ __forceinline__ uint32_t apex_test(const float4 t, const CullRay& r) {
  const float b = fmaf(t.z, r.dz, fmaf(t.y, r.dy, t.x * r.dx));
  return (b * b < t.w) ? 0u : 1u;
}
__device__ __forceinline__ uint32_t line_survivors_camera(const FrameParams& P, const CullRay& r) {
  // constant indices: the table is read straight from the constant bank, eight spheres per uniform branch
  uint32_t m = 0u;
#pragma unroll
  for (int blk = 0; blk < RTRB_APEX_MAX / 8; ++blk) {
    if (blk * 8 < P.n_sph) {
#pragma unroll
      for (int j = 0; j < 8; ++j) m |= apex_test(P.cam_tab[blk * 8 + j], r) << (blk * 8 + j);
    }
  }
  return m;
}
template <bool KT>
__device__ __forceinline__ uint32_t line_survivors_light(const FrameParams& P, const int light_index, const CullRay& r) {
  uint32_t m = 0u;
  if constexpr (!KT) {
    const float4* tab = P.light_tab + (size_t)light_index * P.n_sph;
#pragma unroll 4
    for (int k = 0; k < P.n_sph; ++k) m |= apex_test(__ldg(&tab[k]), r) << k;
  } else {
    // constant-bank table, eight spheres per uniform branch like the camera table
#pragma unroll
    for (int blk = 0; blk < RTRB_APEX_MAX / 8; ++blk) {
      if (blk * 8 < P.n_sph) {
#pragma unroll
        for (int j = 0; j < 8; ++j) m |= apex_test(P.k_light_tab[light_index][blk * 8 + j], r) << (blk * 8 + j);
      }
    }
  }
  return m;
}

// World#intersect (world.rb:37-59) = FP32 filter over every object + exact test of the survivors.
template <class Pol, bool BOX, bool KT>
__device__ __forceinline__ int closest_hit_linear(const FrameParams& P, d3 o, d3 d, const CullRay& r, HitRec& bh,
                                                ThreadCtx& ctx, const bool through_lens) {
  if (P.n_sph > RTRB_APEX_MAX || P.n_pl > RTRB_K_PLANES) return closest_hit_scan_call<Pol, BOX>(P, o, d, bh, ctx);
  const uint32_t mask = (through_lens && P.cam_tab_valid) ? line_survivors_camera(P, r) : line_survivors_generic<KT>(P, r);
  // pass 1 (only when something can be pruned): the smallest certain upper bound; nothing at or beyond
  // max_distance can win (world.rb:39)
  float best_hi = P.max_distance_f;
  // ray-tree kernels: the classification of the first two planes is kept for pass 2 (same ray, same record, 30
  // instructions each: configs 3/4 -1.2 %); the depth-1 kernel is faster recomputing it (registers)
  bool planes_cached = false;
  float plo0 = 0.0f, plo1 = 0.0f;
  int pkind0 = 1, pkind1 = 1;
  if (mask != 0u || P.n_pl > 1) {
    for (uint32_t m = mask; m != 0u; m &= m - 1u) {
      float lo, hi;
      if (classify_sphere<BOX>(__ldg(&P.cull_sph[__ffs(m) - 1]), r, lo, hi) == 2) best_hi = fminf(best_hi, hi);
    }
    for (int k = 0; k < P.n_pl; ++k) {
      float lo, hi;
      const int kind = classify_plane(pl_rec<KT>(P, 2 * k), pl_rec<KT>(P, 2 * k + 1), r, lo, hi);
      if (kind == 2) best_hi = fminf(best_hi, hi);
      if constexpr (!KT) { if (k == 0) { plo0 = lo; pkind0 = kind; } else if (k == 1) { plo1 = lo; pkind1 = kind; } }
    }
    planes_cached = !KT;
  }
  // pass 2: exact FP64 evaluation of whatever can still win; (distance, index) lexicographic order
  // reproduces the strict `<` scan in world_objects order.
  double best = P.max_distance;
  int best_i = -1;
  bool have_dn = false;
  double d_r = 0;
  d3 dn = mk(0, 0, 0);
  for (uint32_t m = mask; m != 0u; m &= m - 1u) {
    const int k = __ffs(m) - 1;
    float lo, hi;
    const int kind = classify_sphere<BOX>(__ldg(&P.cull_sph[k]), r, lo, hi);
    if (kind == 0 || !(lo <= best_hi)) continue;
    if (!have_dn) { d_r = norm(d); dn = mk(d.x / d_r, d.y / d_r, d.z / d_r); have_dn = true; }
    const int i = P.sph_index[k];
    const DevGeom g = P.geom[i];
    HitRec h;
    RTRB_COUNT(ctx, RTRB_CNT_EXACT);
    if ((BOX && g.type == RTRB_OBJ_BOX) ? box_intersect(P.boxes[g.aux], o, d, h) : sphere_intersect<Pol>(g, o, d, d_r, dn, h)) {
      const double new_dis = norm(o - h.p);
      if (new_dis < best || (new_dis == best && best_i >= 0 && i < best_i)) { best = new_dis; best_i = i; keep_hit<BOX>(bh, h); }
    }
  }
  for (int k = 0; k < P.n_pl; ++k) {
    float lo, hi;
    int kind;
    if (planes_cached && k == 0) { lo = plo0; kind = pkind0; }
    else if (planes_cached && k == 1) { lo = plo1; kind = pkind1; }
    else kind = classify_plane(pl_rec<KT>(P, 2 * k), pl_rec<KT>(P, 2 * k + 1), r, lo, hi);
    if (kind == 0 || !(lo <= best_hi)) continue;
    const int i = pl_world_index<KT>(P, k);
    const DevGeom g = P.geom[i];
    HitRec h;
    double den;
    RTRB_COUNT(ctx, RTRB_CNT_EXACT);
    if (plane_intersect(g, o, d, h, den)) {
      const double new_dis = norm(o - h.p);
      if (new_dis < best || (new_dis == best && best_i >= 0 && i < best_i)) { best = new_dis; best_i = i; keep_hit<BOX>(bh, h); }
    }
  }
  return best_i;
}

// World#lit_area (world.rb:62-69) = filter + exact cover of the survivors, subtracted in index order.
// An object the probe ray certainly misses (or certainly meets beyond the light) has factor 0, hence
// cover exactly 0 (sphere.rb:29,45-53 multiply everything by factor; world_object.rb:43-47), and
// total - 0 == total, so skipping it leaves the running difference bit-identical.
template <class Pol, bool BOX, bool KT>
__device__ __forceinline__ double lit_area_linear(const FrameParams& P, d3 target, const DevLight& L, const int light_index,
                                                  ThreadCtx& ctx) {
  CullRay r;
  float far;
  CoverRay c = make_cover_probe(P, target, L, r, far);
  if (P.n_sph > RTRB_APEX_MAX || P.n_pl > RTRB_K_PLANES) return lit_area_call<Pol, BOX>(P, target, L, ctx);
  // the probe ray's line passes through the light: apex table of this light when there is one
  uint32_t sm = (P.k_has_light_tab != 0) ? line_survivors_light<KT>(P, light_index, r) : line_survivors_generic<KT>(P, r);
  uint32_t qm = 0u;
  for (int k = 0; k < P.n_pl; ++k) {
    float lo, hi;
    const int kind = classify_plane(pl_rec<KT>(P, 2 * k), pl_rec<KT>(P, 2 * k + 1), r, lo, hi);
    if (kind != 0 && !(lo > far)) qm |= 1u << k;
  }
  double total = 1;
  bool have_n = false;
  // merge the two survivor sets (each ascending in world_objects index) so covers subtract in order
  while (sm != 0u || qm != 0u) {
    const int ks = sm ? __ffs(sm) - 1 : -1, kq = qm ? __ffs(qm) - 1 : -1;
    const int is = ks >= 0 ? P.sph_index[ks] : 0x7fffffff;
    const int iq = kq >= 0 ? pl_world_index<KT>(P, kq) : 0x7fffffff;
    if (is < iq) {
      sm &= sm - 1u;
      float lo, hi;
      const int kind = classify_sphere<BOX>(__ldg(&P.cull_sph[ks]), r, lo, hi);
      if (kind == 0 || lo > far) continue;
      if (!have_n) { cover_ray_unit(c); have_n = true; }
      RTRB_COUNT(ctx, RTRB_CNT_EXACT);
      total -= cover_object_exact<Pol, BOX, 1>(P, P.geom[is], c, L.radius, ctx);
    } else {
      qm &= qm - 1u;
      RTRB_COUNT(ctx, RTRB_CNT_EXACT);
      total -= cover_object_exact<Pol, BOX, 2>(P, P.geom[iq], c, L.radius, ctx);
    }
  }
  return fmax(total, 0.0);
}

// Only UNIFORMLY indexed tables are read from the constant bank (every lane the same element: the apex-table
// and plane loops, the lights).  Survivor lookups (cull_sph[k], sph_index[k] with a per-lane k) stay in global
// memory: divergent constant loads serialise, measured +3.7 % on the depth-8 kernels.
// Lights: constant-bank copies in the KT kernels (<= RTRB_K_LIGHTS lights), global memory otherwise.
template <bool KT>
__device__ __forceinline__ const DevLight& light_at(const FrameParams& P, int l) {
  if constexpr (KT) return P.k_lights[l]; else return P.lights[l];
}
template <bool KT>
__device__ __forceinline__ const DevLightF& light_f_at(const FrameParams& P, int l) {
  if constexpr (KT) return P.k_lights_f[l]; else return P.lights_f[l];
}

// Compile-time choice: kernels are instantiated once per filter so each stays compact (the linear
// scan wins below ~32 spheres: measured 5.56 vs 6.05 ms on config 3; the BVH wins 5x on config 5).
template <class Pol, bool BVH, bool BOX, bool KT>
__device__ __forceinline__ int closest_hit_fast(const FrameParams& P, d3 o, d3 d, const CullRay& r, HitRec& bh,
                                                ThreadCtx& ctx, const bool through_lens) {
  if constexpr (BVH) return closest_hit_bvh<Pol, BOX>(P, o, d, r, bh, ctx);
  else return closest_hit_linear<Pol, BOX, KT>(P, o, d, r, bh, ctx, through_lens);
}
template <class Pol, bool BVH, bool BOX, bool KT>
__device__ __forceinline__ double lit_area_fast(const FrameParams& P, d3 target, const DevLight& L, const int light_index,
                                                ThreadCtx& ctx) {
  if constexpr (BVH) return lit_area_bvh<Pol, BOX>(P, target, L, ctx);
  else return lit_area_linear<Pol, BOX, KT>(P, target, L, light_index, ctx);
}

// The reference's own expression of the highlight match (world.rb:86-93), register-only interface.  Only the depth-1
// builds call it (Policy::outline_libm), so its acos is their out-of-line copy.
static __device__ __noinline__ bool highlight_match_exact(double lx, double ly, double lz, double threshold, double ox, double oy,
                                                         double oz, double dx, double dy, double dz, uint32_t* status) {
  ThreadCtx t;
  t.status = 0; t.detail = false;
  const d3 a = mk(lx, ly, lz) - mk(ox, oy, oz);
  const double ct = vcos(mk(dx, dy, dz), a, t);
  const double ang = rb_acos<Generic::at<1>>(ct, t);
  *status = t.status;
  return ang < threshold;
}

// World#high_lights match for one light (world.rb:86-93): acos(|cos|) < threshold, filtered in FP32 on
// cos^2 against cos^2(threshold); the exact FP64 expression decides only inside the error band.
template <class Pol>
__device__ __forceinline__ bool highlight_match_fast(const DevLight& L, const DevLightF& F, d3 o, d3 d,
                                                     const CullRay& r, ThreadCtx& ctx) {
  const float eps = 5.9604645e-8f;
  const float ax = F.px - r.ox, ay = F.py - r.oy, az = F.pz - r.oz;
  const float ret = fmaf(az, r.dz, fmaf(ay, r.dy, ax * r.dx));
  const float a2 = fmaf(az, az, fmaf(ay, ay, ax * ax));
  const float ea = 8.0f * eps * (F.pmax + r.mo);
  const float c2 = ret * ret * rcp_approx(a2);
  const float rho = 8.0f * (ea * rsqrt_approx(a2) + 8.0f * eps);  // absolute error bound on |cos| (<= 1)
  const float tol = fmaf(rho, rho, 2.0f * rho);                    // ... hence on cos^2
  if (F.mode == 1 && rho < 0.25f) {
    if (c2 - tol > F.cos2_thr) return true;
    if (c2 + tol < F.cos2_thr) return false;
  }
  // exact (also reached for thresholds outside (0, 90 degrees), NaNs, and rays starting at the light)
  if constexpr (Pol::outline_libm) {
    // depth-1 builds: rare there, and out of line so that its two divisions, square root and acos do not sit between
    // the hot blocks (config 2: -1 %; the ray-tree kernels lose 1 % with it and keep the inline form)
    uint32_t st = 0u;
    const bool hit = highlight_match_exact(L.px, L.py, L.pz, L.hl_threshold, o.x, o.y, o.z, d.x, d.y, d.z, &st);
    ctx.status |= st;
    return hit;
  } else {
    d3 a = mk(L.px, L.py, L.pz) - o;
    double ct = vcos(d, a, ctx);
    double ang = rb_acos<Pol>(ct, ctx);
    return ang < L.hl_threshold;
  }
}

// `attenuation.r < 0.0001` (ray_tracer.rb:52) without the square root outside a narrow band.
__device__ __forceinline__ bool attenuation_dead(d3 att) {
  const double s2 = sumsq(att);
  if (s2 > 1.0001e-8) return false;
  if (s2 < 0.9999e-8) return true;
  return sqrt(s2) < 0.0001;
}

// rt_map (ray_tracer.rb:50-164) for ONE popped work item, FAST64 evaluation, in two phases so that the lockstep item
// loop (rtrb_trace.cuh) can put a block barrier between them:
//   phase A  the cut at :52, World#high_lights, World#intersect  -> index of the hit object, or -1 when the item ends
//            here (dead, terminated by a highlight, or a miss);
//   phase B  intersect_parameters, the children (pushed onto `stack`), World#local_lights and local_lighting.
// Emitted colours are added to `sum` in emission order.
template <class Pol, int MAXS, bool BVH, bool BOX>
__device__ __forceinline__ int item_phase_a(const FrameParams& P, const StackItem& it, d3& sum, ThreadCtx& ctx, bool is_first,
                                            int* primary_hit, HitRec& bh) {
  constexpr bool KT = !BVH && MAXS == 1;  // constant-bank tables: depth-1 linear-filter kernels only (see pl_rec)
  const d3 o = mk(it.ox, it.oy, it.oz), d = mk(it.dx, it.dy, it.dz), att = mk(it.ax, it.ay, it.az);
  if (it.depth <= 0 || attenuation_dead(att)) return -1;  // rt_map :52
  ctx.rays++;

  const CullRay r = make_cull_ray(P, o, d);

  // ---- World#high_lights ----
  {
    unsigned long long hl_mask = 0ull;
    int hl_n = 0;
    for (int l = 0; l < Pol::n_lights(P); ++l)
      if (highlight_match_fast<Pol>(light_at<KT>(P, l), light_f_at<KT>(P, l), o, d, r, ctx)) { hl_mask |= 1ull << l; hl_n++; }
    if (hl_n > 0) {
      for (int l = 0; l < Pol::n_lights(P); ++l) {
        if (!((hl_mask >> l) & 1ull)) continue;
        d3 c = att * ld3(light_at<KT>(P, l).color_hl);
        if (hl_n != 1) c = c / (double)hl_n;  // x / 1.0 == x
        emit(sum, c, ctx);
      }
      RTRB_COUNT(ctx, RTRB_CNT_HIGHLIGHT);
      if (is_first) *primary_hit = -2;
      return -1;
    }
  }

  // ---- World#intersect ----
  bh.p = mk(0, 0, 0); bh.dir_in = false;
  if constexpr (BOX) bh.face = 0;
  const int best_i = closest_hit_fast<Pol, BVH, BOX, KT>(P, o, d, r, bh, ctx, is_first);
  if (best_i < 0) return -1;
  if (is_first) *primary_hit = best_i;
  RTRB_COUNT(ctx, RTRB_CNT_HITS);
  return best_i;
}

// trace_depth <= 1, near normal incidence: the direction math of the children that are born dead (world_object.rb:121-137)
// is evaluated only for the conditions it could raise on.  Rare; out of line with a register-only interface.
static __device__ __noinline__ uint32_t born_dead_children_status(double dx, double dy, double dz, double nx, double ny, double nz,
                                                                 double nnx, double nny, double nnz, double rate, bool can_refract) {
  ThreadCtx t;
  t.status = 0; t.detail = false;
  const d3 d = mk(dx, dy, dz), n = mk(nx, ny, nz), nn = mk(nnx, nny, nnz);
  const double d_r = norm(d);
  const double cos_theta = vcos(d, -n, t);
  const d3 refl_dir = normalize(nn * (2 * cos_theta * d_r) + d, t);
  if (can_refract) {
    const double sin_i = rb_sqrt(1 - cos_theta * cos_theta, t);
    const double sin_r = sin_i / rate;
    if (!(sin_r >= 1)) {
      if (sin_r < -1 || sin_r > 1) t.status |= RTRB_ST_MATH_DOMAIN;
      (void)normalize(refl_dir + d, t);
    }
  }
  return t.status;
}

template <class Pol, int MAXS, bool BVH, bool BOX>
__device__ __forceinline__ void item_phase_b(const FrameParams& P, const StackItem& it, const int best_i, const HitRec& bh,
                                             StackItem* stack, int& sp, d3& sum, ThreadCtx& ctx, uint32_t pixel,
                                             uint32_t sample) {
  const uint32_t K = (uint32_t)(Pol::mc(P) + 2);
  constexpr bool KT = !BVH && MAXS == 1;
  {
    const d3 o = mk(it.ox, it.oy, it.oz), d = mk(it.dx, it.dy, it.dz), att = mk(it.ax, it.ay, it.az);
    (void)o;
    const DevGeom g = P.geom[best_i];
    const DevMat& M = P.mat[best_i];
    const auto [n, delta, rate, can_refract] = intersect_parameters<BOX>(P, g, M, bh, d);
    d3 nn;
    if ((BOX ? g.type == RTRB_OBJ_PLANE : g.type != RTRB_OBJ_SPHERE) && M.plane_nn_valid) {
      // n is +-front: its normalisation is a per-plane constant baked on the host (-(x / r) == (-x) / r)
      const d3 pn = ld3(M.plane_nn);
      nn = (n.x == g.nx && n.y == g.ny && n.z == g.nz) ? pn : -pn;
    } else {
      nn = normalize(n, ctx);
    }

    // ---- children (ray_tracer.rb:87-121), computed only if they can survive the cut at :52.
    // A child with trace_depth - 1 <= 0, or whose attenuation norm is certainly < 1e-4, is popped and
    // dropped by the reference without any observable effect; skipping its direction math changes
    // nothing except in the one case where that math would RAISE (normalize of an exactly zero
    // reflection + d, world_object.rb:136, or a zero normal) — caught by a cheap necessary condition.
    const d3 a_refl = att * ld3(M.refl), a_refr = att * ld3(M.refr);
    const bool depth_ok = it.depth - 1 > 0;
    const bool refl_alive = depth_ok && !(sumsq(a_refl) < 0.99e-8);
    const bool refr_alive = depth_ok && !(sumsq(a_refr) < 0.99e-8);
    const double dn_dot = dot(d, n);
    const bool near_normal = !(dn_dot * dn_dot < (1.0 - 1e-9) * (sumsq(d) * sumsq(n)));  // possible raise site
    if constexpr (MAXS == 1) {
      // trace_depth <= 1: every child is born with depth 0 and dropped at ray_tracer.rb:52; only the
      // raise sites of their direction math can be observed, and only near normal incidence
      if (near_normal) ctx.status |= born_dead_children_status(d.x, d.y, d.z, n.x, n.y, n.z, nn.x, nn.y, nn.z, rate, can_refract);
    } else if (refl_alive || refr_alive || near_normal) {
      if (sp + 2 > MAXS) { ctx.status |= RTRB_ST_STACK_OVERFLOW; return; }
      const double d_r = norm(d);
      const double cos_theta = vcos(d, -n, ctx);  // == vcos(d, n): both square the dot product
      const d3 refl_dir = normalize(nn * (2 * cos_theta * d_r) + d, ctx);
      if (refl_alive || near_normal) {
        set_item(stack[sp++], bh.p + delta, refl_dir, a_refl, it.depth - 1, it.path * K + 0u);
      }
      if (can_refract && (refr_alive || near_normal)) {
        const double sin_i = rb_sqrt(1 - cos_theta * cos_theta, ctx);
        const double sin_r = sin_i / rate;
        if (!(sin_r >= 1)) {
          if (sin_r < -1 || sin_r > 1) ctx.status |= RTRB_ST_MATH_DOMAIN;
          const double rr = m_asin<Pol>(sin_r);
          const d3 refr_dir = nn * (-m_cos<Pol>(rr)) + normalize(refl_dir + d, ctx) * sin_r;
          const d3 refr_org = bh.p - nn * RTRB_EPSILON;
          RTRB_COUNT(ctx, RTRB_CNT_REFR);
          set_item(stack[sp++], refr_org, refr_dir, a_refr, it.depth - 1, it.path * K + 1u);
        }
      }
    }

    // ---- World#local_lights + WorldObject#local_lighting ----
    const d3 shade_from = bh.p + delta;
    d3 contrib = mk(0.0, 0.0, 0.0);
    int n_lit = 0;
    for (int l = 0; l < Pol::n_lights(P); ++l) {
      const DevLight& L = light_at<KT>(P, l);
      ctx.shadow++;
      const double area = lit_area_fast<Pol, BVH, BOX, KT>(P, shade_from, L, l, ctx);
      if (area > 0) {
        double w = rb_pow<Pol>(area, Pol::shadow_exponent(P));
        if (Pol::n_lights(P) != 1) w = w / (double)Pol::n_lights(P);  // x / 1.0 == x
        d3 lc = ld3(L.color) * w;
        d3 lv = normalize(mk(L.px, L.py, L.pz) - bh.p, ctx);
        double ldn = dot(lv, nn);
        if (ldn > 1) ldn = 1.0; else if (ldn < 0) ldn = 0.0;
        contrib = contrib + lc * ldn;
        n_lit++;
      }
    }
    if (n_lit == 0) {
      if (MAXS == 1 && Pol::mc(P) > 0 && ctx.detail) ctx.c[RTRB_CNT_MC] += Pol::mc(P);  // spawned, born dead
      if (MAXS > 1 && Pol::mc(P) > 0) {
        if (sp + Pol::mc(P) > MAXS) { ctx.status |= RTRB_ST_STACK_OVERFLOW; return; }
        const d3 att_pt = ld3(M.diffuse) / (double)Pol::mc(P);
        const d3 a2 = att * att_pt;
        const bool mc_alive = depth_ok && !(sumsq(a2) < 0.99e-8);
        const d3 vv = a_vertical_vector(n, ctx);
        if (mc_alive || sumsq(vv) == 0) {
          const d3 leftv = normalize(vv, ctx);
          const d3 upv = cross(nn, leftv);
          for (int m = 0; m < Pol::mc(P); ++m) {
            uint32_t child = it.path * K + (uint32_t)(2 + m);
            uint32_t c0 = pixel, c1 = sample, c2 = child, c3 = 1u;
            philox4x32_10(P.key0, P.key1, c0, c1, c2, c3);
            double theta = res53(c0, c1) * RTRB_PI / 2, phi = res53(c2, c3) * RTRB_PI * 2;
            d3 dir = nn * m_sin<Pol>(theta) + (leftv * m_cos<Pol>(phi) + upv * m_sin<Pol>(phi)) * m_cos<Pol>(theta);
            set_item(stack[sp++], shade_from, dir, a2, it.depth - 1, child);
          }
        }
        if (ctx.detail) ctx.c[RTRB_CNT_MC] += Pol::mc(P);
      }
    } else {
      RTRB_COUNT(ctx, RTRB_CNT_LOCAL);
      if (ctx.detail) ctx.c[RTRB_CNT_LIT] += n_lit;
      if (n_lit != 1) contrib = contrib / (double)n_lit;  // x / 1.0 == x
      d3 filter = mk(1.0, 1.0, 1.0);
      if (Pol::textured(M)) {
        double u, v;
        object_uv(g, M, bh.p, u, v, ctx);
        RTRB_COUNT(ctx, RTRB_CNT_TEXEL);
        filter = texture_color<Pol>(M, u, v, ctx) * filter;
      }
      d3 local = ((contrib * ld3(M.diffuse)) * filter) + ld3(M.ambient);
      emit(sum, att * local, ctx);
    }
  }
}

template <class Pol, int MAXS, bool BVH, bool BOX>
__device__ __forceinline__ void process_item_fast(const FrameParams& P, const StackItem& it, StackItem* stack, int& sp,
                                                  d3& sum, ThreadCtx& ctx, uint32_t pixel, uint32_t sample,
                                                  bool is_first, int* primary_hit) {
  HitRec bh;
  const int best_i = item_phase_a<Pol, MAXS, BVH, BOX>(P, it, sum, ctx, is_first, primary_hit, bh);
  if (best_i >= 0) item_phase_b<Pol, MAXS, BVH, BOX>(P, it, best_i, bh, stack, sp, sum, ctx, pixel, sample);
}

// RayTracer#trace_sync for one sample, free-running: the item loop of the depth-1, extra-sample and ray-query kernels
// (the ray-tree frame kernels run trace_sample_fast_lockstep).
template <class Pol, int MAXS, bool BVH, bool BOX>
__device__ __forceinline__ d3 trace_sample_fast(const FrameParams& P, d3 ro, d3 rd, uint32_t pixel, uint32_t sample,
                                                ThreadCtx& ctx, int* primary_hit) {
  StackItem stack[MAXS > 1 ? MAXS : 1];
  // the root item starts in registers (no round trip through the local-memory stack)
  StackItem it;
  set_item(it, ro, rd, mk(1.0, 1.0, 1.0), P.trace_depth, 1u);
  int sp = 0;
  d3 sum = mk(0.0, 0.0, 0.0);
  bool first = true;
  *primary_hit = -1;
  ctx.max_stack = max(ctx.max_stack, 1u);
  while (true) {
    process_item_fast<Pol, MAXS, BVH, BOX>(P, it, stack, sp, sum, ctx, pixel, sample, first, primary_hit);
    first = false;
    if (MAXS == 1 || sp == 0) break;
    if ((uint32_t)sp > ctx.max_stack) ctx.max_stack = (uint32_t)sp;
    it = stack[--sp];
  }
  return sum;
}

// ---- ray-tree kernels (trace_depth > 1): lockstep item loop + render_at finished inside the CTA ----------------
//
// One thread per (pixel, sample), 512-thread CTAs.  LOCKSTEP: every thread of the CTA takes part in one block barrier
// per work item, so the CTA's warps execute the same phase of rt_map at the same time and share what the instruction
// caches hold (these kernels are ~150 KB of SASS; free-running, `no_instruction` was the top stall at 3.3 - 13.5
// cycles per issued instruction; profiles/README.md has the measurements, including the persistent warp-refill
// variant that was tried in round 2 and rejected: mixing tree depths inside a CTA makes every round as slow as its
// slowest item kind, config 3 3.5 -> 5.0 ms).
//
// IN-CTA RESOLVE: when the CTA holds every sample of its pixels (pre_sample_times divides the CTA size), the sample
// colours go to shared memory after the loop and one thread per pixel finishes render_at (camera.rb:79-98): ordered
// mean, variance of the signed maximum, adaptive decision, quantisation.  No per-sample FP64 buffer crosses HBM
// (24 B per sample: 12.7 GB for one 4K / 64 spp frame) and no resolve kernel runs.  RTRB_RESOLVE_IN_CTA selects it;
// other sample counts (3, 10, ...) write the sample buffer for resolve_kernel.
// PASS: a progressive frame's pass, whose launch holds pass_end - pass_begin samples of each pixel.
template <class Pol, int MAXS, bool BVH, bool BOX, bool PASS = false>
__device__ __forceinline__ d3 trace_sample_fast_lockstep(const FrameParams& P, d3 ro, d3 rd, uint32_t pixel, uint32_t sample,
                                                         ThreadCtx& ctx, int* primary_hit, bool active) {
  StackItem stack[MAXS > 1 ? MAXS : 1];
  StackItem it;
  set_item(it, ro, rd, mk(1.0, 1.0, 1.0), P.trace_depth, 1u);
  int sp = 0;
  d3 sum = mk(0.0, 0.0, 0.0);
  bool first = true, have = active;
  *primary_hit = -1;
  if (active) ctx.max_stack = max(ctx.max_stack, 1u);
  const bool mid_barrier = BVH && (PASS ? P.pass_end - P.pass_begin : P.pre) < 32;
  while (__syncthreads_or(have ? 1 : 0)) {
    HitRec bh;
    int best_i = -1;
    if (have) best_i = item_phase_a<Pol, MAXS, BVH, BOX>(P, it, sum, ctx, first, primary_hit, bh);
    // phase boundary: with the BVH filter the whole CTA also moves from intersection to shading together when a warp
    // holds several pixels (config 5 at 4 spp: 3.90 -> 3.53 ms); with a whole warp on one pixel (>= 32 spp) the warps are
    // even enough without it (config 5 at 64 spp: 956 -> 944 ms without), and with the linear filter the second
    // barrier costs more than it saves (config 3: +3 %)
    if constexpr (BVH) { if (mid_barrier) __syncthreads(); }
    if (have) {
      if (best_i >= 0) item_phase_b<Pol, MAXS, BVH, BOX>(P, it, best_i, bh, stack, sp, sum, ctx, pixel, sample);
      first = false;
      if (sp == 0) have = false;
      else {
        if ((uint32_t)sp > ctx.max_stack) ctx.max_stack = (uint32_t)sp;
        it = stack[--sp];
      }
    }
  }
  return sum;
}

// Kernel body: the first loop of render_at (camera.rb:73-78) for the CTA's samples, then (RTRB_RESOLVE_IN_CTA) its tail.
// PASS: a progressive frame's pass, samples j in [pass_begin, pass_end) into the sample buffer at (slot * pre + j),
// as trace_pre_body; never resolves in the CTA.
template <class Pol, int MAXS, bool BVH, bool DETAIL, bool PASS = false>
__device__ __forceinline__ void trace_pre_tree_body(const FrameParams& P) {
  extern __shared__ double rtrb_cta_samples[];  // [blockDim.x][3] when RTRB_RESOLVE_IN_CTA
  const uint32_t S = PASS ? (uint32_t)(P.pass_end - P.pass_begin) : (uint32_t)P.pre;
  const unsigned long long w = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long total = (unsigned long long)P.n_tiles * RTRB_SUPER_PIXELS * S;
  ThreadCtx ctx;
  init_ctx(ctx, DETAIL);
  int x = 0, y = 0;
  bool active = false;
  // every thread of the CTA enters the item loop (threads without a sample only take part in its barriers)
  uint32_t slot = 0, j = 0, pixel = 0;
  d3 ro = mk(0, 0, 0), rd = mk(1, 0, 0);
  if (w < total) {
    decode_work(w, S, slot, j);
    if constexpr (PASS) j += (uint32_t)P.pass_begin;
    active = decode_pixel(P, slot, x, y);
    if (active) {
      pixel = (uint32_t)y * (uint32_t)P.width + (uint32_t)x;
      camera_ray<Pol>(P, x, y, pixel, j, ro, rd);
    }
  }
  int ph = -1;
  const d3 col = trace_sample_fast_lockstep<Pol, MAXS, BVH, DETAIL, PASS>(P, ro, rd, pixel, j, ctx, &ph, active);
  if (active) {
    RTRB_COUNT(ctx, RTRB_CNT_SAMPLES);
    if (j == 0 && P.hit) P.hit[(size_t)y * P.width + x] = ph;
  }
  if constexpr (PASS) {
    if (active) {
      double* out = P.samples + ((unsigned long long)slot * (uint32_t)P.pre + j) * 3ull;
      out[0] = col.x; out[1] = col.y; out[2] = col.z;
    }
  } else if (P.fuse_resolve == RTRB_RESOLVE_IN_CTA) {
    // S divides blockDim.x, so the S samples of a pixel are S consecutive threads of this CTA
    double* mine = rtrb_cta_samples + (size_t)threadIdx.x * 3u;
    mine[0] = col.x; mine[1] = col.y; mine[2] = col.z;
    __syncthreads();
    const bool resolver = active && j == 0u;
    double ax = 0, ay = 0, az = 0, variance = 0;
    if (S < 8u) {
      if (resolver) pre_mean_of(mine, (int)S, ax, ay, az, variance);
    } else {
      // Many samples per pixel: the ORDER of both sums is the reference's (sample 0 first, camera.rb:79-86), but the
      // three channels of the mean run on three threads and every thread forms its own squared deviation, so the
      // CTA's tail is two serial chains of S additions instead of one of 9 S operations.
      double* first = mine - (size_t)j * 3u;            // sample 0 of this thread's pixel
      double m = 0.0;
      if (active && j < 3u) {
        for (uint32_t k = 0; k < S; ++k) m += first[k * 3u + j];
        m = m / (double)S;
      }
      __syncthreads();                                  // every thread has read what the next store overwrites
      const double cx = mine[0], cy = mine[1], cz = mine[2];
      __syncthreads();
      if (active && j < 3u) first[j] = m;               // the pixel's mean replaces sample 0's colour
      __syncthreads();
      ax = first[0]; ay = first[1]; az = first[2];
      const double dx = cx - ax, dy = cy - ay, dz = cz - az;
      const double mm = fmax(dx, fmax(dy, dz));         // (sample - mean).to_a.max, signed
      __syncthreads();
      mine[0] = mm * mm;
      __syncthreads();
      if (resolver) {
        for (uint32_t k = 0; k < S; ++k) variance += first[k * 3u];
        variance /= (double)S;
      }
    }
    // every thread of the CTA gets here (the barriers above), so every warp is whole
    const bool queued = queue_adaptive(P, resolver && variance >= P.variant_threshold, slot, ax, ay, az);
    if (resolver && !queued) write_pixel(P, x, y, ax, ay, az);
  } else if (active) {
    double* out = P.samples + w * 3ull;
    out[0] = col.x; out[1] = col.y; out[2] = col.z;
  }
  flush_ctx(P, ctx, x, y, active);
}

}  // namespace rtrb
