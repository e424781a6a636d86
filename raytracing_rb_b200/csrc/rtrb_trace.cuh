// rtrb_trace.cuh — the ray-tree engine of raytracing_rb as device code (sm_100a).
//
// One thread owns one pixel-sample: it builds the thin-lens primary ray (camera.rb:129-151), then
// runs RayTracer#trace_sync (ray_tracer.rb:16-46) with the work stack as an explicit per-thread
// LIFO array in local memory, popping the LAST pushed item exactly like `@queue.pop` (:32), and
// accumulates the colours in emission order (rt_reduce, :292-298).
//
// STRICT arithmetic contract: this translation unit is compiled with -fmad=false and every
// expression keeps the reference's association order, every division and square root the
// reference performs is performed, so FP64 results equal the CPU oracle's bit for bit except where
// libm's transcendental functions (sin cos acos asin pow) round differently from CUDA's.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/rtrb_b200.h"
#include "rtrb_types.h"

namespace rtrb {

#define RTRB_EPSILON 1e-5                 // src/libs/algebra.rb:2
#define RTRB_PI 3.141592653589793         // Math::PI

struct d3 { double x, y, z; };

// ---- build policies ------------------------------------------------------------------------------------------------
// What a kernel build knows at compile time.  The policy is the first template argument of every function whose code
// depends on it, from the kernel body down.  STRICT is one build; the FAST64 kernels exist in several builds that differ
// only in what is known about the scene (checked when it is baked, FrameParams::scene_class) or the frame, so that code
// the class cannot reach is not compiled in.  Same source, same arithmetic, bit-identical results; what changes is code
// size, register pressure and - these kernels being bound by instruction fetch and dependent issue - speed:
//   fast          the exact-preserving shortcuts of FAST64 inside the shared STRICT functions (sphere_intersect).
//   one_light     exactly one light and soft_shadow_exponent == 2 (every BASELINE.json config): no loops over
//                 lights, no division by the number of matching / lit lights (x / 1.0 == x), no pow.
//                 Ray-tree kernels: configs 3 / 4 / 5 -8.6 / -9.1 / -4.3 %.
//   no_mc         monte_carlo_diffusion_times == 0: no Monte-Carlo ray code (configs 3 / 5 a further -1.6 / -4.9 %).
//   lean          one_light plus: the light's radius is exactly 0 (hard shadows) and no object is textured: no
//                 texture lookup, no penumbra branch in Sphere#cover_area.  Depth-1 kernels (config 2): -13 %.
//   outline_libm  the FAST64 depth-1 builds (at<1>).  libm's FP64 transcendentals are 100-500 SASS instructions each.
//                 In a depth-1 frame they (acos / sin of the penumbra and highlight fallbacks, pow, fmod) are cold, yet
//                 inlined they put ~1 700 instructions between the hot blocks of a kernel whose top stall after `wait`
//                 is `no_instruction`; as one out-of-line copy each (and the exact highlight test out of line) they sit
//                 behind the kernel (config 2: -2 %).  The ray-tree kernels, where these calls are warm, keep them
//                 inline: out of line measured +2 % .. +5 % there (round 1: config 3 4.38 -> 4.62 ms).
template <bool FAST, bool ONE_LIGHT, bool LEAN, bool NO_MC, bool OUTLINE_LIBM = false>
struct Policy {
  static_assert(!LEAN || ONE_LIGHT, "a lean scene is a one-light scene");
  static constexpr bool fast = FAST, one_light = ONE_LIGHT, lean = LEAN, no_mc = NO_MC, outline_libm = OUTLINE_LIBM;
  // CTAs per SM that the depth-1 kernel's __launch_bounds__ asks for (128 threads each).  Generic: 5 (96 registers;
  // config 2: 0.101 ms at 4 CTAs / 128 registers, 0.095 - 0.098 at 5 .. 8 CTAs / 96 .. 64 registers; 256 x 2: 0.103).
  // Lean (124 registers unconstrained): 8, from 0.086 / 0.080 / 0.078 / 0.076 / 0.078 / 0.088 ms on config 2 at
  // 4 / 5 / 7 / 8 / 10 / 12 CTAs per SM (124 / 96 / 72 / 64 / 48 / 40 registers).
  static constexpr int d1_min_blocks = LEAN ? 8 : 5;
  // this class's build for a work stack of MAXS items
  template <int MAXS>
  using at = Policy<FAST, ONE_LIGHT, LEAN, NO_MC, FAST && MAXS == 1>;

  // FrameParams / material fields, or the constant the class fixes
  __device__ static __forceinline__ int n_lights(const FrameParams& P) { return ONE_LIGHT ? 1 : P.n_lights; }
  __device__ static __forceinline__ double shadow_exponent(const FrameParams& P) { return ONE_LIGHT ? 2.0 : P.soft_shadow_exponent; }
  __device__ static __forceinline__ bool textured(const DevMat& M) { return LEAN ? false : M.tex != nullptr; }
  __device__ static __forceinline__ int mc(const FrameParams& P) { return NO_MC ? 0 : P.mc; }
};
using Strict = Policy<false, false, false, false>;
using Generic = Policy<true, false, false, false>;
using OneLight = Policy<true, true, false, false>;
using OneLightNoMc = Policy<true, true, false, true>;
using Lean = Policy<true, true, true, false>;

// libm wrappers: m_sin<Pol>(x) calls the one out-of-line copy cold::sin in the Policy::outline_libm builds and inlines
// libm's sin in all others.  Likewise for the other functions.
namespace cold {
static __device__ __noinline__ double sin(double x) { return ::sin(x); }
static __device__ __noinline__ double cos(double x) { return ::cos(x); }
static __device__ __noinline__ double asin(double x) { return ::asin(x); }
static __device__ __noinline__ double acos(double x) { return ::acos(x); }
static __device__ __noinline__ double pow(double x, double y) { return ::pow(x, y); }
static __device__ __noinline__ double fmod(double x, double y) { return ::fmod(x, y); }
}  // namespace cold
template <class Pol> __device__ __forceinline__ double m_sin(double x) {
  if constexpr (Pol::outline_libm) return cold::sin(x); else return ::sin(x);
}
template <class Pol> __device__ __forceinline__ double m_cos(double x) {
  if constexpr (Pol::outline_libm) return cold::cos(x); else return ::cos(x);
}
template <class Pol> __device__ __forceinline__ double m_asin(double x) {
  if constexpr (Pol::outline_libm) return cold::asin(x); else return ::asin(x);
}
template <class Pol> __device__ __forceinline__ double m_acos(double x) {
  if constexpr (Pol::outline_libm) return cold::acos(x); else return ::acos(x);
}
template <class Pol> __device__ __forceinline__ double m_pow(double x, double y) {
  if constexpr (Pol::outline_libm) return cold::pow(x, y); else return ::pow(x, y);
}
template <class Pol> __device__ __forceinline__ double m_fmod(double x, double y) {
  if constexpr (Pol::outline_libm) return cold::fmod(x, y); else return ::fmod(x, y);
}

__device__ __forceinline__ d3 mk(double x, double y, double z) { d3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ d3 ld3(const double* p) { return mk(p[0], p[1], p[2]); }
__device__ __forceinline__ d3 operator+(d3 a, d3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ d3 operator-(d3 a, d3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ d3 operator-(d3 a) { return mk(-a.x, -a.y, -a.z); }
__device__ __forceinline__ d3 operator*(d3 a, d3 b) { return mk(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ d3 operator*(d3 a, double s) { return mk(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ d3 operator/(d3 a, double s) { return mk(a.x / s, a.y / s, a.z / s); }
// Vec3_method_dot (fast_4d_matrix.c:98-108): ((a0*b0) + a1*b1) + a2*b2
__device__ __forceinline__ double dot(d3 a, d3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
// sum of squares as Vec3_c_create computes it (c:67)
__device__ __forceinline__ double sumsq(d3 a) { return (a.x * a.x + a.y * a.y) + a.z * a.z; }
__device__ __forceinline__ double norm(d3 a) { return sqrt(sumsq(a)); }
__device__ __forceinline__ d3 cross(d3 a, d3 b) {
  return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}

struct ThreadCtx {
  uint32_t status;
  // lean counters (always)
  uint32_t rays, shadow;
  // detailed counters (count_detail only)
  uint32_t c[RTRB_CNT_N];
  bool detail;
  uint32_t max_stack;
};

#define RTRB_COUNT(ctx, which) do { if ((ctx).detail) (ctx).c[which]++; } while (0)

// Vec3#normalize (c:286-293)
__device__ __forceinline__ d3 normalize(d3 a, ThreadCtx& ctx) {
  double r = norm(a);
  if (r == 0) ctx.status |= RTRB_ST_ZERO_VECTOR;
  return mk(a.x / r, a.y / r, a.z / r);
}
// Vec3#cos (c:109-129): |cos| clamped to <= 1
__device__ __forceinline__ double vcos(d3 a, d3 b, ThreadCtx& ctx) {
  double ret = dot(a, b);
  double r1 = sumsq(a), r2 = sumsq(b);
  if (r1 == 0 || r2 == 0) ctx.status |= RTRB_ST_ZERO_VECTOR;
  double v = sqrt(ret * ret / r1 / r2);
  if (v > 1) v = 1;
  return v;
}
__device__ __forceinline__ double rb_sqrt(double x, ThreadCtx& ctx) {
  if (x < 0) ctx.status |= RTRB_ST_MATH_DOMAIN;
  return sqrt(x);
}
template <class Pol>
__device__ __forceinline__ double rb_acos(double x, ThreadCtx& ctx) {
  if (x < -1 || x > 1) ctx.status |= RTRB_ST_MATH_DOMAIN;
  return m_acos<Pol>(x);
}
// Float ** exponent (world.rb:76).  pow(x, 2.0) is the correctly rounded x*x.
template <class Pol>
__device__ __forceinline__ double rb_pow(double x, double y) { return (y == 2.0) ? x * x : m_pow<Pol>(x, y); }

// ---- counter RNG: Philox4x32-10 keyed by (seed; pixel, sample, ray path, purpose) ---------------
__device__ __forceinline__ void philox4x32_10(uint32_t k0, uint32_t k1, uint32_t& c0, uint32_t& c1, uint32_t& c2,
                                              uint32_t& c3) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
}
__device__ __forceinline__ double res53(uint32_t a, uint32_t b) {
  a >>= 5; b >>= 6;
  return ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
}

// ---- object tests ------------------------------------------------------------------------------
struct HitRec {
  d3 p;        // intersection
  bool dir_in; // :in / :out
  uint8_t face;  // box only: Box#intersect's data[:index] (box.rb:89)
};

// Sphere#intersect (sphere.rb:60-85).  d_r = |d|, dn = d / d_r are ray invariants.
template <class Pol>
__device__ __forceinline__ bool sphere_intersect(const DevGeom& g, d3 o, d3 d, double d_r, d3 dn, HitRec& h) {
  d3 c = mk(g.px, g.py, g.pz);
  d3 oc = c - o;
  double t = dot(oc, d) / (d_r * d_r);  // r2 = r*r (c:280-284)
  d3 np = o + d * t;
  d3 ncv = np - c;
  double nd = norm(ncv);
  if (!(nd <= g.radius)) return false;  // unless inner?(nearest_point)
  double hh = sqrt(g.radius * g.radius - nd * nd);
  d3 vec = dn * hh;
  // from_inner = |O - C| <= R (|O - C| == |C - O| bit for bit)
  bool from_inner;
  if constexpr (Pol::fast) {
    // FAST64: sqrt is monotone and correctly rounded, so away from the surface the comparison of the squares decides
    // (1e-14 >> 2^-52 covers the roundings of R*R and of the sum); inside that band, and for NaNs, negative or
    // overflowing radii, the reference's own expression is evaluated.
    const double oc2 = sumsq(oc), rr2 = g.radius * g.radius;
    if (g.radius >= 0 && rr2 < 1e300 && oc2 < rr2 * (1.0 - 1e-14)) from_inner = true;
    else if (g.radius >= 0 && rr2 < 1e300 && oc2 > rr2 * (1.0 + 1e-14)) from_inner = false;
    else from_inner = sqrt(oc2) <= g.radius;
  } else {
    from_inner = norm(oc) <= g.radius;
  }
  h.dir_in = !from_inner;
  h.p = h.dir_in ? (np - vec) : (np + vec);
  if (!from_inner && t < 0) return false;
  return true;
}
// Plane#intersect (plane.rb:38-51)
__device__ __forceinline__ bool plane_intersect(const DevGeom& g, d3 o, d3 d, HitRec& h, double& den_out) {
  d3 n = mk(g.nx, g.ny, g.nz);
  double den = dot(n, d);
  den_out = den;
  if (den == 0) return false;
  double t = dot(mk(g.px, g.py, g.pz) - o, n) / den;
  h.p = o + d * t;
  if (t < 0) return false;
  h.dir_in = den < 0;
  return true;
}

// Box#intersect (box.rb:80-99): Plane#intersect on each of the six faces in order, kept when Plane#get_uv
// of the hit lies in [-0.5, 0.5]^2, nearest by |hit - origin| with a strict `<` (lowest face wins ties).
// Returns the winning face or -1.  Not inlined and register-only interface: boxes are rare, and the
// hot sphere/plane kernels must not pay registers or local memory for this loop.
static __device__ __noinline__ int box_nearest_face(const DevBox* bx, double ox, double oy, double oz, double dx,
                                                    double dy, double dz) {
  const d3 o = mk(ox, oy, oz), d = mk(dx, dy, dz);
  double nearest = CUDART_INF;
  int face = -1;
#pragma unroll 1
  for (int k = 0; k < 6; ++k) {
    const DevBoxFace& F = bx->f[k];
    const d3 n = mk(F.nx, F.ny, F.nz), pt = mk(F.px, F.py, F.pz);
    const double den = dot(n, d);
    if (den == 0) continue;                    // plane.rb:41
    const double t = dot(pt - o, n) / den;
    const d3 ip = o + d * t;
    if (t < 0) continue;                       // plane.rb:46
    const d3 rel = ip - pt;
    const double u = dot(rel, mk(F.lx, F.ly, F.lz)) / F.u_unit;  // plane.rb:82
    const double v = dot(rel, mk(F.ux, F.uy, F.uz)) / F.v_unit;  // plane.rb:83
    if (-0.5 <= u && u <= 0.5 && -0.5 <= v && v <= 0.5) {
      const double dd = norm(ip - o);
      if (dd < nearest) { nearest = dd; face = k; }
    }
  }
  return face;
}
__device__ __forceinline__ bool box_intersect(const DevBox& bx, d3 o, d3 d, HitRec& h) {
  const int face = box_nearest_face(&bx, o.x, o.y, o.z, d.x, d.y, d.z);
  if (face < 0) return false;
  // the winning face's Plane#intersect again: same expressions, same bits
  const DevBoxFace& F = bx.f[face];
  const d3 n = mk(F.nx, F.ny, F.nz);
  const double den = dot(n, d);
  const double t = dot(mk(F.px, F.py, F.pz) - o, n) / den;
  h.p = o + d * t;
  h.dir_in = den < 0;
  h.face = (uint8_t)face;
  return true;
}

// Probe ray of cover_area (world_object.rb:42): from `target` towards the light, unnormalised.
struct CoverRay {
  d3 target, lp, lt, ltn, tl;
  double lt_r;
};
// lt_r = |lt| and ltn = lt / lt_r: Sphere#intersect's invariants of the probe ray
__device__ __forceinline__ void cover_ray_unit(CoverRay& c) {
  c.lt_r = norm(c.lt);
  c.ltn = mk(c.lt.x / c.lt_r, c.lt.y / c.lt_r, c.lt.z / c.lt_r);
}
__device__ __forceinline__ CoverRay make_cover_ray(d3 target, const DevLight& L) {
  CoverRay c;
  c.target = target;
  c.lp = mk(L.px, L.py, L.pz);
  c.lt = c.lp - target;
  cover_ray_unit(c);
  c.tl = target - c.lp;
  return c;
}

// cover_area of ONE object, exactly as the reference evaluates it:
// Sphere#cover_area (sphere.rb:28-57) / WorldObject#cover_area (world_object.rb:41-49).
// BOX = false compiles the box branch out (kernels specialised for sphere/plane scenes).
// KIND tells what the caller already knows about g.type, so that the other branches are not compiled into its loop
// (the sphere branch with its penumbra code is 800 instructions): 0 = anything (the reference's own scan), 1 = a sphere
// or a box (an entry of the sphere filter), 2 = a plane.
template <class Pol, bool BOX = true, int KIND = 0>
__device__ __forceinline__ double cover_object_exact(const FrameParams& P, const DevGeom& g, const CoverRay& c,
                                                     double light_radius, ThreadCtx& ctx) {
  if (KIND != 2 && g.type == RTRB_OBJ_SPHERE) {
    RTRB_COUNT(ctx, RTRB_CNT_COV_SPH);
    HitRec h;
    int factor = 0;
    if (sphere_intersect<Pol>(g, c.target, c.lt, c.lt_r, c.ltn, h) && dot(h.p - c.lp, c.tl) > 0) factor = 1;
    d3 cc = mk(g.px, g.py, g.pz);
    double t = dot(cc - c.target, c.lt) / (c.lt_r * c.lt_r);
    d3 x1 = c.target + c.lt * t;
    double r1 = light_radius * (norm(x1 - c.target) / c.lt_r);
    double dd = norm(x1 - cc);
    if (dd >= r1 + g.radius) return 0;
    double s1 = RTRB_PI * r1 * r1;
    // Lean scenes: light_radius == 0.0, so r1 is a zero or a NaN (0 * inf).  Past the test above dd < R (or a comparison
    // with a NaN failed); then `dd > |R - r1|` = `dd > |R|` cannot hold (R >= 0: dd < R; R < 0: no dd >= 0 is < R; NaN:
    // false), so the partial-overlap branch (sphere.rb:37-47) is unreachable and its acos / sin / divisions are not
    // compiled in
    if constexpr (!Pol::lean) {
      if (dd > fabs(g.radius - r1)) {
        RTRB_COUNT(ctx, RTRB_CNT_COV_SPH_PEN);
        double ct1 = fmin((r1 * r1 + dd * dd - g.radius * g.radius) / (2 * r1 * dd), 1.0);
        double ct2 = fmin((g.radius * g.radius + dd * dd - r1 * r1) / (2 * g.radius * dd), 1.0);
        double th1 = rb_acos<Pol>(ct1, ctx), th2 = rb_acos<Pol>(ct2, ctx);
        double delta_s = ((th1 - m_sin<Pol>(th1)) * r1 * r1 + (th2 - m_sin<Pol>(th2)) * g.radius * g.radius) / 2;
        return factor * delta_s / s1;
      }
    }
    RTRB_COUNT(ctx, RTRB_CNT_COV_SPH_FULL);
    if (r1 > g.radius) return factor * RTRB_PI * g.radius * g.radius / s1;
    return factor;
  }
  if constexpr (BOX && KIND != 2) {
    if (g.type == RTRB_OBJ_BOX) {  // WorldObject#cover_area (world_object.rb:41-49) through Box#intersect
      RTRB_COUNT(ctx, RTRB_CNT_COV_BOX);
      HitRec h;
      if (box_intersect(P.boxes[g.aux], c.target, c.lt, h) && dot(h.p - c.lp, c.tl) > 0) {
        RTRB_COUNT(ctx, RTRB_CNT_COV_BOX_ACC);
        return 1;
      }
      return 0;
    }
  }
  if constexpr (KIND == 1) {
    return 0;  // (unreachable: the sphere filter only lists spheres and boxes)
  } else {
    RTRB_COUNT(ctx, RTRB_CNT_COV_PL);
    HitRec h;
    double den;
    if (plane_intersect(g, c.target, c.lt, h, den) && dot(h.p - c.lp, c.tl) > 0) {
      RTRB_COUNT(ctx, RTRB_CNT_COV_PL_ACC);
      return 1;
    }
    return 0;
  }
}

// World#lit_area (world.rb:62-69) for one light seen from `target`:
// max(1 - sum over ALL objects of cover_area, 0), subtraction in world_objects order.
template <class Pol, bool BOX = true>
static __device__ __noinline__ double lit_area(const FrameParams& P, d3 target, const DevLight& L, ThreadCtx& ctx) {
  const CoverRay c = make_cover_ray(target, L);
  double total = 1;
  for (int i = 0; i < P.n_objects; ++i) {
    const DevGeom g = P.geom[i];
    total -= cover_object_exact<Pol, BOX>(P, g, c, L.radius, ctx);
  }
  return fmax(total, 0.0);
}

// get_a_random_vertical_vector (world_object.rb:105-120)
__device__ __forceinline__ d3 a_vertical_vector(d3 n, ThreadCtx& ctx) {
  if (norm(n) == 0) ctx.status |= RTRB_ST_ZERO_VECTOR;
  if (n.x == 0) {
    if (n.y == 0) return mk(1.0, 0.0, 0.0);
    return mk(0.0, -n.z / n.y, 1.0);
  }
  return mk(-(n.y + n.z) / n.x, 1.0, 1.0);
}

// Float#to_i then Integer#% (texture.rb:24-25): truncation toward zero, then FLOORED modulo by a positive size.
// `t` is already truncated.  Values that fit 32 bits take the integer path (the remainder of an integer division is
// exact either way, so the result equals fmod's: -2.6 % instructions on config 3); anything larger goes through fmod.
template <class Pol>
__device__ __forceinline__ int trunc_mod(double t, int n) {
  if (fabs(t) < 2147483648.0) {
    int m = (int)t % n;
    return m < 0 ? m + n : m;
  }
  double m = m_fmod<Pol>(t, (double)n);
  if (m < 0) m += n;
  return (int)m;
}

// Texture#color (texture.rb:23-28)
template <class Pol>
__device__ __forceinline__ d3 texture_color(const DevMat& m, double uu, double vv, ThreadCtx& ctx) {
  double fu = (uu + m.uoff) / m.hscale, fv = (vv + m.voff) / m.vscale;
  if (!isfinite(fu) || !isfinite(fv)) { ctx.status |= RTRB_ST_NAN_TO_INT; return mk(0, 0, 0); }
  const int u = trunc_mod<Pol>(trunc(fu), m.tex_w), v = trunc_mod<Pol>(trunc(fv), m.tex_h);
  const uint8_t* p = m.tex + ((size_t)v * m.tex_w + u) * 3;
  return mk(__ldg(p) / 256.0, __ldg(p + 1) / 256.0, __ldg(p + 2) / 256.0);
}

// RTRB_RNG_MT: a thread's position in the host-generated MT19937 stream (Random.rand, camera.rb:135 and
// world_object.rb:84, consumed in program order).
struct MtCursor {
  const double* s;
  uint32_t pos, len;
  bool overflow;
  __device__ __forceinline__ double next() {
    double v = 0.0;
    if (pos < len) v = s[pos]; else overflow = true;
    pos++;
    return v;
  }
};

struct StackItem {
  double ox, oy, oz, dx, dy, dz, ax, ay, az;
  int32_t depth;
  uint32_t path;
};
// Fills a work item in place (a StackItem returned by value reorders the local-memory stores of the ray-tree kernels).
__device__ __forceinline__ void set_item(StackItem& s, d3 o, d3 d, d3 att, int32_t depth, uint32_t path) {
  s.ox = o.x; s.oy = o.y; s.oz = o.z;
  s.dx = d.x; s.dy = d.y; s.dz = d.z;
  s.ax = att.x; s.ay = att.y; s.az = att.z;
  s.depth = depth; s.path = path;
}

// intersect_parameters (sphere.rb:88-101 / plane.rb:54-67) of the object g hit by direction d at bh: the normal n
// (not normalised), the offset delta of the children's origins, the refractive rate and whether it may refract.
// BOX = false compiles the box branch out.
struct SurfaceParams {
  d3 n, delta;
  double rate;
  bool can_refract;
};
template <bool BOX>
__device__ __forceinline__ SurfaceParams intersect_parameters(const FrameParams& P, const DevGeom& g, const DevMat& M,
                                                              const HitRec& bh, d3 d) {
  d3 n, delta;
  double rate;
  bool can_refract;
  if (g.type == RTRB_OBJ_SPHERE) {
    d3 c = mk(g.px, g.py, g.pz);
    delta = ((bh.p - c) * RTRB_EPSILON) * (bh.dir_in ? 1.0 : -1.0);  // sphere.rb:84
    n = bh.dir_in ? (bh.p - c) : (c - bh.p);
    rate = bh.dir_in ? M.refractive_rate : 1.0 / M.refractive_rate;
    can_refract = true;
  } else {
    // a plane, or the face of a box that was hit (Box#intersect_parameters delegates, box.rb:102-107)
    d3 f = mk(g.nx, g.ny, g.nz);
    if constexpr (BOX) {
      if (g.type == RTRB_OBJ_BOX) { const DevBoxFace& F = P.boxes[g.aux].f[bh.face]; f = mk(F.nx, F.ny, F.nz); }
    }
    double fd = dot(f, d);
    double nfd = -fd;
    double sgn = nfd > 0 ? 1.0 : (nfd < 0 ? -1.0 : 0.0);
    delta = (f * RTRB_EPSILON) * sgn;  // plane.rb:50
    n = fd > 0 ? -f : f;               // plane.rb:55
    rate = M.refractive_rate;
    can_refract = M.has_refraction != 0;
  }
  return {n, delta, rate, can_refract};
}

// Adds an emitted colour to the sample's sum in emission order (rt_reduce); a channel of the sum above 1 sets
// RTRB_ST_COLOR_GT_1.
__device__ __forceinline__ void emit(d3& sum, d3 c, ThreadCtx& ctx) {
  sum = sum + c;
  if (sum.x > 1 || sum.y > 1 || sum.z > 1) ctx.status |= RTRB_ST_COLOR_GT_1;
}

// Sphere#get_uv (sphere.rb:111-120) / Plane#get_uv (plane.rb:81-85) of the point p of the textured object g.
__device__ __forceinline__ void object_uv(const DevGeom& g, const DevMat& M, d3 p, double& u, double& v, ThreadCtx& ctx) {
  if (g.type == RTRB_OBJ_SPHERE) {
    d3 vec = p - mk(g.px, g.py, g.pz);
    double x = dot(vec, ld3(M.e0)) / g.radius;
    double y = dot(vec, ld3(M.e1)) / g.radius;
    double z = dot(vec, ld3(M.e2)) / g.radius;
    double mm = rb_sqrt(x * x + y * y + z * z + 2 * x + 1, ctx);
    u = (y / mm + 1) / 2;
    v = (-z / mm + 1) / 2;
  } else {
    d3 rel = p - mk(g.px, g.py, g.pz);
    u = dot(rel, ld3(M.e0)) / M.u_unit;
    v = dot(rel, ld3(M.e1)) / M.v_unit;
  }
}

// RayTracer#trace_sync for one sample.  Returns the summed colour; *primary_hit gets the root ray's
// World#intersect winner (-1 miss, -2 highlight-terminated).
template <class Pol, int MAXS, bool MT = false>
__device__ __forceinline__ d3 trace_sample(const FrameParams& P, d3 ro, d3 rd, uint32_t pixel, uint32_t sample,
                                           ThreadCtx& ctx, int* primary_hit, MtCursor* mt = nullptr) {
  StackItem stack[MAXS];
  set_item(stack[0], ro, rd, mk(1.0, 1.0, 1.0), P.trace_depth, 1u);
  int sp = 1;
  d3 sum = mk(0.0, 0.0, 0.0);
  bool first = true;
  const uint32_t K = (uint32_t)(P.mc + 2);
  *primary_hit = -1;

  while (sp > 0) {
    if ((uint32_t)sp > ctx.max_stack) ctx.max_stack = (uint32_t)sp;
    const StackItem it = stack[--sp];
    const bool is_first = first;
    first = false;
    d3 o = mk(it.ox, it.oy, it.oz), d = mk(it.dx, it.dy, it.dz), att = mk(it.ax, it.ay, it.az);
    // rt_map :52
    if (it.depth <= 0 || norm(att) < 0.0001) continue;
    ctx.rays++;

    // ---- World#high_lights (world.rb:83-98); occluders never block (lit_area is truthy) ----
    unsigned long long hl_mask = 0ull;
    int hl_n = 0;
    for (int l = 0; l < P.n_lights; ++l) {
      const DevLight& L = P.lights[l];
      d3 a = mk(L.px, L.py, L.pz) - o;
      double ct = vcos(d, a, ctx);
      double ang = rb_acos<Pol>(ct, ctx);
      if (ang < L.hl_threshold) { hl_mask |= 1ull << l; hl_n++; }
    }
    if (hl_n > 0) {
      for (int l = 0; l < P.n_lights; ++l) {
        if (!((hl_mask >> l) & 1ull)) continue;
        emit(sum, (att * ld3(P.lights[l].color_hl)) / (double)hl_n, ctx);  // ray_tracer.rb:65
      }
      RTRB_COUNT(ctx, RTRB_CNT_HIGHLIGHT);
      if (is_first) *primary_hit = -2;
      continue;
    }

    // ---- World#intersect (world.rb:37-59): linear scan, strict `<`, lowest index wins ties ----
    const double d_r = norm(d);
    const d3 dn = mk(d.x / d_r, d.y / d_r, d.z / d_r);
    double best = P.max_distance;
    int best_i = -1;
    HitRec bh; bh.p = mk(0, 0, 0); bh.dir_in = false; bh.face = 0;
    for (int i = 0; i < P.n_objects; ++i) {
      const DevGeom g = P.geom[i];
      HitRec h;
      bool ok;
      if (g.type == RTRB_OBJ_SPHERE) {
        RTRB_COUNT(ctx, RTRB_CNT_SPH_TEST);
        ok = sphere_intersect<Pol>(g, o, d, d_r, dn, h);
        if (ok) RTRB_COUNT(ctx, RTRB_CNT_SPH_ACC);
      } else if (g.type == RTRB_OBJ_BOX) {
        RTRB_COUNT(ctx, RTRB_CNT_BOX_TEST);
        ok = box_intersect(P.boxes[g.aux], o, d, h);
        if (ok) RTRB_COUNT(ctx, RTRB_CNT_BOX_ACC);
      } else {
        RTRB_COUNT(ctx, RTRB_CNT_PL_TEST);
        double den;
        ok = plane_intersect(g, o, d, h, den);
        if (ok) RTRB_COUNT(ctx, RTRB_CNT_PL_ACC);
      }
      if (ok) {
        double new_dis = norm(o - h.p);  // Ray#distance (algebra.rb:10-12)
        if (new_dis < best) { best = new_dis; best_i = i; bh = h; }
      }
    }
    if (best_i < 0) continue;  // light_dead
    if (is_first) *primary_hit = best_i;
    RTRB_COUNT(ctx, RTRB_CNT_HITS);

    const DevGeom g = P.geom[best_i];
    const DevMat& M = P.mat[best_i];
    const auto [n, delta, rate, can_refract] = intersect_parameters<true>(P, g, M, bh, d);
    const d3 nn = normalize(n, ctx);
    // get_reflection_by_ray_and_n (world_object.rb:121-125)
    double cos_theta = vcos(d, -n, ctx);
    d3 refl_dir = normalize(nn * (2 * cos_theta * d_r) + d, ctx);
    d3 refl_org = bh.p + delta;
    // get_refraction_by_ray_and_n (world_object.rb:127-137)
    bool has_refr = false;
    d3 refr_dir = mk(0, 0, 0), refr_org = mk(0, 0, 0);
    if (can_refract) {
      double cc = vcos(d, n, ctx);
      double sin_i = rb_sqrt(1 - cc * cc, ctx);
      double sin_r = sin_i / rate;
      if (!(sin_r >= 1)) {
        if (sin_r < -1 || sin_r > 1) ctx.status |= RTRB_ST_MATH_DOMAIN;
        double r = m_asin<Pol>(sin_r);
        refr_dir = nn * (-m_cos<Pol>(r)) + normalize(refl_dir + d, ctx) * sin_r;
        refr_org = bh.p - nn * RTRB_EPSILON;
        has_refr = true;
      }
    }
    // push children: reflection first, refraction second (popped first)  ray_tracer.rb:87-121
    if (sp + 2 + P.mc > MAXS) { ctx.status |= RTRB_ST_STACK_OVERFLOW; continue; }
    set_item(stack[sp++], refl_org, refl_dir, att * ld3(M.refl), it.depth - 1, it.path * K + 0u);
    if (has_refr) {
      RTRB_COUNT(ctx, RTRB_CNT_REFR);
      set_item(stack[sp++], refr_org, refr_dir, att * ld3(M.refr), it.depth - 1, it.path * K + 1u);
    }

    // ---- World#local_lights (world.rb:72-80) fused with WorldObject#local_lighting (:51-74) ----
    const d3 shade_from = bh.p + delta;
    d3 contrib = mk(0.0, 0.0, 0.0);
    int n_lit = 0;
    for (int l = 0; l < P.n_lights; ++l) {
      const DevLight& L = P.lights[l];
      ctx.shadow++;
      double area = lit_area<Pol>(P, shade_from, L, ctx);
      if (area > 0) {
        d3 lc = ld3(L.color) * (rb_pow<Pol>(area, P.soft_shadow_exponent) / (double)P.n_lights);
        d3 lv = normalize(mk(L.px, L.py, L.pz) - bh.p, ctx);  // shading point is WITHOUT delta (:152)
        double ldn = dot(lv, nn);
        if (ldn > 1) ldn = 1.0; else if (ldn < 0) ldn = 0.0;
        contrib = contrib + lc * ldn;
        n_lit++;
      }
    }
    if (n_lit == 0) {
      // WorldObject#path_tracing (world_object.rb:76-90): mc rays, no local/ambient colour
      if (P.mc > 0) {
        d3 att_pt = ld3(M.diffuse) / (double)P.mc;
        d3 leftv = normalize(a_vertical_vector(n, ctx), ctx);
        d3 upv = cross(nn, leftv);
        for (int m = 0; m < P.mc; ++m) {
          uint32_t child = it.path * K + (uint32_t)(2 + m);
          double u_theta, u_phi;  // theta's draw first (world_object.rb:84)
          if constexpr (MT) {
            u_theta = mt->next(); u_phi = mt->next();
          } else {
            uint32_t c0 = pixel, c1 = sample, c2 = child, c3 = 1u;
            philox4x32_10(P.key0, P.key1, c0, c1, c2, c3);
            u_theta = res53(c0, c1); u_phi = res53(c2, c3);
          }
          double theta = u_theta * RTRB_PI / 2, phi = u_phi * RTRB_PI * 2;
          d3 dir = nn * m_sin<Pol>(theta) + (leftv * m_cos<Pol>(phi) + upv * m_sin<Pol>(phi)) * m_cos<Pol>(theta);
          RTRB_COUNT(ctx, RTRB_CNT_MC);
          StackItem& s = stack[sp++];
          d3 a2 = att * att_pt;
          s.ox = shade_from.x; s.oy = shade_from.y; s.oz = shade_from.z;
          s.dx = dir.x; s.dy = dir.y; s.dz = dir.z;
          s.ax = a2.x; s.ay = a2.y; s.az = a2.z;
          s.depth = it.depth - 1; s.path = child;
        }
      }
    } else {
      RTRB_COUNT(ctx, RTRB_CNT_LOCAL);
      if (ctx.detail) ctx.c[RTRB_CNT_LIT] += n_lit;
      contrib = contrib / (double)n_lit;  // world_object.rb:66-68
      d3 filter = mk(1.0, 1.0, 1.0);
      if (M.tex != nullptr) {
        double u, v;
        object_uv(g, M, bh.p, u, v, ctx);
        RTRB_COUNT(ctx, RTRB_CNT_TEXEL);
        filter = texture_color<Pol>(M, u, v, ctx) * filter;
      }
      d3 local = ((contrib * ld3(M.diffuse)) * filter) + ld3(M.ambient);
      emit(sum, att * local, ctx);  // ray_tracer.rb:152
    }
  }
  return sum;
}

// Camera#lens_func (camera.rb:129-151) for pixel (x, y) and aperture angle theta.
template <class Pol>
__device__ __forceinline__ void lens_ray(const FrameParams& P, int x, int y, double theta, d3& ro, d3& rd) {
  d3 pos = ld3(P.pos), left = ld3(P.left), upn = ld3(P.up_n), front = ld3(P.front);
  // host-built tables of 2.0 * (x.to_f / width - 0.5) * retina_width and the y analogue (camera.rb:133-134)
  const double sx = P.lens_sx[x];
  const double sy = P.lens_sy[y];
  d3 retina_position = (ld3(P.retina_center) + left * sx) + upn * sy;
  // aperture_radius == 0.0 (pinhole): the reference still evaluates (left*cos + up*sin) * 0.0 = (+-0, +-0, +-0);
  // adding a zero of either sign to `pos` gives `pos` (up to the sign of an exact zero, which no later
  // expression can observe), so the two FP64 transcendentals are skipped.
  d3 rand_vector = mk(0.0, 0.0, 0.0);
  if (P.aperture_radius != 0.0) rand_vector = (ld3(P.left_n) * m_cos<Pol>(theta) + upn * m_sin<Pol>(theta)) * P.aperture_radius;
  d3 aperture = pos + rand_vector;
  d3 rf = pos - retina_position;  // ray retina -> lens centre
  double t = dot(ld3(P.focal_point) - retina_position, front) / dot(front, rf);  // intersect_plane :123-127
  d3 target = retina_position + rf * t;
  ro = aperture;
  rd = target - aperture;
}
// The primary ray of sample j of a frame's pixel (x, y): lens_ray with the aperture angle drawn from Philox
// (Random.rand, camera.rb:135).  The frame kernels and camera_rays share it, so traced camera rays reproduce frames.
template <class Pol>
__device__ __forceinline__ void camera_ray(const FrameParams& P, int x, int y, uint32_t pixel, uint32_t j, d3& ro, d3& rd) {
  double theta = 0.0;
  if (P.aperture_radius != 0.0) {
    uint32_t c0 = pixel, c1 = j, c2 = 0u, c3 = 0u;
    philox4x32_10(P.key0, P.key1, c0, c1, c2, c3);
    theta = res53(c0, c1);
  }
  lens_ray<Pol>(P, x, y, theta, ro, rd);
}

// array_to_color (camera.rb:153-156) + the byte truncation of PNG::Color.new
__device__ __forceinline__ uint8_t quantise_u8(double c) {
  // [c*256, 255].min truncated to a byte; negatives and NaN give 0.  c*256 is an exact scaling, and the
  // saturating round-toward-zero conversion followed by an integer clamp is the same function.
  int v = __double2int_rz(c * 256.0);  // NaN -> 0, +-inf / out of range saturate
  v = v < 0 ? 0 : (v > 255 ? 255 : v);
  return (uint8_t)v;
}
// render_at's result for pixel (x, y): row = y, column = x (camera.rb:98,105)
__device__ __forceinline__ void write_pixel(const FrameParams& P, int x, int y, double r, double g, double b) {
  size_t px = (size_t)y * P.width + x;
  if (P.rgb) { P.rgb[px * 3 + 0] = r; P.rgb[px * 3 + 1] = g; P.rgb[px * 3 + 2] = b; }
  if (P.pixel_format == RTRB_FMT_PNG_RGB8) {
    // PNG scanline: filter-type byte 0, then the row's RGB8 pixels (the stream a PNG encoder deflates into IDAT)
    uint8_t* row = P.rgba + (size_t)y * ((size_t)P.width * 3 + 1);
    if (x == 0) row[0] = 0;
    uint8_t* o = row + 1 + (size_t)x * 3;
    o[0] = quantise_u8(r); o[1] = quantise_u8(g); o[2] = quantise_u8(b);
    return;
  }
  if (P.pixel_format == RTRB_FMT_RGB8) {
    // alpha is the constant 255 (camera.rb:155): three byte stores; a warp's 8x4 pixel block is four
    // 24-byte runs which the L2 merges before the frame leaves over PCIe / NVLink
    uint8_t* o = P.rgba + px * 3;
    o[0] = quantise_u8(r); o[1] = quantise_u8(g); o[2] = quantise_u8(b);
    return;
  }
  uchar4 q = make_uchar4(quantise_u8(r), quantise_u8(g), quantise_u8(b), 255);
  reinterpret_cast<uchar4*>(P.rgba)[px] = q;
}

// Work item w of a frame with S samples per pixel -> (tile slot, sample j); the samples of a slot are consecutive.
__device__ __forceinline__ void decode_work(unsigned long long w, uint32_t S, uint32_t& slot, uint32_t& j) {
  if (S == 1u) { slot = (uint32_t)w; j = 0u; }
  else { slot = (uint32_t)(w / S); j = (uint32_t)(w - (unsigned long long)slot * S); }
}

// Decodes work item -> (tile slot k, in-tile q, x, y); returns false when the pixel is outside the window.
__device__ __forceinline__ bool decode_pixel(const FrameParams& P, uint32_t slot, int& x, int& y) {
  uint32_t k = slot / RTRB_SUPER_PIXELS, q = slot % RTRB_SUPER_PIXELS;
  uint32_t tx, ty;
  if (P.tiles_magic != 0u) {  // whole frame, one renderer: row-major tiles, no dependent load
    ty = __umulhi(k, P.tiles_magic);
    tx = k - ty * (uint32_t)P.stx_count;
  } else {
    const uint32_t tile = (uint32_t)P.tiles[k];  // tx | ty << 16
    tx = tile & 0xffffu; ty = tile >> 16;
  }
  int qx, qy;
  rtrb_morton_decode(q, &qx, &qy);
  x = (int)tx * RTRB_SUPER + qx;
  y = (int)ty * RTRB_SUPER + qy;
  return x >= P.x0 && x < P.x1 && y >= P.y0 && y < P.y1;
}

// Super-tile row of the sky-fill order (rtrb_sky_fill) that holds item i of one kind, traced tiles or sky-run tiles, given
// `before(r)`, the items of the rows < r: the last row r with before(r) <= i.  i comes from blockIdx, so the search runs on
// the uniform datapath, once per warp.
template <class Before>
__device__ __forceinline__ int sky_fill_row(const FrameParams& P, uint32_t i, Before before) {
  const int sty = (P.height + RTRB_SUPER - 1) / RTRB_SUPER;
  int r = 0;
#pragma unroll
  for (int s = 64; s > 0; s >>= 1)
    if (r + s < sty && before(r + s) <= i) r += s;
  return r;
}

// decode_pixel of a sky-fill frame: slot k * 1024 + q is pixel q of the k-th traced tile in row-major order.  One sample
// per pixel, so k comes from blockIdx alone.
__device__ __forceinline__ bool decode_traced_pixel(const FrameParams& P, uint32_t slot, int& x, int& y) {
  const uint32_t k = blockIdx.x / (RTRB_SUPER_PIXELS / blockDim.x), q = slot % RTRB_SUPER_PIXELS;
  const int ty = sky_fill_row(P, k, [&](int r) { return (uint32_t)P.k_trace_before[r]; });
  const uint32_t c = k - P.k_trace_before[ty];
  const uchar2 run = P.k_sky_run[ty];
  const uint32_t tx = c < run.x ? c : c + (uint32_t)(run.y - run.x);
  int qx, qy;
  rtrb_morton_decode(q, &qx, &qy);
  x = (int)tx * RTRB_SUPER + qx;
  y = ty * RTRB_SUPER + qy;
  return x >= P.x0 && x < P.x1 && y >= P.y0 && y < P.y1;
}

// A fill CTA of a sky-fill frame: sky tiles [f, f + RTRB_SKY_FILL_TILES) of the runs in row-major order, f = the CTA's index
// past the trace CTAs times RTRB_SKY_FILL_TILES, clipped to the frame.  Each pixel gets what trace_pre_body's sky branch
// gives it: black in the pixel format, +0.0 in rgb, hit id -1, one ray and one sample in ctx.  A warp stores a pixel row
// at a time, lane = pixel, with short independent stores: a lone warp's latency, not bandwidth, bounds the CTA.
__device__ __forceinline__ void store_sky_tiles(const FrameParams& P, ThreadCtx& ctx) {
  const uint32_t f0 = (blockIdx.x - P.sky_fill_traced * (RTRB_SUPER_PIXELS / blockDim.x)) * RTRB_SKY_FILL_TILES;
  const uint32_t f1 = min(f0 + RTRB_SKY_FILL_TILES, P.sky_fill_tiles);
  const int lane = threadIdx.x & 31;
  uint32_t px = 0;
  for (uint32_t i = f0; i < f1; ++i) {
    auto sky_before = [&](int r) { return (uint32_t)(r * P.stx_count - P.k_trace_before[r]); };
    const int ty = sky_fill_row(P, i, sky_before);
    const int x = (P.k_sky_run[ty].x + (int)(i - sky_before(ty))) * RTRB_SUPER + lane, y0 = ty * RTRB_SUPER;
    if (x >= P.width) continue;
    const int y1 = min(y0 + RTRB_SUPER, P.height);
    for (int y = y0 + (int)(threadIdx.x >> 5); y < y1; y += (int)(blockDim.x >> 5)) {
      const size_t px_i = (size_t)y * P.width + x;
      if (P.pixel_format == RTRB_FMT_RGBA8) {
        reinterpret_cast<uchar4*>(P.rgba)[px_i] = make_uchar4(0, 0, 0, 255);
      } else {
        uint8_t* o = P.rgba + px_i * 3;
        if (P.pixel_format == RTRB_FMT_PNG_RGB8) {  // PNG scanline: the filter-type byte 0 ahead of pixel 0
          o = P.rgba + (size_t)y * ((size_t)P.width * 3 + 1) + 1 + (size_t)x * 3;
          if (x == 0) o[-1] = 0;
        }
        o[0] = 0; o[1] = 0; o[2] = 0;
      }
      if (P.rgb) { P.rgb[px_i * 3 + 0] = 0.0; P.rgb[px_i * 3 + 1] = 0.0; P.rgb[px_i * 3 + 2] = 0.0; }
      if (P.hit) P.hit[px_i] = -1;
      ++px;
    }
  }
  ctx.rays = px;
  if (ctx.detail) ctx.c[RTRB_CNT_SAMPLES] = px;
}

// Records a pixel whose sample set a status bit (the reference would have raised there): status word and the
// first offending pixel in the reference's pixel order (x outer, y inner).  Clears ctx.status so that a thread
// which goes on to other pixels (grid-stride / persistent loops) attributes later bits to the right pixel.
__device__ __forceinline__ void report_status(const FrameParams& P, ThreadCtx& ctx, int x, int y) {
  if (ctx.status) {
    atomicOr(&P.status[0], ctx.status);
    // smallest x*H + y wins; stored complemented (atomicMax) so the control block can be zero-initialised
    atomicMax(P.first_bad, ~((unsigned long long)x * (unsigned long long)P.height + (unsigned long long)y));
    ctx.status = 0;
  }
}

__device__ __forceinline__ void flush_ctx(const FrameParams& P, ThreadCtx& ctx, int x, int y, bool active) {
  // warp totals by hardware reduction (REDUX), then one fire-and-forget RED per warp and counter, spread over
  // RTRB_HOT_SLICES address pairs (the host sums the slices): no block barrier, and no single L2 line taking
  // 65 K atomics per frame
  const unsigned full = 0xffffffffu;
  const uint32_t rays = __reduce_add_sync(full, ctx.rays), shadow = __reduce_add_sync(full, ctx.shadow),
                 ms = __reduce_max_sync(full, ctx.max_stack);
  const int lane = threadIdx.x & 31;
  if (lane == 0) {
    unsigned long long* hot = P.hot + 2u * ((blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) & (RTRB_HOT_SLICES - 1));
    if (rays) atomicAdd(&hot[0], (unsigned long long)rays);
    if (shadow) atomicAdd(&hot[1], (unsigned long long)shadow);
    if (ms > 1u) atomicMax(&P.status[1], ms);  // 1 (just the root) is the host-side default
  }
  if (ctx.detail) {
#pragma unroll
    for (int i = 0; i < RTRB_CNT_N; ++i) {
      if (i == RTRB_CNT_RAYS || i == RTRB_CNT_SHADOW) continue;
      const uint32_t v = __reduce_add_sync(full, ctx.c[i]);
      if (lane == 0 && v) atomicAdd(&P.counters[i], (unsigned long long)v);
    }
  }
  if (active) report_status(P, ctx, x, y);
}

__device__ __forceinline__ void init_ctx(ThreadCtx& ctx, bool detail) {
  ctx.status = 0; ctx.rays = 0; ctx.shadow = 0; ctx.max_stack = 0; ctx.detail = detail;
  if (detail) {  // the lean kernels never touch c[]: no zeroing, no local-memory array
#pragma unroll
    for (int i = 0; i < RTRB_CNT_N; ++i) ctx.c[i] = 0;
  }
}

// Folds the counters / status a callee collected in its own block into the thread's.
__device__ __forceinline__ void merge_ctx(ThreadCtx& ctx, const ThreadCtx& t) {
  ctx.status |= t.status;
  ctx.rays += t.rays; ctx.shadow += t.shadow;
  if (t.max_stack > ctx.max_stack) ctx.max_stack = t.max_stack;
  if (ctx.detail) {
#pragma unroll
    for (int i = 0; i < RTRB_CNT_N; ++i) ctx.c[i] += t.c[i];
  }
}

// FAST64 entry point, defined in rtrb_trace_fast.cuh (only instantiated by that translation unit).  CULL: the depth-1
// frame kernels' candidate masks (FrameParams::k_cam_tx, light_cand); cam_cand = those of the pixel's super-tile, and
// no_highlight = its tile certificate rules out every highlight (FrameParams::k_tile_rows), and ground = its ground
// certificate holds and its mask is empty (FrameParams::k_ground_rows).
template <class Pol, int MAXS, bool BVH, bool BOX, bool CULL = false>
__device__ __forceinline__ d3 trace_sample_fast(const FrameParams& P, d3 ro, d3 rd, uint32_t pixel, uint32_t sample,
                                                ThreadCtx& ctx, int* primary_hit, uint32_t cam_cand = 0xffffffffu,
                                                bool no_highlight = false, bool ground = false);

// BVH: FAST64 with the sphere BVH instead of the linear filter.
// BOX: the FAST64 kernels carry the Box code only in their full-counter (DETAIL) variants; scenes with a
// box are always dispatched there (rtrb_api.cu, pick_trace_kernels), so the lean hot kernels stay sphere/plane-only.
template <class Pol, int MAXS, bool BVH, bool BOX, bool CULL = false>
__device__ __forceinline__ d3 trace_dispatch(const FrameParams& P, d3 ro, d3 rd, uint32_t pixel, uint32_t sample,
                                             ThreadCtx& ctx, int* primary_hit, uint32_t cam_cand = 0xffffffffu,
                                             bool no_highlight = false, bool ground = false) {
  if constexpr (Pol::fast)
    return trace_sample_fast<Pol, MAXS, BVH, BOX, CULL>(P, ro, rd, pixel, sample, ctx, primary_hit, cam_cand, no_highlight,
                                                        ground);
  else return trace_sample<Pol, MAXS>(P, ro, rd, pixel, sample, ctx, primary_hit);
}

// One thread per (pixel, sample j < pre_sample_times): the first loop of render_at (camera.rb:73-78).
// The FAST64 depth-1 kernels may be launched with programmatic stream serialization (frame overlap, rtrb_api.cu): every
// CTA lets the next frame's kernel launch as soon as it starts, and every thread traces before it waits for the
// previous grid on the stream to complete, so the only things ordered behind that grid are this frame's global writes.
// Everything before the wait reads only FrameParams, the scene tables and the lens tables.  Launched without the
// attribute, the wait returns at once.
// PASS: the pass kernels of a progressive frame.  One thread per (pixel, sample j in [pass_begin, pass_end)); the
// colour goes to the sample buffer at (slot * pre + j), the stride of the whole frame.  No overlap, no in-thread resolve.
// The FAST64 depth-1 linear-filter kernels (the pass kernels included) narrow the camera apex test to the candidate masks
// of the pixel's super-tile, store sky tiles without tracing and skip the highlight test where the tile certificates
// (FrameParams::k_tile_rows) allow, and skip the camera filter on ground tiles (FrameParams::k_ground_rows).
template <class Pol, int MAXS, bool DETAIL, bool BVH = false, bool PASS = false>
__device__ __forceinline__ void trace_pre_body(const FrameParams& P) {
  constexpr bool kOverlap = Pol::fast && MAXS == 1 && !PASS;
  constexpr bool kCull = Pol::fast && MAXS == 1 && !BVH;
  if constexpr (kOverlap) cudaTriggerProgrammaticLaunchCompletion();
  const uint32_t S = PASS ? (uint32_t)(P.pass_end - P.pass_begin) : (uint32_t)P.pre;
  const unsigned long long w = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long total = (unsigned long long)P.n_tiles * RTRB_SUPER_PIXELS * S;
  ThreadCtx ctx;
  init_ctx(ctx, DETAIL);
  int x = 0, y = 0;
  bool active = false;
  // sky-fill frames (FrameParams::sky_fill_tiles): the CTAs past those of the traced tiles store the sky runs
  bool fill = false, fill_frame = false;
  if constexpr (kOverlap && kCull) {
    fill_frame = P.sky_fill_tiles != 0u;
    fill = fill_frame && blockIdx.x >= P.sky_fill_traced * (RTRB_SUPER_PIXELS / blockDim.x);
  }
  if (!fill && w < total) {
    uint32_t slot, j;
    decode_work(w, S, slot, j);
    if constexpr (PASS) j += (uint32_t)P.pass_begin;
    active = fill_frame ? decode_traced_pixel(P, slot, x, y) : decode_pixel(P, slot, x, y);
    if (active) {
      const uint32_t pixel = (uint32_t)y * (uint32_t)P.width + (uint32_t)x;
      d3 ro, rd;
      int ph;
      d3 col;
      if constexpr (kCull) {
        const int tx = x >> 5, ty = y >> 5;
        const uint32_t cand = P.k_cam_tx[min(tx, RTRB_CAM_TX - 1)] & P.k_cam_ty[min(ty, RTRB_CAM_TY - 1)];
        const uchar4 rows = tx < RTRB_CAM_TX ? P.k_tile_rows[tx] : make_uchar4(0, 0, 0, 0);
        if (cand == 0u && ty >= rows.x && ty < rows.y) {
          // sky tile: the ray meets no sphere (empty mask), no plane and no highlight cone, and no exact test runs, so
          // rt_map's result is known: one ray, nothing emitted (sum stays +0.0), hit id -1
          col = mk(0.0, 0.0, 0.0);
          ph = -1;
          ctx.rays = 1;
        } else {
          const uchar2 gr = tx < RTRB_CAM_TX ? P.k_ground_rows[tx] : make_uchar2(0, 0);
          const bool ground = cand == 0u && ty >= gr.x && ty < gr.y;
          camera_ray<Pol>(P, x, y, pixel, j, ro, rd);
          col = trace_dispatch<Pol, MAXS, BVH, DETAIL, true>(P, ro, rd, pixel, j, ctx, &ph, cand, ty >= rows.z && ty < rows.w,
                                                             ground);
        }
      } else {
        camera_ray<Pol>(P, x, y, pixel, j, ro, rd);
        col = trace_dispatch<Pol, MAXS, BVH, DETAIL>(P, ro, rd, pixel, j, ctx, &ph);
      }
      RTRB_COUNT(ctx, RTRB_CNT_SAMPLES);
      if constexpr (kOverlap) cudaGridDependencySynchronize();
      if constexpr (PASS) {
        double* out = P.samples + ((unsigned long long)slot * (uint32_t)P.pre + j) * 3ull;
        out[0] = col.x; out[1] = col.y; out[2] = col.z;
      } else if (P.fuse_resolve != RTRB_RESOLVE_SAMPLE_BUFFER) {  // RTRB_RESOLVE_IN_THREAD (IN_CTA is ray-tree only)
        // one sample, positive threshold: mean = s / 1.0 = s and variance = 0 < threshold (camera.rb:80-87)
        write_pixel(P, x, y, col.x, col.y, col.z);
      } else {
        double* out = P.samples + w * 3ull;
        out[0] = col.x; out[1] = col.y; out[2] = col.z;
      }
      if (j == 0 && P.hit) P.hit[(size_t)y * P.width + x] = ph;
    }
  }
  if (kOverlap && !active) cudaGridDependencySynchronize();  // before flush_ctx's counters
  if (fill) store_sky_tiles(P, ctx);
  flush_ctx(P, ctx, x, y, active);
  // the next frame's control block: that frame touches it only after its own wait, i.e. after this grid completed
  if (kOverlap && blockIdx.x == 0u && P.ctl_next != nullptr)
    for (uint32_t i = threadIdx.x; i < P.ctl_next_words; i += blockDim.x) P.ctl_next[i] = 0ull;
}

// Extra samples j in [pre, max) of the pixels that failed the variance test (camera.rb:88-93);
// persistent grid-stride loop because the pixel count is only known on the device.
template <class Pol, int MAXS, bool DETAIL, bool BVH = false>
__device__ __forceinline__ void trace_extra_body(const FrameParams& P) {
  const uint32_t E = (uint32_t)(P.max_samples - P.pre);
  const unsigned long long total = (unsigned long long)(*P.extra_count) * E;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  ThreadCtx ctx;
  init_ctx(ctx, DETAIL);
  int x = 0, y = 0;
  bool any = false;
  for (unsigned long long w = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += stride) {
    const uint32_t e = (uint32_t)(w / E), j = (uint32_t)P.pre + (uint32_t)(w % E);
    const uint32_t slot = P.extra_list[e];
    if (!decode_pixel(P, slot, x, y)) continue;
    any = true;
    const uint32_t pixel = (uint32_t)y * (uint32_t)P.width + (uint32_t)x;
    d3 ro, rd;
    camera_ray<Pol>(P, x, y, pixel, j, ro, rd);
    int ph;
    d3 col = trace_dispatch<Pol, MAXS, BVH, DETAIL>(P, ro, rd, pixel, j, ctx, &ph);
    RTRB_COUNT(ctx, RTRB_CNT_SAMPLES);
    double* out = P.extra_samples + w * 3ull;
    out[0] = col.x; out[1] = col.y; out[2] = col.z;
    report_status(P, ctx, x, y);  // this pixel's bits, before the loop moves to another pixel
  }
  flush_ctx(P, ctx, x, y, any);
}

// mean of the pre samples in order, then the variance test (camera.rb:72-87); `s` = the pixel's S sample colours
__device__ __forceinline__ void pre_mean_of(const double* s, const int S, double& ax, double& ay, double& az,
                                            double& variance) {
  ax = 0.0; ay = 0.0; az = 0.0;
  for (int j = 0; j < S; ++j) { ax += s[j * 3 + 0]; ay += s[j * 3 + 1]; az += s[j * 3 + 2]; }
  ax = ax / (double)S; ay = ay / (double)S; az = az / (double)S;
  variance = 0;
  for (int j = 0; j < S; ++j) {
    double dx = s[j * 3 + 0] - ax, dy = s[j * 3 + 1] - ay, dz = s[j * 3 + 2] - az;
    double m = fmax(dx, fmax(dy, dz));  // (sample - mean).to_a.max, signed
    variance += m * m;
  }
  variance /= (double)S;
}
__device__ __forceinline__ void pre_mean(const FrameParams& P, uint32_t slot, double& ax, double& ay, double& az,
                                         double& variance) {
  pre_mean_of(P.samples + (size_t)slot * P.pre * 3, P.pre, ax, ay, az, variance);
}

// (average * pre + extra) / max  (camera.rb:93), in place.  The empty extra loop passes an extra sum of literal 0.0:
// the addition turns a -0.0 product into +0.0, and the FP RGB output keeps that sign.
__device__ __forceinline__ void final_average(double& ax, double& ay, double& az, int pre, double cx, double cy,
                                              double cz, int max_samples) {
  const double fp = (double)pre, fm = (double)max_samples;
  ax = (ax * fp + cx) / fm; ay = (ay * fp + cy) / fm; az = (az * fp + cz) / fm;
}

// The extra-sample branch of render_at (camera.rb:87-93) for the pixels whose variance test failed (`adaptive`):
// counts them, and when max > pre queues each one for the extra-sample pass (slot in extra_list[], its mean (ax, ay,
// az) in pre_avg[]) and returns true; when max <= pre the extra loop is empty and the mean is rescaled in place.
// One ballot over the warp, one atomic per warp for the counter and one for the list, each lane's list position from
// a prefix popcount of the ballot.  ALL 32 LANES OF THE WARP MUST CALL IT (full-mask ballot and shuffle).
__device__ __forceinline__ bool queue_adaptive(const FrameParams& P, bool adaptive, uint32_t slot, double& ax, double& ay,
                                               double& az) {
  const unsigned amask = __ballot_sync(0xffffffffu, adaptive);
  bool queued = false;
  if (amask != 0u) {
    const int lane = threadIdx.x & 31, leader = __ffs(amask) - 1;
    uint32_t base = 0;
    if (lane == leader) {
      const uint32_t n = __popc(amask);
      atomicAdd(&P.counters[RTRB_CNT_ADAPTIVE], (unsigned long long)n);
      if (P.max_samples > P.pre) base = atomicAdd(P.extra_count, n);
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    if (adaptive) {
      if (P.max_samples > P.pre) {
        const uint32_t e = base + __popc(amask & ((1u << lane) - 1u));
        P.extra_list[e] = slot;
        double* m = P.pre_avg + (size_t)e * 3u;
        m[0] = ax; m[1] = ay; m[2] = az;
        queued = true;
      } else {
        final_average(ax, ay, az, P.pre, 0.0, 0.0, 0.0, P.max_samples);
      }
    }
  }
  return queued;
}

// RTRB_RNG_MT: Camera#render_at (camera.rb:70-99) for ONE pixel in ONE thread, because the reference's
// MT19937 draws are consumed in program order: every sample's lens draw (camera.rb:135, drawn even when the
// aperture is 0), its Monte-Carlo draws in LIFO ray order, then the next sample, then the adaptive samples.
// The thread reads its draws from mt_stream starting at mt_offset[pixel order] and reports how many it used;
// the host iterates offsets = prefix sums of the counts until they stop changing (rtrb_api.cu).
template <class Pol, int MAXS, bool DETAIL>
__device__ __forceinline__ void trace_mt_body(const FrameParams& P) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  ThreadCtx ctx;
  init_ctx(ctx, DETAIL);
  int x = 0, y = 0;
  bool active = false;
  if (slot < (uint32_t)P.n_tiles * RTRB_SUPER_PIXELS) active = decode_pixel(P, slot, x, y);
  if (active) {
    const uint32_t pixel = (uint32_t)y * (uint32_t)P.width + (uint32_t)x;
    const uint32_t order = (uint32_t)(x - P.x0) * (uint32_t)(P.y1 - P.y0) + (uint32_t)(y - P.y0);
    MtCursor cur;
    cur.s = P.mt_stream; cur.pos = P.mt_offset[order]; cur.len = P.mt_len; cur.overflow = false;
    const uint32_t start = cur.pos;
    const int S = P.pre;
    double* smp = P.samples + (size_t)slot * S * 3;
    for (int j = 0; j < S; ++j) {
      const double theta = cur.next();
      d3 ro, rd;
      lens_ray<Pol>(P, x, y, theta, ro, rd);
      int ph;
      d3 col = trace_sample<Pol, MAXS, true>(P, ro, rd, pixel, (uint32_t)j, ctx, &ph, &cur);
      RTRB_COUNT(ctx, RTRB_CNT_SAMPLES);
      smp[j * 3 + 0] = col.x; smp[j * 3 + 1] = col.y; smp[j * 3 + 2] = col.z;
      if (j == 0 && P.hit) P.hit[(size_t)y * P.width + x] = ph;
    }
    double ax, ay, az, variance;
    pre_mean(P, slot, ax, ay, az, variance);
    if (variance >= P.variant_threshold) {
      atomicAdd(&P.counters[RTRB_CNT_ADAPTIVE], 1ull);
      double cx = 0.0, cy = 0.0, cz = 0.0;
      for (int j = S; j < P.max_samples; ++j) {
        const double theta = cur.next();
        d3 ro, rd;
        lens_ray<Pol>(P, x, y, theta, ro, rd);
        int ph;
        d3 col = trace_sample<Pol, MAXS, true>(P, ro, rd, pixel, (uint32_t)j, ctx, &ph, &cur);
        RTRB_COUNT(ctx, RTRB_CNT_SAMPLES);
        cx += col.x; cy += col.y; cz += col.z;
      }
      final_average(ax, ay, az, S, cx, cy, cz, P.max_samples);
    }
    write_pixel(P, x, y, ax, ay, az);
    P.mt_count[order] = cur.overflow ? 0xFFFFFFFFu : cur.pos - start;
  }
  flush_ctx(P, ctx, x, y, active);
}

}  // namespace rtrb
