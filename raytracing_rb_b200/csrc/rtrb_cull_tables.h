// rtrb_cull_tables.h — host-only builders of the candidate masks of the depth-1 linear-filter kernels (DESIGN.md §4,
// "candidate masks").  Plain C++ (no CUDA types), so tests/cull_tables_harness.cpp compiles the same code with g++.
//
// The apex tables (FrameParams::cam_tab, light_tab) keep sphere k for a line through the apex A with FP32 unit
// direction u unless b*b < Kq, b = V.u, where entry k = (V, Kq) = (C - A rounded to float, Kq).  Each mask below holds,
// for one set of lines, every sphere whose apex test can keep one of those lines; the kernels then run the apex test
// on the set bits only, so the survivor mask is exactly the one the full scan yields.
//
// Both maps are of LINES through the apex (the apex test cannot tell u from -u): a line is parametrised by direction
// ratios, which are linear-fractional in any point on it, so the range of a ratio over a box is taken at the box's
// vertices and is bounded whenever the denominator keeps one sign over the box.
#pragma once
#include <math.h>
#include <stdint.h>

#define RTRB_CAM_TX 128      // camera masks: super-tile columns / rows (4096 x 2560 pixels); tiles beyond the
#define RTRB_CAM_TY 80       // last one share its entry, which then holds the union of their masks
#define RTRB_LIGHT_BINS 32   // light masks: bins per direction ratio

// Radius of the cylinder around V that holds every line through the apex the test can keep, or -1 when the test can
// keep any line (NaN / non-finite entries, Kq <= 0, magnitudes where FP32 rounding is not bounded this way).
// The test's error: |u| = 1 +- 2^-18 (FP32 normalisation with rsqrt.approx), b = V.u within 3 ulp-sums of |V||u|,
// b*b rounded.  Kept only if |V.u^| >= q (below), so the line's distance h to V has h^2 <= |V|^2 - q^2.  The bound is
// widened by 2^-18 |V|^2 and 2^-20 relative.
inline double rtrb_apex_reach(const float t[4]) {
  const double eps = 5.9604644775390625e-8, du = 3.814697265625e-6;  // 2^-24, 2^-18
  const double vx = t[0], vy = t[1], vz = t[2], kq = t[3];
  if (!(isfinite(vx) && isfinite(vy) && isfinite(vz))) return -1.0;
  const double v2 = vx * vx + vy * vy + vz * vz, vn = sqrt(v2);
  if (!(vn < 1e18)) return -1.0;         // b * b may overflow to +inf (or NaN) and survive any Kq
  if (kq == INFINITY) return 0.0;        // padding: never survives
  if (!(kq > 1e-30)) return -1.0;        // NaN Kq is stored as -inf: always survives; tiny Kq: subnormal products
  const double q = (sqrt(kq) * (1.0 - 2.0 * eps) - 3.01 * eps * vn * (1.0 + du)) / (1.0 + du);
  if (!(q > 0.0)) return -1.0;
  const double h2 = v2 - q * q + du * v2;
  return sqrt(h2 > 0.0 ? h2 : 0.0) * (1.0 + 9.5367431640625e-7) + 1e-300;
}

// Range [lo, hi] of n / d over the box n in [n0 - hn, n0 + hn], d in [d0 - hd, d0 + hd]; false when d can be 0 there or
// anything is not finite.
inline bool rtrb_ratio_range(double n0, double hn, double d0, double hd, double& lo, double& hi) {
  const double dl = d0 - hd, dh = d0 + hd;
  if (!(dl > 0.0 || dh < 0.0)) return false;
  const double r[4] = {(n0 - hn) / dl, (n0 - hn) / dh, (n0 + hn) / dl, (n0 + hn) / dh};
  lo = fmin(fmin(r[0], r[1]), fmin(r[2], r[3]));
  hi = fmax(fmax(r[0], r[1]), fmax(r[2], r[3]));
  return isfinite(lo) && isfinite(hi);
}

// Pixels [i0, i1] of a W-pixel axis whose lens-table value 2 * (i / W - 0.5) * half lies in [lo, hi], dilated by one
// pixel (the host's and the device's rounding of the same direction).  Returns false when the set is empty.
inline bool rtrb_lens_pixels(double lo, double hi, double half, int W, int& i0, int& i1) {
  double a = W * (lo / (2.0 * half) + 0.5), b = W * (hi / (2.0 * half) + 0.5);
  if (half < 0.0) { const double s = a; a = b; b = s; }
  const double f0 = floor(a) - 1.0, f1 = ceil(b) + 1.0;
  if (f1 < 0.0 || f0 > W - 1.0) return false;
  i0 = f0 < 0.0 ? 0 : (int)f0;
  i1 = f1 > W - 1.0 ? W - 1 : (int)f1;
  return true;
}

// What the camera masks and the tile certificates know about the primary rays of a pinhole frame.  Pixel (x, y) looks
// along rf = front^ * D - left * sx(x) - up^ * sy(y) from the camera (camera.rb:130-134; the ray's FP64 direction is a
// positive or negative multiple of rf).  The FP32 u the kernel tests and the pixel's exact direction differ by the FP32
// normalisation (< 2^-20 rad) and by the FP64 ray's own rounding: rd = target - pos = rf (t - 1) with |t - 1| = |od| /
// |rf . front^| (od: distance of the focal plane), so |rd| >= |od| while the rounding of target is below 64 eps (|pos| +
// |focal| + 2 rf_max (1 + |od| / c_min)).  `dir` bounds that angle; in retina units it moves (sx, sy) by at most
// dir * rf_max^2 / c_min, which must stay under a quarter pixel for the one-pixel dilation.
struct RtrbPinhole {
  double f[3];    // front^
  double c_min;   // |rf . front^| >= c_min over the frame
  double rf_max;  // |rf| <= rf_max
  double od;      // (focal_point - pos) . front^ (signed)
  double dir;     // angle between the pixel's exact direction and the FP32 u of its ray
  bool ok;        // the bounds hold and the direction error is under a quarter pixel
};
inline RtrbPinhole rtrb_pinhole(const double pos[3], const double focal_point[3], const double left[3], const double up_n[3],
                                const double front[3], double D, double rw, double rh, int W, int H) {
  RtrbPinhole c;
  const double fl = sqrt(front[0] * front[0] + front[1] * front[1] + front[2] * front[2]);
  for (int i = 0; i < 3; ++i) c.f[i] = front[i] / fl;
  const double* f = c.f;
  const double lf = fabs(left[0] * f[0] + left[1] * f[1] + left[2] * f[2]);
  const double uf = fabs(up_n[0] * f[0] + up_n[1] * f[1] + up_n[2] * f[2]);
  const double ln = sqrt(left[0] * left[0] + left[1] * left[1] + left[2] * left[2]);
  const double un = sqrt(up_n[0] * up_n[0] + up_n[1] * up_n[1] + up_n[2] * up_n[2]);
  c.c_min = fabs(D) - fabs(rw) * lf - fabs(rh) * uf;
  c.rf_max = fabs(D) + fabs(rw) * ln + fabs(rh) * un;
  const double dp[3] = {focal_point[0] - pos[0], focal_point[1] - pos[1], focal_point[2] - pos[2]};
  c.od = dp[0] * f[0] + dp[1] * f[1] + dp[2] * f[2];
  const double od = fabs(c.od);
  const double pn = sqrt(pos[0] * pos[0] + pos[1] * pos[1] + pos[2] * pos[2]);
  const double fn = sqrt(focal_point[0] * focal_point[0] + focal_point[1] * focal_point[1] + focal_point[2] * focal_point[2]);
  c.dir = 9.5367431640625e-7 + 64.0 * 1.1102230246251565e-16 * (pn + fn + 2.0 * c.rf_max * (1.0 + od / c.c_min)) / od;
  const double shift = c.dir * c.rf_max * c.rf_max / c.c_min;
  const double pitch = fmin(2.0 * fabs(rw) / W, 2.0 * fabs(rh) / H);
  c.ok = isfinite(fl) && fl > 0.0 && isfinite(D) && c.c_min > 1e-9 * c.rf_max && isfinite(shift) && isfinite(pitch) &&
         shift < 0.25 * pitch && W > 0 && H > 0;
  return c;
}

// Camera masks of a pinhole frame: tx[c] / ty[r] = the spheres whose camera apex test can keep the primary ray of some
// pixel in super-tile column c / row r.  A point p = a left + b up^ + c front^ (relative to the camera) is on the line
// of (sx, sy) = (-D a / c, -D b / c) (rtrb_pinhole).  A ball of radius rho around V lies in the box of half-widths
// rho |row_i(B^-1)| in (a, b, c) (B = [left up^ front^]).
// Everything is set when the camera is degenerate or the FP64 ray direction cannot be bounded to well under a pixel.
inline void rtrb_camera_masks(const float* tab, int n, const double pos[3], const double focal_point[3], const double left[3],
                              const double up_n[3], const double front[3], double D, double rw, double rh, int W, int H,
                              uint32_t tx[RTRB_CAM_TX], uint32_t ty[RTRB_CAM_TY]) {
  const uint32_t all = n >= 32 ? 0xffffffffu : ((1u << n) - 1u);
  for (int i = 0; i < RTRB_CAM_TX; ++i) tx[i] = 0u;
  for (int i = 0; i < RTRB_CAM_TY; ++i) ty[i] = 0u;
  auto fill = [&](uint32_t m) {
    for (int i = 0; i < RTRB_CAM_TX; ++i) tx[i] |= m;
    for (int i = 0; i < RTRB_CAM_TY; ++i) ty[i] |= m;
  };
  const RtrbPinhole cam = rtrb_pinhole(pos, focal_point, left, up_n, front, D, rw, rh, W, H);
  const double* f = cam.f;
  // rows of B^-1: cross products of the other two columns over det
  double inv[3][3];
  const double c0[3] = {up_n[1] * f[2] - up_n[2] * f[1], up_n[2] * f[0] - up_n[0] * f[2], up_n[0] * f[1] - up_n[1] * f[0]};
  const double c1[3] = {f[1] * left[2] - f[2] * left[1], f[2] * left[0] - f[0] * left[2], f[0] * left[1] - f[1] * left[0]};
  const double c2[3] = {left[1] * up_n[2] - left[2] * up_n[1], left[2] * up_n[0] - left[0] * up_n[2],
                        left[0] * up_n[1] - left[1] * up_n[0]};
  const double det = left[0] * c0[0] + left[1] * c0[1] + left[2] * c0[2];
  for (int k = 0; k < 3; ++k) { inv[0][k] = c0[k] / det; inv[1][k] = c1[k] / det; inv[2][k] = c2[k] / det; }
  double rown[3];
  for (int i = 0; i < 3; ++i) rown[i] = sqrt(inv[i][0] * inv[i][0] + inv[i][1] * inv[i][1] + inv[i][2] * inv[i][2]);
  const bool ok = cam.ok && isfinite(det) && fabs(det) > 1e-6 && isfinite(rown[0] + rown[1] + rown[2]);
  if (!ok) { fill(all); return; }
  for (int k = 0; k < n; ++k) {
    const float* t = tab + 4 * (size_t)k;
    const double rho = rtrb_apex_reach(t);
    if (rho == 0.0) continue;
    if (rho < 0.0) { fill(1u << k); continue; }
    double cf[3];
    for (int i = 0; i < 3; ++i) cf[i] = inv[i][0] * (double)t[0] + inv[i][1] * (double)t[1] + inv[i][2] * (double)t[2];
    double xlo, xhi, ylo, yhi;
    // sx = -D a / c: the range of a / c scaled by -D
    if (!rtrb_ratio_range(cf[0], rho * rown[0], cf[2], rho * rown[2], xlo, xhi) ||
        !rtrb_ratio_range(cf[1], rho * rown[1], cf[2], rho * rown[2], ylo, yhi)) {
      fill(1u << k);
      continue;
    }
    const double sx0 = -D * xlo, sx1 = -D * xhi, sy0 = -D * ylo, sy1 = -D * yhi;
    int x0, x1, y0, y1;
    if (!rtrb_lens_pixels(fmin(sx0, sx1), fmax(sx0, sx1), rw, W, x0, x1)) continue;
    if (!rtrb_lens_pixels(fmin(sy0, sy1), fmax(sy0, sy1), rh, H, y0, y1)) continue;
    for (int c = x0 >> 5; c <= (x1 >> 5); ++c) tx[c < RTRB_CAM_TX ? c : RTRB_CAM_TX - 1] |= 1u << k;
    for (int r = y0 >> 5; r <= (y1 >> 5); ++r) ty[r < RTRB_CAM_TY ? r : RTRB_CAM_TY - 1] |= 1u << k;
  }
}

// Light masks of one light: m[a][0][i] / m[a][1][i] = the spheres whose light apex test can keep a line whose
// direction w has its largest component on axis a and ratio w[(a+1)%3] / w[a] (resp. w[(a+2)%3] / w[a]) in bin i of
// [-1, 1] (N = RTRB_LIGHT_BINS bins, bin = floor((s + 1) N / 2) clamped), dilated by one bin.  The box is the
// axis-aligned cube of half-size rho around V = C - L.  An axis along which the cube reaches both sides of the light
// (the light inside or near the sphere) gets every bin.
inline void rtrb_light_masks(const float* tab, int n, uint32_t m[3][2][RTRB_LIGHT_BINS]) {
  const int N = RTRB_LIGHT_BINS;
  for (int a = 0; a < 3; ++a)
    for (int j = 0; j < 2; ++j)
      for (int i = 0; i < N; ++i) m[a][j][i] = 0u;
  for (int k = 0; k < n; ++k) {
    const float* t = tab + 4 * (size_t)k;
    const double rho = rtrb_apex_reach(t);
    if (rho == 0.0) continue;
    for (int a = 0; a < 3; ++a) {
      for (int j = 0; j < 2; ++j) {
        const int b = (a + 1 + j) % 3;
        double lo = -1.0, hi = 1.0;
        if (rho > 0.0 && !rtrb_ratio_range(t[b], rho, t[a], rho, lo, hi)) { lo = -1.0; hi = 1.0; }
        else if (rho < 0.0) { lo = -1.0; hi = 1.0; }
        const double f0 = floor((lo + 1.0) * (N / 2)) - 1.0, f1 = floor((hi + 1.0) * (N / 2)) + 1.0;
        if (f1 < 0.0 || f0 > N - 1.0) continue;
        const int i0 = f0 < 0.0 ? 0 : (int)f0, i1 = f1 > N - 1.0 ? N - 1 : (int)f1;
        for (int i = i0; i <= i1; ++i) m[a][j][i] |= 1u << k;
      }
    }
  }
}

// FP32 view of a light for the highlight filter (DevLightF, rtrb_types.h).
struct RtrbLightF {
  float px, py, pz;
  float pmax;       // |position|_inf
  float cos2_thr;   // cos^2(high_light_angle), valid when mode == 1
  int32_t mode;     // 1: threshold in (0, 90 deg) -> FP32 filter usable; 0: always take the exact path
};

// Tile certificates of a pinhole frame: rows[c] = {s0, s1, h0, h1} for super-tile column c < RTRB_CAM_TX.  Every primary
// ray of the super-tiles (c, r), r in [s0, s1), is rejected by classify_plane for every plane as certainly behind its
// origin (kind 0), and every primary ray of the rows [s0, s1) and [h0, h1) fails highlight_match_fast for every light
// at its FP32 test (c2 + tol < cos2_thr): the kernels reach neither the exact plane test nor the exact highlight
// expression there, so skipping those filters cannot change a frame, a hit id or a counter.  A column's certified rows
// need not be contiguous (the light's image splits them); each interval is its longest run.  All zero = nothing.
//
// Bounds, per tile dilated by one pixel: the device's FP32 u is within dir + 2^-17 of the pixel's exact unit direction
// (rtrb_pinhole; the 2^-17 covers |u| = 1 +- 2^-18).  With rf = D f - sx left - sy up (f = front^), any n . rf is linear
// and separable in (sx, sy), so its range over a tile is the sum of a column term and a row term; |rf| <= rf_max and
// |rf|^2 >= lam (D^2 + sx^2 + sy^2), lam a Gershgorin bound on the Gram matrix of (f, left, up).  The FP32 evaluations
// of den, num, t, e_t (classify_plane) and of ret, a2, c2, rho, tol (highlight_match_fast) are bounded with margins
// well above their documented error: a few ulp per fmaf chain, rcp.approx / rsqrt.approx within 2^-21 relative.
// `o` is the FP32 ray origin (the camera position rounded to float); pl = k_cull_pl (8 floats per plane).
inline void rtrb_tile_rows(const float* pl, int n_pl, const RtrbLightF* lf, int n_lights, const double pos[3],
                           const double focal_point[3], const double left[3], const double up_n[3], const double front[3],
                           double D, double rw, double rh, int W, int H, uint8_t rows[RTRB_CAM_TX][4]) {
  for (int c = 0; c < RTRB_CAM_TX; ++c) rows[c][0] = rows[c][1] = rows[c][2] = rows[c][3] = 0;
  const RtrbPinhole cam = rtrb_pinhole(pos, focal_point, left, up_n, front, D, rw, rh, W, H);
  const double eps = 5.9604644775390625e-8;  // 2^-24
  // the ray runs along +rf when D > 0 and the focal plane is in front (rd = rf (t - 1), t - 1 = od / (rf . f))
  if (!cam.ok || !(D > 0.0) || !(cam.od > 0.0) || n_pl > 8 || n_lights > 2) return;
  const double* f = cam.f;
  const double dl = cam.dir + 7.62939453125e-6;  // |u - u_exact|
  const float o32[3] = {(float)pos[0], (float)pos[1], (float)pos[2]};
  const double o[3] = {o32[0], o32[1], o32[2]};
  const double mo = fmax(fabs(o[0]), fmax(fabs(o[1]), fabs(o[2])));
  auto dot = [](const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; };
  // a . rf over the tile = a.f D + X(sx) + Y(sy): range of the column / row terms
  const int nc = (W + 31) / 32 < RTRB_CAM_TX ? (W + 31) / 32 : RTRB_CAM_TX;
  const int nr = (H + 31) / 32 < 255 ? (H + 31) / 32 : 255;
  auto sx = [&](int x) { return 2.0 * ((double)x / W - 0.5) * rw; };
  auto sy = [&](int y) { return 2.0 * ((double)y / H - 0.5) * rh; };
  auto range = [](double k, double s0, double s1, double& lo, double& hi) {  // of -k s over [s0, s1] (either order)
    const double a = -k * s0, b = -k * s1;
    lo = a < b ? a : b; hi = a < b ? b : a;
  };
  auto sq_min = [](double s0, double s1) { return (s0 <= 0.0) == (s1 <= 0.0) ? (s0 * s0 < s1 * s1 ? s0 * s0 : s1 * s1) : 0.0; };
  // ---- planes: certainly behind the origin when s g >= g_th over the tile (s = -sign(num), g = n . rf) ----
  double p_sgn[8], p_c[8], p_th[8], p_kl[8], p_ku[8];
  bool planes_ok = true;
  for (int k = 0; k < n_pl && planes_ok; ++k) {
    const float* a = pl + 8 * k;
    const double n[3] = {a[0], a[1], a[2]}, aw = a[3], pw = a[7];
    const double num = ((double)a[4] - o[0]) * n[0] + ((double)a[5] - o[1]) * n[1] + ((double)a[6] - o[2]) * n[2];
    const double e_num = 16.0 * eps * aw * (pw + mo) * 1.0001, e_den = 16.0 * eps * aw;
    const double n_lo = fabs(num) - 0.5 * e_num;  // |num| on the device (its error is below 5/16 e_num)
    const double q = 0.999 / 1.1002 - e_num / n_lo;
    // |den| > 16 e_den (else kind 1), and t + e_t < 0 once 1.1002 (e_num / |num| + e_den / |den|) < 0.999
    const double den_req = fmax(256.0 * eps * aw * 1.0001, e_den / q);
    const double nn = sqrt(dot(n, n));
    const double m_n = nn * dl + 8.0 * eps * aw * (1.0 + dl);  // |den - n . u_exact|
    p_sgn[k] = num > 0.0 ? -1.0 : 1.0;
    p_c[k] = p_sgn[k] * dot(n, f) * D;
    p_th[k] = (den_req + m_n) * cam.rf_max * (1.0 + 1e-9) + 1e-300;
    p_kl[k] = p_sgn[k] * dot(n, left);
    p_ku[k] = p_sgn[k] * dot(n, up_n);
    planes_ok = aw > 0.0 && n_lo > 0.0 && q > 0.0 && isfinite(num) && isfinite(p_th[k]) && isfinite(p_c[k]) &&
                isfinite(p_kl[k]) && isfinite(p_ku[k]);
  }
  // ---- lights: |a . u| < cthr |a| with margin, i.e. h^2 < K (D^2 + sx^2 + sy^2), h = a . rf ----
  double g[3][3];
  const double* B[3] = {f, left, up_n};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) g[i][j] = dot(B[i], B[j]);
  double lam = 1e300;
  for (int i = 0; i < 3; ++i) lam = fmin(lam, g[i][i] - fabs(g[i][(i + 1) % 3]) - fabs(g[i][(i + 2) % 3]));
  lam *= 1.0 - 1e-9;
  double l_c[2], l_kl[2], l_ku[2], l_K[2];
  bool lights_ok = lam > 0.0;
  for (int l = 0; l < n_lights && lights_ok; ++l) {
    const RtrbLightF& F = lf[l];
    const double a[3] = {(double)F.px - o[0], (double)F.py - o[1], (double)F.pz - o[2]};
    const double an = sqrt(dot(a, a)), a1 = fabs(a[0]) + fabs(a[1]) + fabs(a[2]);
    const double ea = 8.0 * eps * ((double)F.pmax + mo) * 1.0001;
    const double rho = 8.0 * (ea / (an * (1.0 - 1e-5)) + 8.0 * eps) * 1.0001;
    const double tol = (rho * rho + 2.0 * rho) * 1.0001;
    // c2 <= (ret / |a|)^2 (1 + 2^-18); the FP32 sum c2 + tol must not round up to cos2_thr
    const double c2_room = ((double)F.cos2_thr * (1.0 - 1e-6) - tol) / (1.0 + 3.814697265625e-6);
    const double m_a = an * (dl + 2.0 * eps) + 8.0 * eps * a1 * (1.0 + dl);           // |ret - a . u_exact|
    const double room = c2_room > 0.0 ? sqrt(c2_room) * an - m_a : -1.0;
    l_c[l] = dot(a, f) * D;
    l_kl[l] = dot(a, left);
    l_ku[l] = dot(a, up_n);
    l_K[l] = room * room * lam * (1.0 - 1e-9);
    lights_ok = F.mode == 1 && rho < 0.25 && room > 0.0 && isfinite(l_K[l]) && isfinite(l_c[l]) && isfinite(l_kl[l]) &&
                isfinite(l_ku[l]) && an > 0.0;
  }
  if (!lights_ok) return;  // every certificate needs the highlight one
  // per row: the row terms (tile rows r, dilated by one pixel)
  double ry_lo[8][255], ry_hi[2][255], ry_hl[2][255], ry_s2[255];
  for (int r = 0; r < nr; ++r) {
    const double s0 = sy(32 * r - 1), s1 = sy(32 * r + 32);
    ry_s2[r] = sq_min(s0, s1);
    double lo, hi;
    for (int k = 0; k < n_pl; ++k) { range(p_ku[k], s0, s1, lo, hi); ry_lo[k][r] = lo; }
    for (int l = 0; l < n_lights; ++l) { range(l_ku[l], s0, s1, lo, hi); ry_hl[l][r] = lo; ry_hi[l][r] = hi; }
  }
  for (int c = 0; c < nc; ++c) {
    const double s0 = sx(32 * c - 1), s1 = sx(32 * c + 32);
    const double D2 = D * D + sq_min(s0, s1);
    double cx_lo[8], hx_lo[2], hx_hi[2], lo, hi;
    for (int k = 0; k < n_pl; ++k) { range(p_kl[k], s0, s1, lo, hi); cx_lo[k] = p_c[k] + lo; }
    for (int l = 0; l < n_lights; ++l) { range(l_kl[l], s0, s1, lo, hi); hx_lo[l] = l_c[l] + lo; hx_hi[l] = l_c[l] + hi; }
    // branch-free passes over the column's rows (they vectorise), then the longest run of each kind
    uint8_t hl[256], sky[256];
    for (int r = 0; r < nr; ++r) hl[r] = 1;
    for (int l = 0; l < n_lights; ++l)
      for (int r = 0; r < nr; ++r) {
        const double h0 = -(hx_lo[l] + ry_hl[l][r]), h1 = hx_hi[l] + ry_hi[l][r], h = h0 > h1 ? h0 : h1;
        hl[r] &= (uint8_t)(h * h < l_K[l] * (D2 + ry_s2[r]));
      }
    for (int r = 0; r < nr; ++r) sky[r] = hl[r] & (uint8_t)planes_ok;
    for (int k = 0; k < n_pl; ++k)
      for (int r = 0; r < nr; ++r) sky[r] &= (uint8_t)(cx_lo[k] + ry_lo[k][r] >= p_th[k]);
    hl[nr] = sky[nr] = 0;
    int run[2] = {0, 0}, best0[2] = {0, 0}, best1[2] = {0, 0};
    for (int r = 0; r <= nr; ++r) {
      const uint8_t in[2] = {sky[r], hl[r]};
      for (int i = 0; i < 2; ++i) {
        if (in[i]) { run[i]++; continue; }
        if (run[i] > best1[i] - best0[i]) { best0[i] = r - run[i]; best1[i] = r; }
        run[i] = 0;
      }
    }
    for (int i = 0; i < 2; ++i) { rows[c][2 * i] = (uint8_t)best0[i]; rows[c][2 * i + 1] = (uint8_t)best1[i]; }
  }
}

// Longest run of set flags in f[0, n): [b0, b1), empty = [0, 0).
inline void rtrb_longest_run(const uint8_t* f, int n, int& b0, int& b1) {
  b0 = b1 = 0;
  int run = 0;
  for (int r = 0; r <= n; ++r) {
    if (r < n && f[r]) { run++; continue; }
    if (run > b1 - b0) { b0 = r - run; b1 = r; }
    run = 0;
  }
}

// Sky-fill layout of a whole frame of stx x sty super-tiles (sty <= RTRB_CAM_TY): run[r] = {a, b}, the longest run of
// columns c < RTRB_CAM_TX of super-tile row r whose tiles lie in their column's sky rows [tile_rows[c][0],
// tile_rows[c][1]) and have an empty candidate mask cam_tx[c] & cam_ty[r], so every tile of it is one the kernels store
// through their sky branch; before[r] = the tiles outside the runs (the traced tiles) of the rows < r.  The kernels trace
// those in row-major order, traced tile t of row r being column t - before[r] left of a and t - before[r] + b - a from a
// on, and store the runs' tiles from separate CTAs (trace_pre_body).  Returns the number of tiles in the runs; 0 (and no
// runs) when the frame does not fit the tables.
inline int rtrb_sky_fill(const uint32_t cam_tx[RTRB_CAM_TX], const uint32_t cam_ty[RTRB_CAM_TY],
                         const uint8_t tile_rows[RTRB_CAM_TX][4], int stx, int sty, uint8_t run[RTRB_CAM_TY][2],
                         uint16_t before[RTRB_CAM_TY]) {
  for (int r = 0; r < RTRB_CAM_TY; ++r) run[r][0] = run[r][1] = 0, before[r] = 0;
  if (stx < 1 || sty < 1 || sty > RTRB_CAM_TY || stx * sty > 0xffff) return 0;
  const int nc = stx < RTRB_CAM_TX ? stx : RTRB_CAM_TX;
  int r0 = 255, r1 = 0;  // rows that hold sky tiles at all
  for (int c = 0; c < nc; ++c) {
    if (tile_rows[c][0] >= tile_rows[c][1]) continue;
    r0 = tile_rows[c][0] < r0 ? tile_rows[c][0] : r0;
    r1 = tile_rows[c][1] > r1 ? tile_rows[c][1] : r1;
  }
  int n_sky = 0;
  for (int r = 0; r < sty; ++r) {
    before[r] = (uint16_t)(r * stx - n_sky);
    int a = 0, b = 0, len = 0;  // the first longest run
    for (int c = 0; c < (r >= r0 && r < r1 ? nc : 0); ++c) {
      len = r >= tile_rows[c][0] && r < tile_rows[c][1] && (cam_tx[c] & cam_ty[r]) == 0u ? len + 1 : 0;
      if (len > b - a) { a = c + 1 - len; b = c + 1; }
    }
    run[r][0] = (uint8_t)a; run[r][1] = (uint8_t)b;
    n_sky += b - a;
  }
  if (n_sky == 0) for (int r = 0; r < sty; ++r) run[r][0] = run[r][1] = 0;
  return n_sky;
}

// Ground certificates of a pinhole frame whose scene has exactly one plane: rows[c] = {g0, g1} for super-tile column
// c < RTRB_CAM_TX, the longest run of rows in which, for every primary ray of the tile (dilated by one pixel),
// classify_plane does not return kind 0 for the plane and its lo <= max_distance_f, inside tile_rows' no-highlight rows.
// A ground tile whose camera candidate mask is empty therefore sends exactly the plane to the exact test, and nothing
// else.  All zero = nothing.
// Bounds: den = n . u is within m_n of n . rf / |rf| (rtrb_tile_rows), so s (n . rf) >= m_n rf_max, s = sign(num), gives
// den the sign of num (or |den| below the grazing cut, kind 1): t = num rcp(den) >= 0, never kind 0; and lo <= t <=
// (|num| + e_num / 2) (1 + 1e-5) / (s g_min / rf_max - m_n).
inline void rtrb_ground_rows(const float* pl, int n_pl, float max_distance_f, const double pos[3], const double focal_point[3],
                             const double left[3], const double up_n[3], const double front[3], double D, double rw,
                             double rh, int W, int H, const uint8_t tile_rows[RTRB_CAM_TX][4],
                             uint8_t rows[RTRB_CAM_TX][2]) {
  for (int c = 0; c < RTRB_CAM_TX; ++c) rows[c][0] = rows[c][1] = 0;
  const RtrbPinhole cam = rtrb_pinhole(pos, focal_point, left, up_n, front, D, rw, rh, W, H);
  const double eps = 5.9604644775390625e-8;  // 2^-24
  if (!cam.ok || !(D > 0.0) || !(cam.od > 0.0) || n_pl != 1) return;
  auto dot = [](const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; };
  const double* f = cam.f;
  const double dl = cam.dir + 7.62939453125e-6;
  const double o[3] = {(float)pos[0], (float)pos[1], (float)pos[2]};
  const double mo = fmax(fabs(o[0]), fmax(fabs(o[1]), fabs(o[2])));
  const double n[3] = {pl[0], pl[1], pl[2]}, aw = pl[3], pw = pl[7];
  const double num = ((double)pl[4] - o[0]) * n[0] + ((double)pl[5] - o[1]) * n[1] + ((double)pl[6] - o[2]) * n[2];
  const double e_num = 16.0 * eps * aw * (pw + mo) * 1.0001;
  const double s = num > 0.0 ? 1.0 : -1.0;
  const double m_n = sqrt(dot(n, n)) * dl + 8.0 * eps * aw * (1.0 + dl);
  const double g_th = m_n * cam.rf_max * (1.0 + 1e-9) + 1e-300;
  if (!(aw > 0.0 && fabs(num) - 0.5 * e_num > 0.0 && isfinite(num) && isfinite(g_th))) return;
  const double kc = s * dot(n, f) * D, kl = s * dot(n, left), ku = s * dot(n, up_n);
  const int nc = (W + 31) / 32 < RTRB_CAM_TX ? (W + 31) / 32 : RTRB_CAM_TX;
  const int nr = (H + 31) / 32 < 255 ? (H + 31) / 32 : 255;
  auto sx = [&](int x) { return 2.0 * ((double)x / W - 0.5) * rw; };
  auto sy = [&](int y) { return 2.0 * ((double)y / H - 0.5) * rh; };
  double ry_lo[255];
  for (int r = 0; r < nr; ++r) ry_lo[r] = fmin(-ku * sy(32 * r - 1), -ku * sy(32 * r + 32));
  for (int c = 0; c < nc; ++c) {
    const double cx_lo = kc + fmin(-kl * sx(32 * c - 1), -kl * sx(32 * c + 32));
    uint8_t g[256];
    for (int r = 0; r < nr; ++r) {
      const double sg = cx_lo + ry_lo[r];  // min of s (n . rf) over the tile
      const double t_max = (fabs(num) + 0.5 * e_num) * (1.0 + 1e-5) / (sg / cam.rf_max - m_n);
      g[r] = (uint8_t)(sg >= g_th && r >= tile_rows[c][2] && r < tile_rows[c][3] &&
                       (max_distance_f == INFINITY || t_max <= (double)max_distance_f));
    }
    int g0, g1;
    rtrb_longest_run(g, nr, g0, g1);
    rows[c][0] = (uint8_t)g0; rows[c][1] = (uint8_t)g1;
  }
}
