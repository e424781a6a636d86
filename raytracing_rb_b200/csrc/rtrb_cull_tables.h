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

// Camera masks of a pinhole frame: tx[c] / ty[r] = the spheres whose camera apex test can keep the primary ray of some
// pixel in super-tile column c / row r.  Pixel (x, y) looks along rf = front^ * D - left * sx(x) - up^ * sy(y) from the
// camera (camera.rb:130-134; the ray's FP64 direction is a positive or negative multiple of rf), so a point
// p = a left + b up^ + c front^ (relative to the camera) is on the line of (sx, sy) = (-D a / c, -D b / c).
// A ball of radius rho around V lies in the box of half-widths rho |row_i(B^-1)| in (a, b, c) (B = [left up^ front^]).
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
  const double fl = sqrt(front[0] * front[0] + front[1] * front[1] + front[2] * front[2]);
  const double f[3] = {front[0] / fl, front[1] / fl, front[2] / fl};
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
  // |rf| <= rf_max, |rf . front^| >= c_min over the frame
  const double lf = fabs(left[0] * f[0] + left[1] * f[1] + left[2] * f[2]);
  const double uf = fabs(up_n[0] * f[0] + up_n[1] * f[1] + up_n[2] * f[2]);
  const double ln = sqrt(left[0] * left[0] + left[1] * left[1] + left[2] * left[2]);
  const double un = sqrt(up_n[0] * up_n[0] + up_n[1] * up_n[1] + up_n[2] * up_n[2]);
  const double c_min = fabs(D) - fabs(rw) * lf - fabs(rh) * uf;
  const double rf_max = fabs(D) + fabs(rw) * ln + fabs(rh) * un;
  // The FP32 u the kernel tests and the pixel's exact direction differ by the FP32 normalisation (< 2^-20 rad) and by
  // the FP64 ray's own rounding: rd = target - pos = rf (t - 1) with |t - 1| = |od| / |rf . front^| (od: distance of
  // the focal plane), so |rd| >= |od| while the rounding of target is below 64 eps (|pos| + |focal| + 2 rf_max (1 +
  // |od| / c_min)).  In retina units a direction error moves (sx, sy) by at most dir * rf_max^2 / c_min, which must
  // stay under a quarter pixel for the one-pixel dilation.
  const double dp[3] = {focal_point[0] - pos[0], focal_point[1] - pos[1], focal_point[2] - pos[2]};
  const double od = fabs(dp[0] * f[0] + dp[1] * f[1] + dp[2] * f[2]);
  const double pn = sqrt(pos[0] * pos[0] + pos[1] * pos[1] + pos[2] * pos[2]);
  const double fn = sqrt(focal_point[0] * focal_point[0] + focal_point[1] * focal_point[1] + focal_point[2] * focal_point[2]);
  const double dir = 9.5367431640625e-7 + 64.0 * 1.1102230246251565e-16 * (pn + fn + 2.0 * rf_max * (1.0 + od / c_min)) / od;
  const double shift = dir * rf_max * rf_max / c_min;
  const double pitch = fmin(2.0 * fabs(rw) / W, 2.0 * fabs(rh) / H);
  bool ok = isfinite(det) && fabs(det) > 1e-6 && isfinite(D) && c_min > 1e-9 * rf_max && isfinite(shift) && isfinite(pitch) &&
            shift < 0.25 * pitch && W > 0 && H > 0 && isfinite(rown[0] + rown[1] + rown[2]);
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
