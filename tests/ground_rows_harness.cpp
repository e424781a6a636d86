// TEST INFRASTRUCTURE: the host ground-certificate builder of raytracing_rb_b200/csrc/rtrb_cull_tables.h behind a C ABI,
// compiled with g++ by tests/test_ground_rows_host.py.  Tile rows first, as bake_frame does.
#include <chrono>

#include "../raytracing_rb_b200/csrc/rtrb_cull_tables.h"

extern "C" {

// light: (px, py, pz, pmax, cos2_thr) floats and its mode (n_lights 0 or 1)
void rtrb_test_ground_rows(const float* pl, int n_pl, const float* light, int mode, int n_lights, float max_distance_f,
                           const double* pos, const double* focal_point, const double* left, const double* up_n,
                           const double* front, double D, double rw, double rh, int W, int H, uint8_t* tile_rows,
                           uint8_t* rows) {
  RtrbLightF lf[1] = {};
  lf[0].px = light[0]; lf[0].py = light[1]; lf[0].pz = light[2]; lf[0].pmax = light[3]; lf[0].cos2_thr = light[4];
  lf[0].mode = mode;
  rtrb_tile_rows(pl, n_pl, lf, n_lights, pos, focal_point, left, up_n, front, D, rw, rh, W, H, (uint8_t(*)[4])tile_rows);
  rtrb_ground_rows(pl, n_pl, max_distance_f, pos, focal_point, left, up_n, front, D, rw, rh, W, H,
                   (const uint8_t(*)[4])tile_rows, (uint8_t(*)[2])rows);
}

// Host time of one rtrb_ground_rows call (tile rows included), in seconds, averaged over `iters` calls.
double rtrb_test_ground_rows_seconds(int iters, const float* pl, int n_pl, const float* light, int mode, int n_lights,
                                     float max_distance_f, const double* pos, const double* focal_point, const double* left,
                                     const double* up_n, const double* front, double D, double rw, double rh, int W, int H,
                                     uint8_t* tile_rows, uint8_t* rows) {
  const auto t0 = std::chrono::steady_clock::now();
  for (int i = 0; i < iters; ++i)
    rtrb_test_ground_rows(pl, n_pl, light, mode, n_lights, max_distance_f, pos, focal_point, left, up_n, front, D, rw, rh,
                          W, H, tile_rows, rows);
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() / iters;
}

}
