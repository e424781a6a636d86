// TEST INFRASTRUCTURE: the host tile-certificate builder of raytracing_rb_b200/csrc/rtrb_cull_tables.h behind a C ABI,
// compiled with g++ by tests/test_tile_rows_host.py.
#include <chrono>

#include "../raytracing_rb_b200/csrc/rtrb_cull_tables.h"

extern "C" {

int rtrb_test_tile_cols() { return RTRB_CAM_TX; }

// lights: n_lights records of (px, py, pz, pmax, cos2_thr) floats; modes: their RtrbLightF::mode
void rtrb_test_tile_rows(const float* pl, int n_pl, const float* lights, const int* modes, int n_lights, const double* pos,
                         const double* focal_point, const double* left, const double* up_n, const double* front, double D,
                         double rw, double rh, int W, int H, uint8_t* rows) {
  RtrbLightF lf[2] = {};
  for (int l = 0; l < n_lights && l < 2; ++l) {
    lf[l].px = lights[5 * l]; lf[l].py = lights[5 * l + 1]; lf[l].pz = lights[5 * l + 2];
    lf[l].pmax = lights[5 * l + 3]; lf[l].cos2_thr = lights[5 * l + 4]; lf[l].mode = modes[l];
  }
  rtrb_tile_rows(pl, n_pl, lf, n_lights, pos, focal_point, left, up_n, front, D, rw, rh, W, H, (uint8_t(*)[4])rows);
}

// Host time of one rtrb_tile_rows call, in seconds, averaged over `iters` calls with the arguments above.
double rtrb_test_tile_rows_seconds(int iters, const float* pl, int n_pl, const float* lights, const int* modes, int n_lights,
                                   const double* pos, const double* focal_point, const double* left, const double* up_n,
                                   const double* front, double D, double rw, double rh, int W, int H, uint8_t* rows) {
  const auto t0 = std::chrono::steady_clock::now();
  for (int i = 0; i < iters; ++i)
    rtrb_test_tile_rows(pl, n_pl, lights, modes, n_lights, pos, focal_point, left, up_n, front, D, rw, rh, W, H, rows);
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() / iters;
}

}
