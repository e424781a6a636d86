// TEST INFRASTRUCTURE: the host sky-fill layout builder of raytracing_rb_b200/csrc/rtrb_cull_tables.h behind a C ABI,
// compiled with g++ by tests/test_sky_fill_host.py.
#include <chrono>

#include "../raytracing_rb_b200/csrc/rtrb_cull_tables.h"

extern "C" {

int rtrb_test_sky_fill(const uint32_t* cam_tx, const uint32_t* cam_ty, const uint8_t* tile_rows, int stx, int sty,
                       uint8_t* run, uint16_t* before) {
  return rtrb_sky_fill(cam_tx, cam_ty, (const uint8_t(*)[4])tile_rows, stx, sty, (uint8_t(*)[2])run, before);
}

// Host time of one rtrb_sky_fill call, in seconds, averaged over `iters` calls with the arguments above.
double rtrb_test_sky_fill_seconds(int iters, const uint32_t* cam_tx, const uint32_t* cam_ty, const uint8_t* tile_rows,
                                  int stx, int sty, uint8_t* run, uint16_t* before) {
  int sink = 0;
  const auto t0 = std::chrono::steady_clock::now();
  for (int i = 0; i < iters; ++i) sink += rtrb_test_sky_fill(cam_tx, cam_ty, tile_rows, stx, sty, run, before);
  const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() / iters;
  return sink < 0 ? -s : s;
}

}
