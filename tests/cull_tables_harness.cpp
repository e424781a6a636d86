// TEST INFRASTRUCTURE: the host mask builders of raytracing_rb_b200/csrc/rtrb_cull_tables.h behind a C ABI, compiled
// with g++ by tests/test_cull_tables_host.py.
#include "../raytracing_rb_b200/csrc/rtrb_cull_tables.h"

extern "C" {

int rtrb_test_cull_dims(int* out) {
  out[0] = RTRB_CAM_TX; out[1] = RTRB_CAM_TY; out[2] = RTRB_LIGHT_BINS;
  return 3;
}

void rtrb_test_camera_masks(const float* tab, int n, const double* pos, const double* focal_point, const double* left,
                            const double* up_n, const double* front, double D, double rw, double rh, int W, int H,
                            uint32_t* tx, uint32_t* ty) {
  rtrb_camera_masks(tab, n, pos, focal_point, left, up_n, front, D, rw, rh, W, H, tx, ty);
}

void rtrb_test_light_masks(const float* tab, int n, uint32_t* m) {
  rtrb_light_masks(tab, n, (uint32_t(*)[2][RTRB_LIGHT_BINS])m);
}

}
