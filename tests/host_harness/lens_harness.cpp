// TEST-ONLY host harness: the __host__ __device__ model functions of
// robot_camera_calibration_b200/csrc/model.cuh for either lens, compiled with g++ so that their
// arithmetic can be checked against the complex-step oracle without a GPU.  Never loaded by the
// product package.
#include "../../robot_camera_calibration_b200/csrc/model.cuh"
using namespace rcc;

template <bool RIG, Lens L>
static void run(const double* view6, const double* marker6, const double* ext6, const double* sh9, double size,
                const double* pix8, double* r8, double* jv, double* jm, double* js, double* jx, double* depth4) {
  double vx[POSEX], mx[POSEX], xx[POSEX];
  expand_pose(view6, vx);
  expand_marker_pose(marker6, mx);
  if (RIG) expand_pose(ext6, xx);
  BlockGeom<RIG> g;
  block_geometry<RIG>(vx, mx, RIG ? xx : nullptr, g);
  for (int k = 0; k < 4; ++k) {
    double ox, oy;
    corner_xy(k, 0.5 * size, ox, oy);
    CornerRows<RIG> c;
    eval_corner<RIG, true, L>(g, sh9, ox, oy, pix8[2 * k], pix8[2 * k + 1], c);
    for (int i = 0; i < 2; ++i) {
      int row = 2 * k + i;
      r8[row] = c.r[i];
      for (int j = 0; j < 6; ++j) { jv[row * 6 + j] = c.jv[i][j]; jm[row * 6 + j] = c.jm[i][j]; }
      for (int j = 0; j < 9; ++j) js[row * 9 + j] = c.js[i][j];
      if (RIG) for (int j = 0; j < 6; ++j) jx[row * 6 + j] = c.jx[i][j];
    }
    depth4[k] = c.depth;
  }
}

extern "C" void model_eval_block_lens(int lens, int rig, const double* view6, const double* marker6,
                                      const double* ext6, const double* sh9, double size, const double* pix8,
                                      double* r8, double* jv, double* jm, double* js, double* jx, double* depth4) {
  if (lens == LENS_EQUIDISTANT) {
    if (rig) run<true, LENS_EQUIDISTANT>(view6, marker6, ext6, sh9, size, pix8, r8, jv, jm, js, jx, depth4);
    else run<false, LENS_EQUIDISTANT>(view6, marker6, ext6, sh9, size, pix8, r8, jv, jm, js, jx, depth4);
  } else {
    if (rig) run<true, LENS_RADTAN>(view6, marker6, ext6, sh9, size, pix8, r8, jv, jm, js, jx, depth4);
    else run<false, LENS_RADTAN>(view6, marker6, ext6, sh9, size, pix8, r8, jv, jm, js, jx, depth4);
  }
}
