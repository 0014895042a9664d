// Batched PnP initialiser -- the job cv::solvePnP(obj_pts, img_pts, K, dist, rvec,
// tvec, false, CV_ITERATIVE) does once per tag per frame at
// /root/reference/real_preprocessing/src/camera_pose.cpp:163 (tagTcam, :132-173):
// minimise the reprojection error of the four tag corners over cam_T_tag (6 dof).
//
// One thread per tag.  Like OpenCV's iterative solver for planar targets it
// starts from the homography between the tag plane and the undistorted
// normalised image points and refines with Levenberg-Marquardt; the cost and
// its analytic Jacobian are the same model.cuh functions the bundle adjustment
// uses (view = identity, marker = cam_T_tag), for either lens.
//
// pnp_target_kernel does the same for rigid targets, the job cv::calibrateCamera's per-view solvePnP does for a
// board: one warp per (frame, target) problem over all corners of the target's detected tags.
#include "common.cuh"
#include "kernels.h"
#include "model.cuh"

namespace rcc {

// solve the n x n system A x = b in place (partial pivoting); returns false if singular
template <int N>
__device__ bool solve_dense(double (&A)[N][N], double (&b)[N]) {
  for (int c = 0; c < N; ++c) {
    int piv = c;
    double best = fabs(A[c][c]);
    for (int r = c + 1; r < N; ++r)
      if (fabs(A[r][c]) > best) { best = fabs(A[r][c]); piv = r; }
    if (!(best > 1e-300)) return false;
    if (piv != c) {
      for (int k = 0; k < N; ++k) { const double t = A[c][k]; A[c][k] = A[piv][k]; A[piv][k] = t; }
      const double t = b[c]; b[c] = b[piv]; b[piv] = t;
    }
    const double inv = 1.0 / A[c][c];
    for (int r = c + 1; r < N; ++r) {
      const double f = A[r][c] * inv;
      if (f != 0.0) {
        for (int k = c; k < N; ++k) A[r][k] -= f * A[c][k];
        b[r] -= f * b[c];
      }
    }
  }
  for (int r = N - 1; r >= 0; --r) {
    double s = b[r];
    for (int k = r + 1; k < N; ++k) s -= A[r][k] * b[k];
    b[r] = s / A[r][r];
  }
  return true;
}

// rotation matrix (row-major) -> Rodrigues vector
__device__ void rot_to_rvec(const double* R, double* r) {
  const double wx = 0.5 * (R[7] - R[5]), wy = 0.5 * (R[2] - R[6]), wz = 0.5 * (R[3] - R[1]);
  const double s = sqrt(wx * wx + wy * wy + wz * wz);
  const double c = 0.5 * (R[0] + R[4] + R[8] - 1.0);
  const double t = atan2(s, c);
  if (s > 1e-9) {
    const double k = t / s;
    r[0] = wx * k; r[1] = wy * k; r[2] = wz * k;
  } else if (c > 0.0) {
    r[0] = wx; r[1] = wy; r[2] = wz;
  } else {
    // angle ~ pi: axis from the diagonal of (R + I)/2
    const double xx = 0.5 * (R[0] + 1.0), yy = 0.5 * (R[4] + 1.0), zz = 0.5 * (R[8] + 1.0);
    double ax = sqrt(fmax(xx, 0.0)), ay = sqrt(fmax(yy, 0.0)), az = sqrt(fmax(zz, 0.0));
    if (ax >= ay && ax >= az) { ay = copysign(ay, R[1] + R[3]); az = copysign(az, R[2] + R[6]); }
    else if (ay >= az) { ax = copysign(ax, R[1] + R[3]); az = copysign(az, R[5] + R[7]); }
    else { ax = copysign(ax, R[2] + R[6]); ay = copysign(ay, R[5] + R[7]); }
    r[0] = ax * t; r[1] = ay * t; r[2] = az * t;
  }
}

// pixel (u, v) -> undistorted normalised image point (x, y) under lens L: the start of both PnP kernels
template <Lens L>
__device__ __forceinline__ void undistort_corner(const double* sh, double u, double v, double& xo, double& yo) {
  const double x0 = (u - sh[2]) / sh[0], y0 = (v - sh[3]) / sh[1];
  double x = x0, y = y0;
  if (L == LENS_RADTAN) {
    // fixed-point iteration, like cv::undistortPoints
    for (int it = 0; it < 20; ++it) {
      const double r2 = x * x + y * y;
      const double rad = 1.0 + r2 * (sh[4] + r2 * (sh[5] + r2 * sh[8]));
      const double dx = 2.0 * sh[6] * x * y + sh[7] * (r2 + 2.0 * x * x);
      const double dy = sh[6] * (r2 + 2.0 * y * y) + 2.0 * sh[7] * x * y;
      x = (x0 - dx) / rad;
      y = (y0 - dy) / rad;
    }
  } else {
    // th_d = |(x0, y0)|: solve th (1 + k1 th^2 + .. + k4 th^8) = th_d for th by Newton's method (as
    // cv::fisheye::undistortPoints does), then the pinhole point tan(th) along the distorted direction
    const double thd = sqrt(x0 * x0 + y0 * y0);
    double th = thd;
    for (int it = 0; it < 20; ++it) {
      const double t2 = th * th;
      const double f = th * (1.0 + t2 * (sh[4] + t2 * (sh[5] + t2 * (sh[6] + t2 * sh[7])))) - thd;
      const double df = 1.0 + t2 * (3.0 * sh[4] + t2 * (5.0 * sh[5] + t2 * (7.0 * sh[6] + t2 * 9.0 * sh[7])));
      if (!(fabs(df) > 1e-12)) break;
      th -= f / df;
    }
    // a point at or beyond 90 degrees has no pinhole image: clamp just short of it
    th = fmin(fmax(th, 0.0), 1.5);
    if (thd > 1e-300) {
      const double sc = tan(th) / thd;
      x = x0 * sc;
      y = y0 * sc;
    }
  }
  xo = x;
  yo = y;
}

// cost and (optionally) J^T J, J^T r of the 8 residuals wrt pose p (rvec,t)
template <bool WANT_J, Lens L>
__device__ double pnp_cost(const double* p, const double* sh, double hs, const double* pix, double* H, double* g,
                           bool* ok) {
  double idx[POSEX], px[POSEX];
  const double zero[6] = {0, 0, 0, 0, 0, 0};
  expand_pose(zero, idx);
  expand_marker_pose(p, px);   // the tag pose plays the marker role: its Jr slot holds R Jr
  BlockGeom<false> geo;
  block_geometry<false>(idx, px, nullptr, geo);
  double cost = 0.0;
  if (WANT_J) {
    for (int i = 0; i < 36; ++i) H[i] = 0.0;
    for (int i = 0; i < 6; ++i) g[i] = 0.0;
  }
  *ok = true;
  for (int k = 0; k < 4; ++k) {
    double ox, oy;
    corner_xy(k, hs, ox, oy);
    CornerRows<false> c;
    eval_corner<false, WANT_J, L>(geo, sh, ox, oy, pix[2 * k], pix[2 * k + 1], c);
    if (!(c.depth > 0.0) || !isfinite(c.r[0]) || !isfinite(c.r[1])) *ok = false;
    cost += c.r[0] * c.r[0] + c.r[1] * c.r[1];
    if (WANT_J) {
      for (int i = 0; i < 2; ++i)
        for (int a = 0; a < 6; ++a) {
          g[a] += c.jm[i][a] * c.r[i];
          for (int b = a; b < 6; ++b) H[a * 6 + b] += c.jm[i][a] * c.jm[i][b];
        }
    }
  }
  return 0.5 * cost;
}

template <Lens L>
__global__ void __launch_bounds__(128) pnp_kernel(int64_t n, const double* __restrict__ shared9,
                                                  const double* __restrict__ sizes, const double* __restrict__ pixels,
                                                  double* __restrict__ poses, double* __restrict__ final_cost,
                                                  int max_iter) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double sh[9], pix[8], p[6];
  for (int k = 0; k < 9; ++k) sh[k] = shared9[k];
  for (int k = 0; k < 8; ++k) pix[k] = pixels[i * 8 + k];
  for (int k = 0; k < 6; ++k) p[k] = poses[i * 6 + k];
  const double hs = 0.5 * sizes[i];
  bool have_guess = false;
  for (int k = 0; k < 6; ++k) have_guess |= (p[k] != 0.0);

  if (!have_guess) {
    // ---- undistorted normalised image points
    double xn[4], yn[4];
    for (int k = 0; k < 4; ++k) undistort_corner<L>(sh, pix[2 * k], pix[2 * k + 1], xn[k], yn[k]);
    // ---- homography (X,Y,1) -> (x,y,1) from the 4 corners, h33 = 1
    double A[8][8], b[8];
    for (int k = 0; k < 4; ++k) {
      double X, Y;
      corner_xy(k, hs, X, Y);
      const double r0[8] = {X, Y, 1, 0, 0, 0, -xn[k] * X, -xn[k] * Y};
      const double r1[8] = {0, 0, 0, X, Y, 1, -yn[k] * X, -yn[k] * Y};
      for (int c = 0; c < 8; ++c) { A[2 * k][c] = r0[c]; A[2 * k + 1][c] = r1[c]; }
      b[2 * k] = xn[k]; b[2 * k + 1] = yn[k];
    }
    bool okh = solve_dense<8>(A, b);
    double h1[3] = {b[0], b[3], b[6]}, h2[3] = {b[1], b[4], b[7]}, h3[3] = {b[2], b[5], 1.0};
    if (okh) {
      // H = [r1 r2 t] / t_z up to scale (h33 = 1 and t_z > 0 for a tag in front of the camera)
      const double n1 = sqrt(h1[0] * h1[0] + h1[1] * h1[1] + h1[2] * h1[2]);
      const double n2 = sqrt(h2[0] * h2[0] + h2[1] * h2[1] + h2[2] * h2[2]);
      const double lam = 2.0 / (n1 + n2);
      double r1v[3], r2v[3], r3v[3];
      for (int k = 0; k < 3; ++k) r1v[k] = h1[k] / n1;
      const double d12 = r1v[0] * h2[0] + r1v[1] * h2[1] + r1v[2] * h2[2];
      for (int k = 0; k < 3; ++k) r2v[k] = h2[k] - d12 * r1v[k];   // Gram-Schmidt
      const double nn = sqrt(r2v[0] * r2v[0] + r2v[1] * r2v[1] + r2v[2] * r2v[2]);
      for (int k = 0; k < 3; ++k) r2v[k] /= nn;
      r3v[0] = r1v[1] * r2v[2] - r1v[2] * r2v[1];
      r3v[1] = r1v[2] * r2v[0] - r1v[0] * r2v[2];
      r3v[2] = r1v[0] * r2v[1] - r1v[1] * r2v[0];
      const double R[9] = {r1v[0], r2v[0], r3v[0], r1v[1], r2v[1], r3v[1], r1v[2], r2v[2], r3v[2]};
      rot_to_rvec(R, p);
      p[3] = h3[0] * lam; p[4] = h3[1] * lam; p[5] = h3[2] * lam;
    } else {
      p[0] = p[1] = p[2] = 0.0; p[3] = p[4] = 0.0; p[5] = 1.0;
    }
  }

  // ---- Levenberg-Marquardt on the 8 residuals
  double H[36], g[6];
  bool ok;
  double cost = pnp_cost<true, L>(p, sh, hs, pix, H, g, &ok);
  double lambda = 1e-3;
  for (int it = 0; it < max_iter; ++it) {
    double A6[6][6], rhs[6];
    for (int a = 0; a < 6; ++a) {
      for (int c = 0; c < 6; ++c) A6[a][c] = (c >= a) ? H[a * 6 + c] : H[c * 6 + a];
      A6[a][a] += lambda * fmax(H[a * 6 + a], 1e-12);
      rhs[a] = -g[a];
    }
    if (!solve_dense<6>(A6, rhs)) { lambda *= 10.0; continue; }
    double q[6];
    double dn = 0.0, pn = 0.0;
    for (int a = 0; a < 6; ++a) { q[a] = p[a] + rhs[a]; dn += rhs[a] * rhs[a]; pn += p[a] * p[a]; }
    bool ok2;
    const double c2 = pnp_cost<false, L>(q, sh, hs, pix, nullptr, nullptr, &ok2);
    // Accept on "not worse up to rounding": along the weakly determined depth direction of a small tag the cost is
    // flat to 1e-16 relative while the step is still 1e-8, so convergence is declared on the step alone.
    // Below a relative step of 1e-5 the Gauss-Newton model is exact to rounding while the cost comparison is pure
    // noise (it would stall the iteration ~1e-8 short of the minimiser): such steps are taken on trust.
    const bool tiny = dn <= 1e-10 * (pn + 1e-10);
    if (ok2 && (tiny || c2 <= cost * (1.0 + 4e-16))) {
      for (int a = 0; a < 6; ++a) p[a] = q[a];
      cost = pnp_cost<true, L>(p, sh, hs, pix, H, g, &ok);
      lambda = fmax(lambda * 0.1, 1e-12);
      if (dn <= 1e-26 * (pn + 1e-26)) break;
    } else {
      lambda *= 10.0;
      if (lambda > 1e12) break;
    }
  }
  for (int k = 0; k < 6; ++k) poses[i * 6 + k] = p[k];
  if (final_cost) final_cost[i] = ok ? cost : -1.0;
}

// ---- rigid targets: one warp per (frame, target) problem
//
// A problem is the detected tags of one target in one frame; tag t's corners are corners[slot[t]][k] in the board
// frame (z = 0), the 64-byte slot records of rcc_ba_set_corner_layout.  Lane l handles corners l, l + 32, .. of the
// problem (corner c is corner c % 4 of tag c / 4), so every problem size runs on one warp.  Every sum over the
// corners is a per-lane partial followed by warp_sum, so all lanes hold the same bits and take the same branches;
// a problem's result depends only on its own inputs.

// v summed over the warp by a fixed xor butterfly.  Both lanes of a pair add the same two partials (a + b == b + a
// in IEEE arithmetic), so every lane ends with the same bits.
template <int N>
__device__ __forceinline__ void warp_sum(double (&v)[N]) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
}

struct TargetProblem {
  const double* corners;   // slot records: 4 corners (x, y) in the board frame
  const int32_t* slot;     // the problem's tags
  const double* pixels;    // 8 per tag
  int n;                   // corners: 4 per tag
};

// corner c of the problem: board point (X, Y) and its pixel (u, v)
__device__ __forceinline__ void target_corner(const TargetProblem& q, int c, double& X, double& Y, double& u,
                                              double& v) {
  const int t = c >> 2, k = c & 3;
  const double* o = q.corners + 8 * (int64_t)__ldg(q.slot + t) + 2 * k;
  X = __ldg(o);
  Y = __ldg(o + 1);
  u = __ldg(q.pixels + 8 * t + 2 * k);
  v = __ldg(q.pixels + 8 * t + 2 * k + 1);
}

// pose (rvec, t) of a plane from the columns h1 h2 h3 of its homography (X, Y, 1) -> normalised image point, known
// up to a positive scale: H = [r1 r2 t] / s.  The same decomposition as pnp_kernel's, which keeps its inline copy.
__device__ __forceinline__ void homography_pose(const double* h1, const double* h2, const double* h3, double* p) {
  const double n1 = sqrt(h1[0] * h1[0] + h1[1] * h1[1] + h1[2] * h1[2]);
  const double n2 = sqrt(h2[0] * h2[0] + h2[1] * h2[1] + h2[2] * h2[2]);
  const double lam = 2.0 / (n1 + n2);
  double r1v[3], r2v[3], r3v[3];
  for (int k = 0; k < 3; ++k) r1v[k] = h1[k] / n1;
  const double d12 = r1v[0] * h2[0] + r1v[1] * h2[1] + r1v[2] * h2[2];
  for (int k = 0; k < 3; ++k) r2v[k] = h2[k] - d12 * r1v[k];   // Gram-Schmidt
  const double nn = sqrt(r2v[0] * r2v[0] + r2v[1] * r2v[1] + r2v[2] * r2v[2]);
  for (int k = 0; k < 3; ++k) r2v[k] /= nn;
  r3v[0] = r1v[1] * r2v[2] - r1v[2] * r2v[1];
  r3v[1] = r1v[2] * r2v[0] - r1v[0] * r2v[2];
  r3v[2] = r1v[0] * r2v[1] - r1v[1] * r2v[0];
  const double R[9] = {r1v[0], r2v[0], r3v[0], r1v[1], r2v[1], r3v[1], r1v[2], r2v[2], r3v[2]};
  rot_to_rvec(R, p);
  p[3] = h3[0] * lam; p[4] = h3[1] * lam; p[5] = h3[2] * lam;
}

// cost of the problem's corners at pose p (rvec, t) and, with WANT_J, the upper triangle of J^T J (H, 21 values,
// row by row) and J^T r (g), all summed over the warp.  ok: every corner has depth > 0 and finite residuals.
template <bool WANT_J, Lens L>
__device__ double target_cost(const double* p, const double* sh, const TargetProblem& q, int lane, double* H,
                              double* g, bool* ok) {
  double idx[POSEX], px[POSEX];
  const double zero[6] = {0, 0, 0, 0, 0, 0};
  expand_pose(zero, idx);
  expand_marker_pose(p, px);   // the board pose plays the marker role (view = identity), as in pnp_cost
  BlockGeom<false> geo;
  block_geometry<false>(idx, px, nullptr, geo);
  constexpr int NS = WANT_J ? 28 : 1;   // [cost, J^T J (21), J^T r (6)]
  double acc[NS];
#pragma unroll
  for (int i = 0; i < NS; ++i) acc[i] = 0.0;
  bool good = true;
  for (int c = lane; c < q.n; c += 32) {
    double X, Y, u, v;
    target_corner(q, c, X, Y, u, v);
    CornerRows<false> cr;
    eval_corner<false, WANT_J, L>(geo, sh, X, Y, u, v, cr);
    if (!(cr.depth > 0.0) || !isfinite(cr.r[0]) || !isfinite(cr.r[1])) good = false;
    acc[0] += cr.r[0] * cr.r[0] + cr.r[1] * cr.r[1];
    if (WANT_J) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        int m = 1;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
          for (int b = a; b < 6; ++b) acc[m++] += cr.jm[i][a] * cr.jm[i][b];
#pragma unroll
        for (int a = 0; a < 6; ++a) acc[22 + a] += cr.jm[i][a] * cr.r[i];
      }
    }
  }
  warp_sum(acc);
  *ok = __all_sync(0xffffffffu, good);
  if (WANT_J) {
#pragma unroll
    for (int i = 0; i < 21; ++i) H[i] = acc[1 + i];
#pragma unroll
    for (int a = 0; a < 6; ++a) g[a] = acc[22 + a];
  }
  return 0.5 * acc[0];
}

template <Lens L>
__global__ void __launch_bounds__(128) pnp_target_kernel(int64_t n, const double* __restrict__ shared9,
                                                         const double* __restrict__ corners,
                                                         const int64_t* __restrict__ start,
                                                         const int32_t* __restrict__ slot,
                                                         const double* __restrict__ pixels, double* __restrict__ poses,
                                                         double* __restrict__ final_cost, int max_iter) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n) return;   // whole warps leave together: blockDim is a multiple of 32
  const int64_t t0 = start[w];
  const TargetProblem q{corners, slot + t0, pixels + 8 * t0, (int)(4 * (start[w + 1] - t0))};
  double sh[9], p[6];
  for (int k = 0; k < 9; ++k) sh[k] = shared9[k];
  for (int k = 0; k < 6; ++k) p[k] = poses[w * 6 + k];
  bool have_guess = false;
  for (int k = 0; k < 6; ++k) have_guess |= (p[k] != 0.0);

  if (!have_guess) {
    // ---- board points centred on their mean and scaled to a mean distance of sqrt(2) (Hartley)
    double m[2] = {0.0, 0.0};
    for (int c = lane; c < q.n; c += 32) {
      double X, Y, u, v;
      target_corner(q, c, X, Y, u, v);
      m[0] += X;
      m[1] += Y;
    }
    warp_sum(m);
    const double mx = m[0] / q.n, my = m[1] / q.n;
    double dsum[1] = {0.0};
    for (int c = lane; c < q.n; c += 32) {
      double X, Y, u, v;
      target_corner(q, c, X, Y, u, v);
      dsum[0] += sqrt((X - mx) * (X - mx) + (Y - my) * (Y - my));
    }
    warp_sum(dsum);
    const double sc = dsum[0] > 0.0 ? sqrt(2.0) * q.n / dsum[0] : 1.0;
    // ---- homography (X',Y',1) -> (x,y,1), h33 = 1, least squares over all corners: the normal equations, upper
    // triangle of A^T A (36) and A^T b (8), accumulated per lane and summed over the warp
    double ne[44];
#pragma unroll
    for (int i = 0; i < 44; ++i) ne[i] = 0.0;
    for (int c = lane; c < q.n; c += 32) {
      double X, Y, u, v, x, y;
      target_corner(q, c, X, Y, u, v);
      undistort_corner<L>(sh, u, v, x, y);
      X = (X - mx) * sc;
      Y = (Y - my) * sc;
      const double r0[8] = {X, Y, 1, 0, 0, 0, -x * X, -x * Y};
      const double r1[8] = {0, 0, 0, X, Y, 1, -y * X, -y * Y};
      int k = 0;
#pragma unroll
      for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = a; b < 8; ++b) ne[k++] += r0[a] * r0[b] + r1[a] * r1[b];
#pragma unroll
      for (int a = 0; a < 8; ++a) ne[36 + a] += r0[a] * x + r1[a] * y;
    }
    warp_sum(ne);
    double A[8][8], b[8];
    {
      int k = 0;
      for (int a = 0; a < 8; ++a)
        for (int c = a; c < 8; ++c) { A[a][c] = ne[k]; A[c][a] = ne[k]; ++k; }
      for (int a = 0; a < 8; ++a) b[a] = ne[36 + a];
    }
    if (solve_dense<8>(A, b)) {
      // back to the board frame: H = H' T with T = [sc 0 -sc mx; 0 sc -sc my; 0 0 1].  h33' = 1 is the depth of the
      // centroid up to the positive scale, so the decomposition keeps the sign of t.
      const double c1[3] = {b[0], b[3], b[6]}, c2[3] = {b[1], b[4], b[7]}, c3[3] = {b[2], b[5], 1.0};
      double h1[3], h2[3], h3[3];
      for (int k = 0; k < 3; ++k) {
        h1[k] = sc * c1[k];
        h2[k] = sc * c2[k];
        h3[k] = c3[k] - mx * h1[k] - my * h2[k];
      }
      homography_pose(h1, h2, h3, p);
    } else {
      p[0] = p[1] = p[2] = 0.0; p[3] = p[4] = 0.0; p[5] = 1.0;
    }
  }

  // ---- Levenberg-Marquardt on all residuals of the problem: pnp_kernel's acceptance, damping and stopping rules
  double H[21], g[6];
  bool ok;
  double cost = target_cost<true, L>(p, sh, q, lane, H, g, &ok);
  double lambda = 1e-3;
  for (int it = 0; it < max_iter; ++it) {
    double A6[6][6], rhs[6];
    {
      int k = 0;
      for (int a = 0; a < 6; ++a)
        for (int c = a; c < 6; ++c) { A6[a][c] = H[k]; A6[c][a] = H[k]; ++k; }
    }
    for (int a = 0; a < 6; ++a) {
      A6[a][a] += lambda * fmax(A6[a][a], 1e-12);
      rhs[a] = -g[a];
    }
    if (!solve_dense<6>(A6, rhs)) { lambda *= 10.0; continue; }
    double qp[6];
    double dn = 0.0, pn = 0.0;
    for (int a = 0; a < 6; ++a) { qp[a] = p[a] + rhs[a]; dn += rhs[a] * rhs[a]; pn += p[a] * p[a]; }
    bool ok2;
    const double c2 = target_cost<false, L>(qp, sh, q, lane, nullptr, nullptr, &ok2);
    // steps below 1e-5 relative are taken on trust (see pnp_kernel)
    const bool tiny = dn <= 1e-10 * (pn + 1e-10);
    if (ok2 && (tiny || c2 <= cost * (1.0 + 4e-16))) {
      for (int a = 0; a < 6; ++a) p[a] = qp[a];
      cost = target_cost<true, L>(p, sh, q, lane, H, g, &ok);
      lambda = fmax(lambda * 0.1, 1e-12);
      if (dn <= 1e-26 * (pn + 1e-26)) break;
    } else {
      lambda *= 10.0;
      if (lambda > 1e12) break;
    }
  }
  if (lane == 0) {
    for (int k = 0; k < 6; ++k) poses[w * 6 + k] = p[k];
    if (final_cost) final_cost[w] = ok ? cost : -1.0;
  }
}

// ---- plane homographies of rigid-target problems (cv::findHomography, method 0), one warp per problem
//
// Both sides are Hartley-normalised, board points (X', Y') = sb (X - mX, Y - mY) and pixels (x', y') = sp (u - mu,
// v - mv), and the 8 free entries h of the normalised homography Hn (h33 = 1) are solved for there: the DLT start and
// the Levenberg-Marquardt refinement both stay well conditioned although raw pixels are ~1e3 and board points ~1e-1.
// The residual is the pixel residual of H = Tp^-1 Hn Tb: (x'_pred - x') / sp == u_pred - u, so the minimiser is the
// one of cv::findHomography's HomographyRefineCallback cost.  pnp_target_kernel keeps its own inline copy of the
// board-side normalisation and DLT accumulation (it undistorts the image side and normalises only the board side).

// cost (normalised units: times 1 / sp^2 for px^2) of the problem at h and, with WANT_J, the upper triangle of J^T J
// (36 values, row by row) and J^T r, all summed over the warp.  ok: every corner has w' > 0 and finite residuals.
template <bool WANT_J>
__device__ double homography_cost(const double* h, const TargetProblem& q, int lane, const double* nrm, double* H,
                                  double* g, bool* ok) {
  constexpr int NS = WANT_J ? 45 : 1;   // [cost, J^T J (36), J^T r (8)]
  double acc[NS];
#pragma unroll
  for (int i = 0; i < NS; ++i) acc[i] = 0.0;
  bool good = true;
  for (int c = lane; c < q.n; c += 32) {
    double X, Y, u, v;
    target_corner(q, c, X, Y, u, v);
    X = (X - nrm[0]) * nrm[2];
    Y = (Y - nrm[1]) * nrm[2];
    const double x = (u - nrm[3]) * nrm[5], y = (v - nrm[4]) * nrm[5];
    const double wv = h[6] * X + h[7] * Y + 1.0;
    const double iw = 1.0 / wv;
    const double px = (h[0] * X + h[1] * Y + h[2]) * iw, py = (h[3] * X + h[4] * Y + h[5]) * iw;
    const double r[2] = {px - x, py - y};
    if (!(wv > 0.0) || !isfinite(r[0]) || !isfinite(r[1])) good = false;
    acc[0] += r[0] * r[0] + r[1] * r[1];
    if (WANT_J) {
      const double j[2][8] = {{X * iw, Y * iw, iw, 0, 0, 0, -px * X * iw, -px * Y * iw},
                              {0, 0, 0, X * iw, Y * iw, iw, -py * X * iw, -py * Y * iw}};
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        int m = 1;
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = a; b < 8; ++b) acc[m++] += j[i][a] * j[i][b];
#pragma unroll
        for (int a = 0; a < 8; ++a) acc[37 + a] += j[i][a] * r[i];
      }
    }
  }
  warp_sum(acc);
  *ok = __all_sync(0xffffffffu, good);
  if (WANT_J) {
#pragma unroll
    for (int i = 0; i < 36; ++i) H[i] = acc[1 + i];
#pragma unroll
    for (int a = 0; a < 8; ++a) g[a] = acc[37 + a];
  }
  return 0.5 * acc[0];
}

__global__ void __launch_bounds__(128) homography_target_kernel(int64_t n, const double* __restrict__ corners,
                                                                const int64_t* __restrict__ start,
                                                                const int32_t* __restrict__ slot,
                                                                const double* __restrict__ pixels,
                                                                double* __restrict__ Hout,
                                                                double* __restrict__ final_cost, int max_iter) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n) return;   // whole warps leave together: blockDim is a multiple of 32
  const int64_t t0 = start[w];
  const TargetProblem q{corners, slot + t0, pixels + 8 * t0, (int)(4 * (start[w + 1] - t0))};

  // ---- Hartley normalisation of both sides: nrm = {mX, mY, sb, mu, mv, sp}
  double m[4] = {0.0, 0.0, 0.0, 0.0};
  for (int c = lane; c < q.n; c += 32) {
    double X, Y, u, v;
    target_corner(q, c, X, Y, u, v);
    m[0] += X; m[1] += Y; m[2] += u; m[3] += v;
  }
  warp_sum(m);
  double nrm[6] = {m[0] / q.n, m[1] / q.n, 1.0, m[2] / q.n, m[3] / q.n, 1.0};
  double dsum[2] = {0.0, 0.0};
  for (int c = lane; c < q.n; c += 32) {
    double X, Y, u, v;
    target_corner(q, c, X, Y, u, v);
    dsum[0] += sqrt((X - nrm[0]) * (X - nrm[0]) + (Y - nrm[1]) * (Y - nrm[1]));
    dsum[1] += sqrt((u - nrm[3]) * (u - nrm[3]) + (v - nrm[4]) * (v - nrm[4]));
  }
  warp_sum(dsum);
  if (dsum[0] > 0.0) nrm[2] = sqrt(2.0) * q.n / dsum[0];
  if (dsum[1] > 0.0) nrm[5] = sqrt(2.0) * q.n / dsum[1];

  // ---- DLT start, h33 = 1, least squares over all corners: the normal equations, upper triangle of A^T A (36) and
  // A^T b (8), accumulated per lane and summed over the warp
  double ne[44];
#pragma unroll
  for (int i = 0; i < 44; ++i) ne[i] = 0.0;
  for (int c = lane; c < q.n; c += 32) {
    double X, Y, u, v;
    target_corner(q, c, X, Y, u, v);
    X = (X - nrm[0]) * nrm[2];
    Y = (Y - nrm[1]) * nrm[2];
    const double x = (u - nrm[3]) * nrm[5], y = (v - nrm[4]) * nrm[5];
    const double r0[8] = {X, Y, 1, 0, 0, 0, -x * X, -x * Y};
    const double r1[8] = {0, 0, 0, X, Y, 1, -y * X, -y * Y};
    int k = 0;
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = a; b < 8; ++b) ne[k++] += r0[a] * r0[b] + r1[a] * r1[b];
#pragma unroll
    for (int a = 0; a < 8; ++a) ne[36 + a] += r0[a] * x + r1[a] * y;
  }
  warp_sum(ne);
  double h[8];
  bool ok;
  {
    double A[8][8];
    int k = 0;
    for (int a = 0; a < 8; ++a)
      for (int c = a; c < 8; ++c) { A[a][c] = ne[k]; A[c][a] = ne[k]; ++k; }
    for (int a = 0; a < 8; ++a) h[a] = ne[36 + a];
    ok = solve_dense<8>(A, h);
  }

  double cost = -1.0;
  if (ok) {
    // ---- Levenberg-Marquardt on the normalised entries: pnp_target_kernel's acceptance, damping and stopping rules
    double H[36], g[8];
    cost = homography_cost<true>(h, q, lane, nrm, H, g, &ok);
    double lambda = 1e-3;
    for (int it = 0; it < max_iter; ++it) {
      double A8[8][8], rhs[8];
      {
        int k = 0;
        for (int a = 0; a < 8; ++a)
          for (int c = a; c < 8; ++c) { A8[a][c] = H[k]; A8[c][a] = H[k]; ++k; }
      }
      for (int a = 0; a < 8; ++a) {
        A8[a][a] += lambda * fmax(A8[a][a], 1e-12);
        rhs[a] = -g[a];
      }
      if (!solve_dense<8>(A8, rhs)) { lambda *= 10.0; continue; }
      double hq[8];
      double dn = 0.0, pn = 0.0;
      for (int a = 0; a < 8; ++a) { hq[a] = h[a] + rhs[a]; dn += rhs[a] * rhs[a]; pn += h[a] * h[a]; }
      bool ok2;
      const double c2 = homography_cost<false>(hq, q, lane, nrm, nullptr, nullptr, &ok2);
      // steps below 1e-5 relative are taken on trust (see pnp_kernel)
      const bool tiny = dn <= 1e-10 * (pn + 1e-10);
      if (ok2 && (tiny || c2 <= cost * (1.0 + 4e-16))) {
        for (int a = 0; a < 8; ++a) h[a] = hq[a];
        cost = homography_cost<true>(h, q, lane, nrm, H, g, &ok);
        lambda = fmax(lambda * 0.1, 1e-12);
        if (dn <= 1e-26 * (pn + 1e-26)) break;
      } else {
        lambda *= 10.0;
        if (lambda > 1e12) break;
      }
    }
  }

  // ---- back to the board frame and raw pixels: H = Tp^-1 Hn Tb with Tb = [sb 0 -sb mX; 0 sb -sb mY; 0 0 1] and
  // Tp^-1 = [1/sp 0 mu; 0 1/sp mv; 0 0 1], then scaled to H[8] = 1.  Tp^-1 keeps the third row, so w at a corner is
  // w' / H[8] before the scaling: every corner has w > 0 at the result when all w' > 0 and H[8] > 0.
  double R[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  if (ok) {
    const double hn[9] = {h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], 1.0};
    double M[9];   // Hn Tb
    for (int r = 0; r < 3; ++r) {
      M[3 * r + 0] = nrm[2] * hn[3 * r + 0];
      M[3 * r + 1] = nrm[2] * hn[3 * r + 1];
      M[3 * r + 2] = hn[3 * r + 2] - nrm[2] * (nrm[0] * hn[3 * r + 0] + nrm[1] * hn[3 * r + 1]);
    }
    for (int c = 0; c < 3; ++c) {
      R[c] = M[c] / nrm[5] + nrm[3] * M[6 + c];
      R[3 + c] = M[3 + c] / nrm[5] + nrm[4] * M[6 + c];
      R[6 + c] = M[6 + c];
    }
    const double s = R[8];
    ok = s > 0.0 && isfinite(s);
    for (int k = 0; k < 9; ++k) R[k] /= s;
    R[8] = 1.0;
    for (int k = 0; k < 9; ++k) ok = ok && isfinite(R[k]);
  }
  if (lane == 0) {
    for (int k = 0; k < 9; ++k) Hout[w * 9 + k] = ok ? R[k] : 0.0;
    if (final_cost) final_cost[w] = ok ? cost / (nrm[5] * nrm[5]) : -1.0;
  }
}

}  // namespace rcc

extern "C" int rcc_pnp_batch_lens(int32_t device, int32_t lens, int64_t n, const double* shared9, const double* sizes,
                                  const double* pixels, double* cam_T_tag, double* final_cost, int32_t max_iterations) {
  using namespace rcc;
  if (lens != LENS_RADTAN && lens != LENS_EQUIDISTANT) return RCC_BAD_ARG;
  if (n < 0 || !shared9 || (n > 0 && (!sizes || !pixels || !cam_T_tag))) return RCC_BAD_ARG;
  if (n == 0) return RCC_OK;
  try {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
      throw Error(RCC_CUDA_ERROR, "no CUDA device (this library has no CPU fallback)");
    RCC_CUDA(cudaSetDevice(device));
    DBuf<double> dsh, dsz, dpx, dpose, dcost;
    cudaStream_t s;
    RCC_CUDA(cudaStreamCreate(&s));
    dsh.upload(shared9, 9, s);
    dsz.upload(sizes, (size_t)n, s);
    dpx.upload(pixels, (size_t)n * 8, s);
    dpose.upload(cam_T_tag, (size_t)n * 6, s);
    dcost.alloc((size_t)n);
    const int iters = max_iterations > 0 ? max_iterations : 30;
    if (lens == LENS_EQUIDISTANT)
      pnp_kernel<LENS_EQUIDISTANT><<<ceil_div(n, 128), 128, 0, s>>>(n, dsh.p, dsz.p, dpx.p, dpose.p, dcost.p, iters);
    else
      pnp_kernel<LENS_RADTAN><<<ceil_div(n, 128), 128, 0, s>>>(n, dsh.p, dsz.p, dpx.p, dpose.p, dcost.p, iters);
    RCC_CUDA(cudaGetLastError());
    dpose.download(cam_T_tag, (size_t)n * 6, s);
    if (final_cost) dcost.download(final_cost, (size_t)n, s);
    RCC_CUDA(cudaStreamSynchronize(s));
    cudaStreamDestroy(s);
  } catch (const Error& e) {
    fprintf(stderr, "[rcc_pnp_batch] %s\n", e.what());
    return e.status;
  }
  return RCC_OK;
}

extern "C" int rcc_pnp_batch(int32_t device, int64_t n, const double* shared9, const double* sizes,
                             const double* pixels, double* cam_T_tag, double* final_cost, int32_t max_iterations) {
  return rcc_pnp_batch_lens(device, rcc::LENS_RADTAN, n, shared9, sizes, pixels, cam_T_tag, final_cost,
                            max_iterations);
}

extern "C" int rcc_pnp_target_batch(int32_t device, int32_t lens, const double* shared9, int32_t n_slots,
                                    const double* corners, int64_t n_problems, const int64_t* start,
                                    const int32_t* slot, const double* pixels, double* cam_T_target,
                                    double* final_cost, int32_t max_iterations) {
  using namespace rcc;
  if (lens != LENS_RADTAN && lens != LENS_EQUIDISTANT) return RCC_BAD_ARG;
  if (n_problems < 0) return RCC_BAD_ARG;
  if (n_problems == 0) return RCC_OK;
  if (!shared9 || !corners || !start || !slot || !pixels || !cam_T_target) return RCC_BAD_ARG;
  if (n_slots < 1) return RCC_BAD_ARG;
  if (start[0] != 0) return RCC_BAD_ARG;
  for (int64_t p = 0; p < n_problems; ++p)   // every problem has a tag, and no more corners than an int counts
    if (!(start[p + 1] > start[p]) || start[p + 1] - start[p] > (int64_t)(INT32_MAX / 4)) return RCC_BAD_ARG;
  const int64_t n_tags = start[n_problems];
  for (int64_t t = 0; t < n_tags; ++t)
    if (slot[t] < 0 || slot[t] >= n_slots) return RCC_BAD_ARG;
  for (int64_t i = 0; i < (int64_t)n_slots * 8; ++i)
    if (!std::isfinite(corners[i])) return RCC_BAD_ARG;
  cudaStream_t s = nullptr;
  try {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
      throw Error(RCC_CUDA_ERROR, "no CUDA device (this library has no CPU fallback)");
    RCC_CUDA(cudaSetDevice(device));
    DBuf<double> dsh, dcorn, dpx, dpose, dcost;
    DBuf<int64_t> dstart;
    DBuf<int32_t> dslot;
    RCC_CUDA(cudaStreamCreate(&s));
    dsh.upload(shared9, 9, s);
    dcorn.upload(corners, (size_t)n_slots * 8, s);
    dstart.upload(start, (size_t)n_problems + 1, s);
    dslot.upload(slot, (size_t)n_tags, s);
    dpx.upload(pixels, (size_t)n_tags * 8, s);
    dpose.upload(cam_T_target, (size_t)n_problems * 6, s);
    dcost.alloc((size_t)n_problems);
    const int iters = max_iterations > 0 ? max_iterations : 30;
    const int blocks = ceil_div(n_problems, 4);   // 4 warps of 128 threads, one problem each
    if (lens == LENS_EQUIDISTANT)
      pnp_target_kernel<LENS_EQUIDISTANT><<<blocks, 128, 0, s>>>(n_problems, dsh.p, dcorn.p, dstart.p, dslot.p,
                                                                 dpx.p, dpose.p, dcost.p, iters);
    else
      pnp_target_kernel<LENS_RADTAN><<<blocks, 128, 0, s>>>(n_problems, dsh.p, dcorn.p, dstart.p, dslot.p, dpx.p,
                                                            dpose.p, dcost.p, iters);
    RCC_CUDA(cudaGetLastError());
    dpose.download(cam_T_target, (size_t)n_problems * 6, s);
    if (final_cost) dcost.download(final_cost, (size_t)n_problems, s);
    RCC_CUDA(cudaStreamSynchronize(s));
    cudaStreamDestroy(s);
  } catch (const Error& e) {
    if (s) cudaStreamDestroy(s);
    fprintf(stderr, "[rcc_pnp_target_batch] %s\n", e.what());
    return e.status;
  }
  return RCC_OK;
}

extern "C" int rcc_homography_target_batch(int32_t device, int32_t n_slots, const double* corners, int64_t n_problems,
                                           const int64_t* start, const int32_t* slot, const double* pixels, double* H,
                                           double* final_cost, int32_t max_iterations) {
  using namespace rcc;
  if (n_problems < 0) return RCC_BAD_ARG;
  if (n_problems == 0) return RCC_OK;
  if (!corners || !start || !slot || !pixels || !H) return RCC_BAD_ARG;
  if (n_slots < 1) return RCC_BAD_ARG;
  if (start[0] != 0) return RCC_BAD_ARG;
  for (int64_t p = 0; p < n_problems; ++p)   // every problem has a tag, and no more corners than an int counts
    if (!(start[p + 1] > start[p]) || start[p + 1] - start[p] > (int64_t)(INT32_MAX / 4)) return RCC_BAD_ARG;
  const int64_t n_tags = start[n_problems];
  for (int64_t t = 0; t < n_tags; ++t)
    if (slot[t] < 0 || slot[t] >= n_slots) return RCC_BAD_ARG;
  for (int64_t i = 0; i < (int64_t)n_slots * 8; ++i)
    if (!std::isfinite(corners[i])) return RCC_BAD_ARG;
  cudaStream_t s = nullptr;
  try {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
      throw Error(RCC_CUDA_ERROR, "no CUDA device (this library has no CPU fallback)");
    RCC_CUDA(cudaSetDevice(device));
    DBuf<double> dcorn, dpx, dH, dcost;
    DBuf<int64_t> dstart;
    DBuf<int32_t> dslot;
    RCC_CUDA(cudaStreamCreate(&s));
    dcorn.upload(corners, (size_t)n_slots * 8, s);
    dstart.upload(start, (size_t)n_problems + 1, s);
    dslot.upload(slot, (size_t)n_tags, s);
    dpx.upload(pixels, (size_t)n_tags * 8, s);
    dH.alloc((size_t)n_problems * 9);
    dcost.alloc((size_t)n_problems);
    const int iters = max_iterations > 0 ? max_iterations : 30;
    const int blocks = ceil_div(n_problems, 4);   // 4 warps of 128 threads, one problem each
    homography_target_kernel<<<blocks, 128, 0, s>>>(n_problems, dcorn.p, dstart.p, dslot.p, dpx.p, dH.p, dcost.p,
                                                    iters);
    RCC_CUDA(cudaGetLastError());
    dH.download(H, (size_t)n_problems * 9, s);
    if (final_cost) dcost.download(final_cost, (size_t)n_problems, s);
    RCC_CUDA(cudaStreamSynchronize(s));
    cudaStreamDestroy(s);
  } catch (const Error& e) {
    if (s) cudaStreamDestroy(s);
    fprintf(stderr, "[rcc_homography_target_batch] %s\n", e.what());
    return e.status;
  }
  return RCC_OK;
}
