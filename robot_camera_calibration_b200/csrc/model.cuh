// Reprojection cost functor: pinhole + radial-tangential (or equidistant fisheye)
// camera observing the four corners of a square fiducial tag through Rodrigues poses.
//
// Conventions (all from /root/reference/real_preprocessing/src/camera_pose.cpp):
//   intrinsics fx fy cx cy = K[0] K[4] K[2] K[5]                     :61-62
//   distortion k1 k2 p1 p2 k3 (OpenCV order)                         :39, 63-64
//   poses = (Rodrigues rvec, t) of world_T_camera / world_T_target   :88-98, 111-121
//   tag corners bl br tr tl = (-+s/2, -+s/2, 0)                      :123-126, 158-161
//   projection model = the one cv::solvePnP minimises                :163
//
// Every function is __host__ __device__ so the arithmetic can be unit-tested on
// the build box (no GPU there); the product only ever runs it inside kernels.
#pragma once

#include <math.h>

#if defined(__CUDACC__)
#define RCC_HD __host__ __device__ __forceinline__
#else
#define RCC_HD inline
#endif

namespace rcc {

// expanded pose: R (row-major 3x3), Jr = right Jacobian of SO(3) at rvec, t.
// stored as 24 doubles (21 used) so one pose is 6 x 32-byte sectors.
// MARKER records hold R * Jr in the Jr slot (expand_marker_pose): the only use of a marker's Jr is
// K_m = cam_R_marker * Jr = M_t * (R_m Jr), which then no longer waits for cam_R_marker.
constexpr int POSEX = 24;
constexpr int PX_R = 0, PX_JR = 9, PX_T = 18;
constexpr int PX_RJ = PX_JR;   // marker records
constexpr int PX_HS = 21;  // marker records: half tag size (filled by expand_poses_kernel)

// Lens model of a camera (each camera of a problem has its own):
//   LENS_RADTAN       pinhole + radial-tangential, dist = k1 k2 p1 p2 k3 (cv::projectPoints)
//   LENS_EQUIDISTANT  equidistant fisheye (Kannala-Brandt), dist = k1 k2 k3 k4 + one reserved slot that the
//                     projection ignores (cv::fisheye::projectPoints with skew 0)
//   LENS_PER_CAMERA   not a lens: the cost-only kernel K6 picks one of the two per observation block from its
//                     camera (EvalArgs::cam_equidistant); eval_corner never takes it
enum Lens : int { LENS_RADTAN = 0, LENS_EQUIDISTANT = 1, LENS_PER_CAMERA = 2 };

// sin(t)/t, accurate for all t >= 0
RCC_HD double sinc_d(double t2, double t) {
  if (t2 < 1e-6) return 1.0 - t2 * (1.0 / 6.0) + t2 * t2 * (1.0 / 120.0);
  return sin(t) / t;
}

// atan2 as a template, so that code instantiating only the radial-tangential lens never needs atan2 for its scalar
// type (tests/host_harness/flop_count.cpp counts operations through a scalar class)
template <class T>
RCC_HD T atan2_t(T y, T x) {
  return atan2(y, x);
}

// (t - sin t cos t) / t^3 given sc = sin t cos t, accurate for all t >= 0 (series below t = 0.1: no cancellation)
RCC_HD double tsc3_d(double t2, double t, double sc) {
  if (t2 < 1e-2)
    return 2.0 / 3.0 + t2 * (-2.0 / 15.0 + t2 * (4.0 / 315.0 + t2 * (-2.0 / 2835.0 + t2 * (4.0 / 155925.0))));
  return (t - sc) / (t * t2);
}

// rvec,t (6 doubles) -> R, Jr, t.   R = I + A K + B K^2,  Jr = I - B K + C K^2,
// K = [r]x, A = sin t/t, B = (1-cos t)/t^2 (half-angle form: no cancellation),
// C = (t - sin t)/t^3 (series below t = 0.1: no cancellation).
RCC_HD void expand_pose(const double* __restrict__ p, double* __restrict__ o) {
  const double x = p[0], y = p[1], z = p[2];
  const double t2 = x * x + y * y + z * z;
  const double t = sqrt(t2);
  const double A = sinc_d(t2, t);
  const double Ah = sinc_d(0.25 * t2, 0.5 * t);
  const double B = 0.5 * Ah * Ah;
  double C;
  if (t2 < 1e-2) {
    C = 1.0 / 6.0 + t2 * (-1.0 / 120.0 + t2 * (1.0 / 5040.0 + t2 * (-1.0 / 362880.0 + t2 * (1.0 / 39916800.0))));
  } else {
    C = (1.0 - A) / t2;
  }
  // K^2 = r r^T - t2 I
  const double xx = x * x, yy = y * y, zz = z * z, xy = x * y, xz = x * z, yz = y * z;
  // R
  o[PX_R + 0] = 1.0 - B * (yy + zz);
  o[PX_R + 1] = -A * z + B * xy;
  o[PX_R + 2] = A * y + B * xz;
  o[PX_R + 3] = A * z + B * xy;
  o[PX_R + 4] = 1.0 - B * (xx + zz);
  o[PX_R + 5] = -A * x + B * yz;
  o[PX_R + 6] = -A * y + B * xz;
  o[PX_R + 7] = A * x + B * yz;
  o[PX_R + 8] = 1.0 - B * (xx + yy);
  // Jr = I - B K + C K^2
  o[PX_JR + 0] = 1.0 - C * (yy + zz);
  o[PX_JR + 1] = B * z + C * xy;
  o[PX_JR + 2] = -B * y + C * xz;
  o[PX_JR + 3] = -B * z + C * xy;
  o[PX_JR + 4] = 1.0 - C * (xx + zz);
  o[PX_JR + 5] = B * x + C * yz;
  o[PX_JR + 6] = B * y + C * xz;
  o[PX_JR + 7] = -B * x + C * yz;
  o[PX_JR + 8] = 1.0 - C * (xx + yy);
  o[PX_T + 0] = p[3];
  o[PX_T + 1] = p[4];
  o[PX_T + 2] = p[5];
  o[21] = 0.0; o[22] = 0.0; o[23] = 0.0;
}

// C = A B
RCC_HD void mat3_AB(const double* A, const double* B, double* C);

// marker pose: R, R * Jr, t
RCC_HD void expand_marker_pose(const double* __restrict__ p, double* __restrict__ o) {
  expand_pose(p, o);
  double rj[9];
  mat3_AB(o + PX_R, o + PX_JR, rj);
#pragma unroll
  for (int i = 0; i < 9; ++i) o[PX_RJ + i] = rj[i];
}

// C = A^T B   (3x3 row-major)
RCC_HD void mat3_AtB(const double* A, const double* B, double* C) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      C[3 * i + j] = A[0 + i] * B[0 + j] + A[3 + i] * B[3 + j] + A[6 + i] * B[6 + j];
}
// C = A B
RCC_HD void mat3_AB(const double* A, const double* B, double* C) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
// y = A^T x
RCC_HD void mat3_Atx(const double* A, const double* x, double* y) {
#pragma unroll
  for (int i = 0; i < 3; ++i) y[i] = A[i] * x[0] + A[3 + i] * x[1] + A[6 + i] * x[2];
}
// G = s * [p]x M   (3x3)
RCC_HD void cross_mat(const double* p, const double* M, double s, double* G) {
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    G[0 + j] = s * (-p[2] * M[3 + j] + p[1] * M[6 + j]);
    G[3 + j] = s * (p[2] * M[0 + j] - p[0] * M[6 + j]);
    G[6 + j] = s * (-p[1] * M[0 + j] + p[0] * M[3 + j]);
  }
}

// B = s * A [p]x  for a 2x3 A  (row i of B = s * (A_i x p))
RCC_HD void a_cross(const double (*A)[3], const double* p, double s, double (*B)[3]) {
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    B[i][0] = s * (A[i][1] * p[2] - A[i][2] * p[1]);
    B[i][1] = s * (A[i][2] * p[0] - A[i][0] * p[2]);
    B[i][2] = s * (A[i][0] * p[1] - A[i][1] * p[0]);
  }
}
// out[j] = sum_k B[k] M[3k+j]   (row vector times 3x3)
RCC_HD void row_mat(const double* B, const double* M, double* out) {
#pragma unroll
  for (int j = 0; j < 3; ++j) out[j] = B[0] * M[j] + B[1] * M[3 + j] + B[2] * M[6 + j];
}

// Geometry shared by the four corners of one observation block.
template <bool RIG>
struct BlockGeom {
  double Rcm[9];   // cam_R_marker
  double c0[3];    // marker origin in the camera frame
  double Km[9];    // Rcm * Jr(marker rvec)
  double Mt[9];    // d Pc / d t_marker  (= Rv^T single, Rx^T Rb^T rig);  d Pc/d t_view|body = -Mt
  double Jrv[9];   // Jr(view rvec)            (single)  /  Jr(body rvec) (rig)
  // rig only
  double Rbm[9];   // body_R_marker
  double qb0[3];   // marker origin in the body frame
  double RxT[9];   // Rx^T  (row-major)
  double Jrx[9];   // Jr(ext rvec)
};

// vx = expanded view (or body) pose, mx = expanded marker pose, xx = expanded
// body_T_cam (rig only, may be nullptr otherwise)
template <bool RIG>
RCC_HD void block_geometry(const double* __restrict__ vx, const double* __restrict__ mx,
                           const double* __restrict__ xx, BlockGeom<RIG>& g) {
  double dt[3] = {mx[PX_T + 0] - vx[PX_T + 0], mx[PX_T + 1] - vx[PX_T + 1], mx[PX_T + 2] - vx[PX_T + 2]};
#pragma unroll
  for (int i = 0; i < 9; ++i) g.Jrv[i] = vx[PX_JR + i];
  if (!RIG) {
    // [Rcm | Km | c0] = Rv^T [Rm | Rm Jr(rm) | tm - tv]: three independent products
    mat3_AtB(vx + PX_R, mx + PX_R, g.Rcm);
    mat3_Atx(vx + PX_R, dt, g.c0);
    mat3_AtB(vx + PX_R, mx + PX_RJ, g.Km);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) g.Mt[3 * i + j] = vx[PX_R + 3 * j + i];
  } else {
    mat3_AtB(vx + PX_R, mx + PX_R, g.Rbm);
    mat3_Atx(vx + PX_R, dt, g.qb0);
    mat3_AtB(xx + PX_R, g.Rbm, g.Rcm);
    double q[3] = {g.qb0[0] - xx[PX_T + 0], g.qb0[1] - xx[PX_T + 1], g.qb0[2] - xx[PX_T + 2]};
    mat3_Atx(xx + PX_R, q, g.c0);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) g.RxT[3 * i + j] = xx[PX_R + 3 * j + i];
    // Mt = Rx^T Rb^T : Mt[i][j] = sum_k Rx[k][i] Rb[j][k]
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        g.Mt[3 * i + j] = xx[PX_R + 0 + i] * vx[PX_R + 3 * j + 0] + xx[PX_R + 3 + i] * vx[PX_R + 3 * j + 1] +
                          xx[PX_R + 6 + i] * vx[PX_R + 3 * j + 2];
    mat3_AB(g.Mt, mx + PX_RJ, g.Km);   // Rcm Jr(rm) = (Rx^T Rb^T)(Rm Jr(rm))
#pragma unroll
    for (int i = 0; i < 9; ++i) g.Jrx[i] = xx[PX_JR + i];
  }
}

// Two residual rows (u, v) of one corner and their Jacobian rows; the Jacobian rows are written as an eval_corner
// sink.
//   jv : d/d view  (rvec 0:3, t 3:6)   [world_T_camera | world_T_body]
//   jm : d/d marker
//   js : d/d (fx fy cx cy k1 k2 p1 p2 k3)   [equidistant: fx fy cx cy k1 k2 k3 k4, reserved slot 0]
//   jx : d/d body_T_cam (rig only)
template <bool RIG>
struct CornerRows {
  double r[2];
  double jv[2][6];
  double jm[2][6];
  double js[2][9];
  double jx[2][6];
  double depth;
  RCC_HD void shared(int i, const double* v, double) {
#pragma unroll
    for (int k = 0; k < 9; ++k) js[i][k] = v[k];
  }
  RCC_HD void marker(int i, const double* v) {
#pragma unroll
    for (int k = 0; k < 6; ++k) jm[i][k] = v[k];
  }
  RCC_HD void view(int i, const double* v) {
#pragma unroll
    for (int k = 0; k < 6; ++k) jv[i][k] = v[k];
  }
  RCC_HD void ext(int i, const double* v) {
#pragma unroll
    for (int k = 0; k < 6; ++k) jx[i][k] = v[k];
  }
};

// Residuals (r0, r1) = (u, v) of one corner and, with WANT_J, their analytic Jacobian rows.
// shared = fx fy cx cy k1 k2 p1 p2 k3 (LENS_RADTAN) | fx fy cx cy k1 k2 k3 k4 - (LENS_EQUIDISTANT);
// (ox, oy) = corner in the tag frame ; (pu, pv) = observed pixel.
// Every column group of the two rows is handed to `sink` as soon as it is complete, so that a kernel can store
// it (shared memory) immediately and keep register live ranges short:
//   sink.shared(i, js[9], r)   sink.marker(i, jm[6])   sink.view(i, jv[6])   sink.ext(i, jx[6])
// with i = 0 (u row), 1 (v row).  WANT_J = false returns before the first sink call.  Returns the corner's depth.
// The lenses differ only in the residual, js and A = d(u,v)/dPc; the pose column groups are formed from A.
template <bool RIG, bool WANT_J, Lens L = LENS_RADTAN, class Sink>
RCC_HD double eval_corner(const BlockGeom<RIG>& g, const double* __restrict__ sh, double ox, double oy, double pu,
                          double pv, Sink& sink, double& r0, double& r1) {
  static_assert(L == LENS_RADTAN || L == LENS_EQUIDISTANT, "eval_corner takes one lens");
  const double fx = sh[0], fy = sh[1], cx = sh[2], cy = sh[3];
  const double k1 = sh[4], k2 = sh[5], p1 = sh[6], p2 = sh[7], k3 = sh[8];
  double d[3], P[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    d[i] = g.Rcm[3 * i] * ox + g.Rcm[3 * i + 1] * oy;
    P[i] = d[i] + g.c0[i];
  }
  double A[2][3];   // A = d(u,v)/dPc  (2x3)
  if constexpr (L == LENS_RADTAN) {
    const double iz = 1.0 / P[2];
    const double x = P[0] * iz, y = P[1] * iz;
    const double xx = x * x, yy = y * y, xy = x * y;
    const double r2 = xx + yy;
    const double r4 = r2 * r2, r6 = r4 * r2;
    const double rad = 1.0 + k1 * r2 + k2 * r4 + k3 * r6;
    const double tx = 2.0 * xy, ax = r2 + 2.0 * xx, ay = r2 + 2.0 * yy;
    const double xd = x * rad + p1 * tx + p2 * ax;
    const double yd = y * rad + p1 * ay + p2 * tx;
    r0 = fx * xd + cx - pu;
    r1 = fy * yd + cy - pv;
    if (!WANT_J) return P[2];
    {  // intrinsics / distortion
      const double fxx = fx * x, fyy = fy * y;
      const double js0[9] = {xd, 0.0, 1.0, 0.0, fxx * r2, fxx * r4, fx * tx, fx * ax, fxx * r6};
      sink.shared(0, js0, r0);
      const double js1[9] = {0.0, yd, 0.0, 1.0, fyy * r2, fyy * r4, fy * ay, fy * tx, fyy * r6};
      sink.shared(1, js1, r1);
    }
    // d(xd,yd)/d(x,y)
    const double drad = k1 + 2.0 * k2 * r2 + 3.0 * k3 * r4;  // d rad / d r2
    const double dxx = rad + 2.0 * xx * drad + 2.0 * p1 * y + 6.0 * p2 * x;
    const double dxy = 2.0 * xy * drad + 2.0 * p1 * x + 2.0 * p2 * y;
    const double dyy = rad + 2.0 * yy * drad + 6.0 * p1 * y + 2.0 * p2 * x;
    A[0][0] = fx * dxx * iz;
    A[0][1] = fx * dxy * iz;
    A[0][2] = -(A[0][0] * x + A[0][1] * y);
    A[1][0] = fy * dxy * iz;
    A[1][1] = fy * dyy * iz;
    A[1][2] = -(A[1][0] * x + A[1][1] * y);
  } else {
    // equidistant: rho = |(X, Y)|, th = atan2(rho, Z), th_d = th f(th^2), f = 1 + k1 th^2 + .. + k4 th^8,
    // (x', y') = s (X, Y) with s = th_d / rho = f c, c = th / rho = 1 / (R sinc th), R = |Pc|.
    // sin th = rho / R and cos th = Z / R, so no trigonometric function is evaluated besides atan2.
    // Nothing divides by a small rho: c (series of 1 / sinc near the axis), and q = (1/rho) ds/drho below, stay
    // finite on the optical axis.
    const double e1 = sh[4], e2 = sh[5], e3 = sh[6], e4 = sh[7];
    const double rho2 = P[0] * P[0] + P[1] * P[1];
    const double R2 = rho2 + P[2] * P[2], iR2 = 1.0 / R2;
    const double rho = sqrt(rho2);
    const double th = atan2_t(rho, P[2]);
    const double t2 = th * th;
    const double c = t2 < 1e-6 ? 1.0 / (sqrt(R2) * (1.0 - t2 * (1.0 / 6.0) + t2 * t2 * (1.0 / 120.0))) : th / rho;
    const double f = 1.0 + t2 * (e1 + t2 * (e2 + t2 * (e3 + t2 * e4)));
    const double s = f * c;
    const double xd = s * P[0], yd = s * P[1];
    r0 = fx * xd + cx - pu;
    r1 = fy * yd + cy - pv;
    if (!WANT_J) return P[2];
    {  // intrinsics / distortion: d x' / d k_i = th^(2i) c X; the reserved slot has a zero column
      const double t4 = t2 * t2, t6 = t4 * t2, t8 = t4 * t4;
      const double fxc = fx * c * P[0], fyc = fy * c * P[1];
      const double js0[9] = {xd, 0.0, 1.0, 0.0, fxc * t2, fxc * t4, fxc * t6, fxc * t8, 0.0};
      sink.shared(0, js0, r0);
      const double js1[9] = {0.0, yd, 0.0, 1.0, fyc * t2, fyc * t4, fyc * t6, fyc * t8, 0.0};
      sink.shared(1, js1, r1);
    }
    // d th_d / d th = 1 + 3 k1 th^2 + .. + 9 k4 th^8 ;  f'(th) / th = 2 k1 + 4 k2 th^2 + .. + 8 k4 th^6
    const double fd = 1.0 + t2 * (3.0 * e1 + t2 * (5.0 * e2 + t2 * (7.0 * e3 + t2 * (9.0 * e4))));
    const double fp = 2.0 * e1 + t2 * (4.0 * e2 + t2 * (6.0 * e3 + t2 * (8.0 * e4)));
    // dx'/dX = s + X^2 q, dx'/dY = X Y q, dx'/dZ = -X fd / R^2, with q = (fp - fd (th - sin th cos th) / th^3) c^3
    const double q = (fp - fd * tsc3_d(t2, th, rho * P[2] * iR2)) * (c * c * c);
    const double gz = -fd * iR2;
    const double qxy = q * P[0] * P[1];
    A[0][0] = fx * (s + q * P[0] * P[0]);
    A[0][1] = fx * qxy;
    A[0][2] = fx * gz * P[0];
    A[1][0] = fy * qxy;
    A[1][1] = fy * (s + q * P[1] * P[1]);
    A[1][2] = fy * gz * P[1];
  }

  // J = A [p]x M is formed as (A [p]x) M: 12 + 18 operations instead of 27 + 18
  double jvt[2][3];  // d/d t_view = -A Mt (kept until the rotation part is ready)
  double B[2][3];
  a_cross(A, d, -1.0, B);   // marker rotation: -A [d]x Km
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    double jm[6];
    row_mat(B[i], g.Km, jm);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double mt = A[i][0] * g.Mt[j] + A[i][1] * g.Mt[3 + j] + A[i][2] * g.Mt[6 + j];
      jm[3 + j] = mt;
      jvt[i][j] = -mt;
    }
    sink.marker(i, jm);
  }
  if (!RIG) {
    a_cross(A, P, 1.0, B);    // view rotation: A [Pc]x Jr(rv)
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      double jv[6];
      row_mat(B[i], g.Jrv, jv);
#pragma unroll
      for (int j = 0; j < 3; ++j) jv[3 + j] = jvt[i][j];
      sink.view(i, jv);
    }
  } else {
    double qb[3], Ax[2][3];
#pragma unroll
    for (int i = 0; i < 3; ++i) qb[i] = g.Rbm[3 * i] * ox + g.Rbm[3 * i + 1] * oy + g.qb0[i];
#pragma unroll
    for (int i = 0; i < 2; ++i) row_mat(A[i], g.RxT, Ax[i]);   // A Rx^T
    a_cross(Ax, qb, 1.0, B);  // body rotation: A Rx^T [qb]x Jr(rb)
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      double jv[6];
      row_mat(B[i], g.Jrv, jv);
#pragma unroll
      for (int j = 0; j < 3; ++j) jv[3 + j] = jvt[i][j];
      sink.view(i, jv);
    }
    a_cross(A, P, 1.0, B);    // extrinsic rotation: A [Pc]x Jr(rx) ; translation: -A Rx^T
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      double jx[6];
      row_mat(B[i], g.Jrx, jx);
#pragma unroll
      for (int j = 0; j < 3; ++j) jx[3 + j] = -Ax[i][j];
      sink.ext(i, jx);
    }
  }
  return P[2];
}

// eval_corner into a CornerRows (residuals, depth and, with WANT_J, the Jacobian rows)
template <bool RIG, bool WANT_J, Lens L = LENS_RADTAN>
RCC_HD void eval_corner(const BlockGeom<RIG>& g, const double* __restrict__ sh, double ox, double oy, double pu,
                        double pv, CornerRows<RIG>& out) {
  out.depth = eval_corner<RIG, WANT_J, L>(g, sh, ox, oy, pu, pv, out, out.r[0], out.r[1]);
}

// Robust loss rho(s) on s = ||r_block||^2 (all 8 residuals of a tag), Ceres semantics:
// the corrected Gauss-Newton model scales residuals and Jacobian rows of the block by
// sqrt(rho'(s)) (for Huber and Cauchy rho'' <= 0, so Ceres's alpha is 0) and the cost is
// 0.5 * rho(s).   loss: 0 trivial, 1 Huber(a), 2 Cauchy(a);  a2 = a * a.
RCC_HD double robust_rho(int loss, double a2, double s, double& rho1) {
  if (loss == 1) {
    if (s <= a2) { rho1 = 1.0; return s; }
    const double r = sqrt(s), a = sqrt(a2);
    rho1 = a / r;
    return 2.0 * a * r - a2;
  }
  if (loss == 2) {
    const double q = 1.0 + s / a2;
    rho1 = 1.0 / q;
    return a2 * log(q);
  }
  rho1 = 1.0;
  return s;
}

// corner k of a tag of half-size hs: bl br tr tl
RCC_HD void corner_xy(int k, double hs, double& ox, double& oy) {
  ox = (k == 1 || k == 2) ? hs : -hs;
  oy = (k >= 2) ? hs : -hs;
}

}  // namespace rcc
