// Body of the K6 kernels evaluate_kernel and evaluate_target_kernel (evaluate.cuh), included inside each: the including
// kernel defines RIG and L as template parameters and TARGET (the corner source, chunk.cuh) as a constexpr bool.
// Textual inclusion, not a force-inlined function: a body function is optimised before it is inlined and then compiles
// evaluate_kernel<., LENS_PER_CAMERA> to different SASS.
  constexpr int SP = RIG ? 15 : 9;
  constexpr int WPC = EVAL_THREADS / 32;
  __shared__ double red[WPC];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = lane >> 2, t = lane & 3;
  const int64_t n_groups = (a.n + 7) >> 3;
  const int64_t gw = (int64_t)blockIdx.x * WPC + warp, nw = (int64_t)gridDim.x * WPC;
  double cost = 0.0;

  auto load_idx = [&](int64_t grp) -> EvalIdx {
    EvalIdx x;
    const int64_t g = grp * 8 + q;
    x.on = grp < n_groups && g < a.n;
    x.vi = x.mi = x.cam = x.o = 0;
    x.px = make_double2(0.0, 0.0);
    if (x.on) {
      x.vi = a.view_idx[g];
      x.mi = a.marker_idx[g];
      x.cam = a.cam[g];
      x.o = a.orig ? a.orig[g] : (int)g;
      if constexpr (TARGET) x.slot = a.slot[g];
      x.px = *reinterpret_cast<const double2*>(a.pix + g * 8 + 2 * t);
    }
    return x;
  };

  EvalIdx cur = load_idx(gw);
  for (int64_t grp = gw; grp < n_groups; grp += nw) {
    const EvalIdx nxt = load_idx(grp + nw);   // in flight during this group's arithmetic
    double r2 = 0.0;
    if (cur.on) {
      // expanded pose records as 16-byte loads (the 4 corner lanes of a tag read the same lines)
      double vx[POSEX], mx[POSEX], xx[POSEX];
      {
        const double2* pv = reinterpret_cast<const double2*>(a.view_x + (size_t)cur.vi * POSEX);
        const double2* pm = reinterpret_cast<const double2*>(a.marker_x + (size_t)cur.mi * POSEX);
#pragma unroll
        for (int k = 0; k < 11; ++k) {
          const double2 u = pv[k], w = pm[k];
          vx[2 * k] = u.x; vx[2 * k + 1] = u.y;
          mx[2 * k] = w.x; mx[2 * k + 1] = w.y;
        }
        if (RIG) {
          const double2* pe = reinterpret_cast<const double2*>(a.ext_x + (size_t)cur.cam * POSEX);
#pragma unroll
          for (int k = 0; k < 11; ++k) {
            const double2 u = pe[k];
            xx[2 * k] = u.x; xx[2 * k + 1] = u.y;
          }
        }
      }
      BlockGeom<RIG> geo;
      block_geometry<RIG>(vx, mx, RIG ? xx : nullptr, geo);
      double ox, oy;
      if constexpr (TARGET) {
        if (cur.slot >= 0) layout_corner(a.corners, cur.slot, t, ox, oy);
        else corner_xy(t, mx[PX_HS], ox, oy);
      } else {
        corner_xy(t, mx[PX_HS], ox, oy);
      }
      CornerRows<RIG> c;
      const double* sh = a.shared + (size_t)cur.cam * SP;
      if constexpr (L == LENS_PER_CAMERA) {
        // the 4 corner lanes of a block share its camera: a warp takes at most both branches
        if ((a.cam_equidistant >> cur.cam) & 1u)
          eval_corner<RIG, false, LENS_EQUIDISTANT>(geo, sh, ox, oy, cur.px.x, cur.px.y, c);
        else
          eval_corner<RIG, false, LENS_RADTAN>(geo, sh, ox, oy, cur.px.x, cur.px.y, c);
      } else {
        eval_corner<RIG, false, L>(geo, sh, ox, oy, cur.px.x, cur.px.y, c);
      }
      if (!(c.depth > 0.0) || !isfinite(c.r[0]) || !isfinite(c.r[1])) *a.fail_flag = 1;
      r2 = c.r[0] * c.r[0] + c.r[1] * c.r[1];
      if (a.residuals)
        *reinterpret_cast<double2*>(a.residuals + (int64_t)cur.o * 8 + 2 * t) = make_double2(c.r[0], c.r[1]);
    }
    if (a.loss != 0) {
      // the 4 corner threads of a tag are adjacent lanes: rho(sum of the 8 squared residuals) / 4 each
      double sb = r2 + __shfl_xor_sync(0xffffffffu, r2, 1);
      sb += __shfl_xor_sync(0xffffffffu, sb, 2);
      double rho1;
      r2 = cur.on ? 0.25 * robust_rho(a.loss, a.loss_a2, sb, rho1) : 0.0;
    }
    cost += r2;
    cur = nxt;
  }
  const double s = block_sum(cost, red);
  if (threadIdx.x == 0 && a.cost2_partials) a.cost2_partials[blockIdx.x] = s;
