// K1 -- materialised cost-functor evaluation (residuals + per-parameter-block
// Jacobians in the Ceres CostFunction::Evaluate layout: materialise_kernel), and
// K6's cost-only evaluation used for the LM gain ratio (evaluate_kernel).
//
// K1 is HBM-write-bound: 1 408 B out per 72 B in per observation block.
#include "chunk.cuh"
#include "common.cuh"
#include "kernels.h"
#include "model.cuh"

namespace rcc {

constexpr int EVAL_THREADS = 256;
constexpr int EVAL_CTAS_PER_SM = 2;   // 128 registers x 256 threads

int eval_grid(int64_t n) {
  const int64_t groups = (n + 7) / 8;
  return (int)std::max<int64_t>(1, std::min<int64_t>((groups + EVAL_THREADS / 32 - 1) / (EVAL_THREADS / 32),
                                                     (int64_t)NUM_SMS_B200 * EVAL_CTAS_PER_SM));
}

__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0) {
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
  }
  return s;  // valid on thread 0
}

// per-warp staging (doubles), array-major: res[8][8] | intr[8][8x4] | dist[8][8x5] | view[8][8x6] | marker[8][8x6] | ext[8][8x6]
template <bool RIG>
struct EvalRec {
  static constexpr int RES = 0, JI = 64, JD = 320, JV = 640, JM = 1024, JX = 1408;
  static constexpr int SIZE = RIG ? 1792 : 1408;
};

// TMA bulk copy shared::cta -> global (16-byte aligned, size a multiple of 16); SASS: UBLKCP
__device__ __forceinline__ void bulk_store(double* gdst, const double* ssrc, int bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
               "r"((unsigned)__cvta_generic_to_shared(ssrc)), "r"(bytes)
               : "memory");
}

struct EvalIdx {      // raw loads only: nothing here may wait on memory when the next group is prefetched
  int vi, mi, cam;
  int o;          // caller position of the block
  double2 px;
  bool on;
};

// K6: residual / cost evaluation without Jacobians (LM gain ratio, Evaluate() without jacobians).
// Persistent warps, a group of 8 blocks per warp iteration, the next group's indices and pixels in flight.
template <bool RIG, Lens L>
__global__ void __launch_bounds__(EVAL_THREADS, EVAL_CTAS_PER_SM) evaluate_kernel(const EvalArgs a) {
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
      corner_xy(t, mx[PX_HS], ox, oy);
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
}

template <bool RIG, Lens L>
static void launch_evaluate_t(const EvalArgs& a, cudaStream_t s) {
  evaluate_kernel<RIG, L><<<eval_grid(a.n), EVAL_THREADS, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
// materialise_kernel: K1 proper.  The chunk pose pipeline of the fused kernel K2 (chunk.cuh: one
// warp per (own block, camera) chunk, lane 4b+t evaluates corner t of block b and streams its
// rows to shared memory as soon as a column group is complete), but the staged rows are the
// Ceres layout and leave the SM as TMA bulk copies instead of feeding MMAs.
// ---------------------------------------------------------------------------
template <bool RIG, bool OWN_IS_VIEW>
struct CeresSink {
  using ER = EvalRec<RIG>;
  double* rec;   // warp staging
  int q, t;      // block of the group, corner
  double d0[5];  // distortion row of the u residual waits for the v row: 10 contiguous doubles
  __device__ __forceinline__ void put6(int off, int i, const double* v) {
    double2* d = reinterpret_cast<double2*>(rec + off + q * 48 + (2 * t + i) * 6);
    d[0] = make_double2(v[0], v[1]);
    d[1] = make_double2(v[2], v[3]);
    d[2] = make_double2(v[4], v[5]);
  }
  __device__ __forceinline__ void shared(int i, const double* js, double r) {
    double2* d = reinterpret_cast<double2*>(rec + ER::JI + q * 32 + (2 * t + i) * 4);
    d[0] = make_double2(js[0], js[1]);
    d[1] = make_double2(js[2], js[3]);
    rec[ER::RES + q * 8 + 2 * t + i] = r;
    if (i == 0) {
#pragma unroll
      for (int k = 0; k < 5; ++k) d0[k] = js[4 + k];
    } else {
      d = reinterpret_cast<double2*>(rec + ER::JD + q * 40 + 10 * t);
      d[0] = make_double2(d0[0], d0[1]);
      d[1] = make_double2(d0[2], d0[3]);
      d[2] = make_double2(d0[4], js[4]);
      d[3] = make_double2(js[5], js[6]);
      d[4] = make_double2(js[7], js[8]);
    }
  }
  __device__ __forceinline__ void marker(int i, const double* jm) { put6(ER::JM, i, jm); }
  __device__ __forceinline__ void view(int i, const double* jv) { put6(ER::JV, i, jv); }
  __device__ __forceinline__ void ext(int i, const double* jx) { put6(ER::JX, i, jx); }
};

constexpr int MAT_WARPS = 4;
template <bool RIG>
struct MatSmem {   // per warp, doubles: Ceres-layout rows | pose region (chunk.cuh)
  static constexpr int TOTAL = EvalRec<RIG>::SIZE + CHUNK_POSE_SMEM<RIG>;
};

template <bool RIG, bool OWN_IS_VIEW, Lens L>
__global__ void __launch_bounds__(MAT_WARPS * 32, 3) materialise_kernel(const EvalArgs a) {
  using ER = EvalRec<RIG>;
  using MS = MatSmem<RIG>;
  constexpr int BPW = PassGeom<RIG>::BPW;
  extern __shared__ __align__(128) double smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chunk_id = blockIdx.x * MAT_WARPS + warp;
  if (chunk_id >= a.n_chunks) return;
  double* wsm = smem + (size_t)warp * MS::TOTAL;
  double* wrec = wsm;                 // Ceres-layout rows of the current group of 8 blocks
  const Chunk ch = a.chunks[chunk_id];
  const int b = lane >> 2, t = lane & 3;
  ChunkPoses<RIG, OWN_IS_VIEW, EvalArgs> poses(a, ch, wsm + ER::SIZE, lane);
  poses.start();
  auto load_pos = [&](int it) -> int {   // caller position of the lane's block
    return (it + b < ch.count) ? (a.orig ? a.orig[(int64_t)ch.start + it + b] : ch.start + it + b) : 0;
  };
  int pos_nxt = load_pos(0);
  double cost = 0.0;
  int buf = 0;
  for (int it = 0; it < ch.count; it += BPW, buf ^= 1) {
    double2 px;
    BlockGeom<RIG> geo;
    double ox, oy;
    const int pos = pos_nxt;
    if (it + BPW < ch.count) pos_nxt = load_pos(it + BPW);
    const bool valid = poses.group(it, buf, px, geo, ox, oy);
    // the previous group's bulk copies must have read the staging rows before they are rewritten
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    double r2 = 0.0;
    if (valid) {
      CeresSink<RIG, OWN_IS_VIEW> sink{wrec, b, t, {0, 0, 0, 0, 0}};
      double r0, r1;
      const double depth = eval_corner<RIG, true, L>(geo, poses.sh, ox, oy, px.x, px.y, sink, r0, r1);
      if (!(depth > 0.0) || !isfinite(r0) || !isfinite(r1)) *a.fail_flag = 1;
      r2 = r0 * r0 + r1 * r1;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // staged rows -> visible to the async proxy
    __syncwarp();
    // copy-out by the TMA engine: one bulk copy per output array when the group's blocks are
    // consecutive in caller order, one per (block, array) otherwise
    const int nblk = min(BPW, ch.count - it);
    const int p0 = __shfl_sync(0xffffffffu, pos, 0);
    const bool run = __all_sync(0xffffffffu, !valid || pos == p0 + b);
    constexpr int NARR = RIG ? 6 : 5;
    const int n_copies = run ? NARR : nblk * NARR;
    for (int idx = lane; idx < ((n_copies + 31) & ~31); idx += 32) {   // uniform trip count: shuffle inside
      const int qq = run ? 0 : idx / NARR, arr = run ? idx : idx - qq * NARR;
      const int64_t o = __shfl_sync(0xffffffffu, pos, (qq & 7) * 4);
      double* dst = nullptr;
      int off = 0, k = 0;
      switch (arr) {
        case 0: dst = a.residuals; off = ER::RES; k = 8; break;
        case 1: dst = a.jac_intr; off = ER::JI; k = 32; break;
        case 2: dst = a.jac_dist; off = ER::JD; k = 40; break;
        case 3: dst = a.jac_view; off = ER::JV; k = 48; break;
        case 4: dst = a.jac_marker; off = ER::JM; k = 48; break;
        default: dst = a.jac_ext; off = ER::JX; k = 48; break;
      }
      if (idx < n_copies && dst)
        bulk_store(dst + o * k, wrec + off + qq * k, (run ? nblk : 1) * k * (int)sizeof(double));
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    if (a.loss != 0) {
      double sb = r2 + __shfl_xor_sync(0xffffffffu, r2, 1);
      sb += __shfl_xor_sync(0xffffffffu, sb, 2);
      double rho1;
      r2 = valid ? 0.25 * robust_rho(a.loss, a.loss_a2, sb, rho1) : 0.0;
    }
    cost += r2;
  }
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // smem must outlive the reads
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, o);
  if (lane == 0 && a.cost2_partials) a.cost2_partials[chunk_id] = cost;
}

template <bool RIG, bool OWN_IS_VIEW, Lens L>
static void launch_materialise_t(const EvalArgs& a, cudaStream_t s) {
  const size_t smem = (size_t)MAT_WARPS * MatSmem<RIG>::TOTAL * sizeof(double);
  auto k = materialise_kernel<RIG, OWN_IS_VIEW, L>;
  static SmemOptIn optin;
  optin.ensure(k, smem);
  k<<<ceil_div(a.n_chunks, MAT_WARPS), MAT_WARPS * 32, smem, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

int eval_partials(bool want_jac, const EvalArgs& a) { return want_jac ? a.n_chunks : eval_grid(a.n); }

template <Lens L>
static void launch_evaluate_l(bool rig, bool want_jac, const EvalArgs& a, cudaStream_t s) {
  if (want_jac) {
    if (rig) {
      if (a.own_is_view) launch_materialise_t<true, true, L>(a, s);
      else launch_materialise_t<true, false, L>(a, s);
    } else {
      if (a.own_is_view) launch_materialise_t<false, true, L>(a, s);
      else launch_materialise_t<false, false, L>(a, s);
    }
    return;
  }
  if (rig) launch_evaluate_t<true, L>(a, s);
  else launch_evaluate_t<false, L>(a, s);
}

void launch_evaluate(bool rig, bool want_jac, int lens, const EvalArgs& a, cudaStream_t s) {
  if (a.n == 0) return;
  if (lens == LENS_PER_CAMERA) {
    if (want_jac) throw Error(RCC_BAD_ARG, "K1 takes one lens per launch");
    if (rig) launch_evaluate_t<true, LENS_PER_CAMERA>(a, s);
    else launch_evaluate_t<false, LENS_PER_CAMERA>(a, s);
  } else if (lens == LENS_EQUIDISTANT) launch_evaluate_l<LENS_EQUIDISTANT>(rig, want_jac, a, s);
  else launch_evaluate_l<LENS_RADTAN>(rig, want_jac, a, s);
}

void launch_cost(bool rig, int lens, const EvalArgs& a, cudaStream_t s) {
  EvalArgs b = a;
  b.residuals = nullptr;
  b.jac_intr = b.jac_dist = b.jac_view = b.jac_marker = b.jac_ext = nullptr;
  launch_evaluate(rig, false, lens, b, s);
}

// deterministic single-CTA sum
__global__ void __launch_bounds__(1024) sum_kernel(const double* __restrict__ in, int64_t n, double* __restrict__ out,
                                                   double scale) {
  __shared__ double red[1024];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += 1024) s += in[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0] * scale;
}

void launch_sum(const double* in, int64_t n, double* out, double scale, cudaStream_t s) {
  sum_kernel<<<1, 1024, 0, s>>>(in, n, out, scale);
  RCC_CUDA(cudaGetLastError());
}

}  // namespace rcc
