// K2 kernel template (see assemble.cu for the design).  Included by assemble.cu, which instantiates the
// radial-tangential lens, by assemble_equidistant.cu, which instantiates the equidistant lens, and by
// assemble_target.cu and assemble_target_equidistant.cu, which instantiate both lenses with the corners of a corner
// layout, so that the four sets of 16 kernels compile in parallel.  One body, assemble_body, serves both entry points:
// assemble_kernel (the square of the marker's size) and assemble_target_kernel (chunk.cuh: TARGET).
#pragma once

#include "chunk.cuh"
#include "common.cuh"
#include "kernels.h"
#include "model.cuh"

namespace rcc {

// stores the column groups of one corner's two residual rows into the staged row layout
template <bool RIG, bool EPASS, bool OWN_IS_VIEW>
struct RowSink {
  using PG = PassGeom<RIG>;
  double* row[2];
  double w;     // row scale sqrt(rho'(s)) of the block (1 for the trivial loss)
  __device__ __forceinline__ void put6(int i, int col, const double* v) {
    double2* d = reinterpret_cast<double2*>(row[i] + col);
    d[0] = make_double2(w * v[0], w * v[1]);
    d[1] = make_double2(w * v[2], w * v[3]);
    d[2] = make_double2(w * v[4], w * v[5]);
  }
  __device__ __forceinline__ void shared(int i, const double* js, double r) {
    double2* d = reinterpret_cast<double2*>(row[i] + 6);   // fx fy close tile A, the rest + r fill tile B
    d[0] = make_double2(w * js[0], w * js[1]);
    d[1] = make_double2(w * js[2], w * js[3]);
    d[2] = make_double2(w * js[4], w * js[5]);
    d[3] = make_double2(w * js[6], w * js[7]);
    d[4] = make_double2(w * js[8], w * r);
  }
  __device__ __forceinline__ void marker(int i, const double* jm) {
    if (!OWN_IS_VIEW) put6(i, 0, jm);
    else if (EPASS) put6(i, PG::COL_C, jm);
  }
  __device__ __forceinline__ void view(int i, const double* jv) {
    if (OWN_IS_VIEW) put6(i, 0, jv);
    else if (EPASS) put6(i, PG::COL_C, jv);
  }
  __device__ __forceinline__ void ext(int i, const double* jx) { put6(i, PG::COL_X, jx); }
};

// D(8x8) += A(8x4) B(4x8), FP64.  Lane l holds A[l/4][l%4], B[l%4][l/4], D[l/4][2(l%4)], D[l/4][2(l%4)+1].
__device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c[0]), "+d"(c[1])
               : "d"(a), "d"(b));
}

#ifndef RCC_K2_MIN_CTAS
#define RCC_K2_MIN_CTAS 3
#endif
#ifndef RCC_K2_MIN_CTAS_F
#define RCC_K2_MIN_CTAS_F 3   // single-camera F pass: 56 KB smem per CTA would allow 4, measured below
#endif

// per-warp shared memory (doubles): staged rows | pose region (chunk.cuh)
template <bool RIG, bool EPASS>
struct WarpSmem {
  using PG = PassGeom<RIG>;
  static constexpr int RS = EPASS ? PG::RS_E : PG::RS_F;
  static constexpr int BS = 8 * RS + 2;   // block stride: +16 B so the corner lanes of two blocks interleave over the banks
  static constexpr int STAGE = PG::BPW * BS;
  static constexpr int TOTAL = STAGE + CHUNK_POSE_SMEM<RIG>;
};

template <bool RIG, bool EPASS>
constexpr int K2_MIN_CTAS = (RIG && EPASS) ? 2 : ((!RIG && !EPASS) ? RCC_K2_MIN_CTAS_F : RCC_K2_MIN_CTAS);   // rig E pass: 89 KB smem per CTA

// tid = threadIdx.x, read by the __global__ entry point: there the compiler knows its range from the launch bounds
template <bool RIG, bool EPASS, bool OWN_IS_VIEW, bool LOSS, Lens L, bool TARGET>
__device__ __forceinline__ void assemble_body(const AssembleArgs& a, unsigned tid) {
  using PG = PassGeom<RIG>;
  using WS = WarpSmem<RIG, EPASS>;
  constexpr int BPW = PG::BPW, RS = WS::RS, BS = WS::BS;
  constexpr int PART = EPASS ? PG::PART_E : PG::PART_F;
  extern __shared__ __align__(16) double smem[];
  const int warp = tid >> 5, lane = tid & 31;
  const int launch_pos = blockIdx.x * PG::WARPS + warp;
  if (launch_pos >= a.n_chunks) return;  // whole warp leaves together
  const int chunk_id = a.chunk_list ? a.chunk_list[launch_pos] : launch_pos;
  double* wsm = smem + warp * WS::TOTAL;
  double* rows = wsm;                 // [BPW][8 rows][RS]

  const Chunk ch = a.chunks[chunk_id];
  const int b = lane >> 2;            // block of the warp iteration this lane evaluates a corner of
  const int t = lane & 3;             // corner

  // chunk constants -> shared memory; pad columns of the staged rows (never read back as results, but they do enter
  // the MMAs) are cleared once; then the first group's poses and pixels are set in flight
  ChunkPoses<RIG, OWN_IS_VIEW, AssembleArgs, TARGET> poses(a, ch, wsm + WS::STAGE, lane);
  for (int k = lane; k < BPW * BS; k += 32) rows[k] = 0.0;
  poses.start();

  // chunk accumulators: 8x8 tiles in MMA fragment layout
  double cAA[2] = {0.0, 0.0}, cAB[2] = {0.0, 0.0}, cBB[2] = {0.0, 0.0};
  double cAX[2] = {0.0, 0.0}, cBX[2] = {0.0, 0.0}, cXX[2] = {0.0, 0.0};
  double cost_acc = 0.0;
  // rows of corner t live at staged rows t (u) and 4 + t (v): k-step 0 of the MMA sums the u rows, k-step 1 the v rows
  double* my_rows = rows + b * BS + t * RS;
  const double* frag = rows + (lane & 3) * RS + (lane >> 2);   // + block * BS + kstep * 4 * RS + column tile
  int buf = 0;

  for (int it = 0; it < ch.count; it += BPW, buf ^= 1) {
    // ---- phase 1: corner evaluation ---------------------------------------
    double2 px;
    BlockGeom<RIG> geo;
    double ox, oy;
    const bool valid = poses.group(it, buf, px, geo, ox, oy);
    double w = 1.0;
    if (LOSS) {
      // s = sum of the 8 squared residuals of the block: residual-only evaluation, then a
      // butterfly over the block's 4 corner lanes
      double s_blk = 0.0;
      if (valid) {
        CornerRows<RIG> c;
        eval_corner<RIG, false, L>(geo, poses.sh, ox, oy, px.x, px.y, c);
        s_blk = c.r[0] * c.r[0] + c.r[1] * c.r[1];
      }
      s_blk += __shfl_xor_sync(0xffffffffu, s_blk, 1);
      s_blk += __shfl_xor_sync(0xffffffffu, s_blk, 2);
      double rho1;
      const double rho = robust_rho(a.loss, a.loss_a2, s_blk, rho1);
      w = sqrt(rho1);
      if (EPASS && valid && t == 0) cost_acc += rho;
    }
    if (valid) {
      RowSink<RIG, EPASS, OWN_IS_VIEW> sink{{my_rows, my_rows + 4 * RS}, w};
      double r0, r1;
      const double depth = eval_corner<RIG, true, L>(geo, poses.sh, ox, oy, px.x, px.y, sink, r0, r1);
      if (!(depth > 0.0) || !isfinite(r0) || !isfinite(r1)) *a.fail_flag = 1;
    }
    __syncwarp();
    // ---- phase 2: tile products over the 8 residual rows of every block ----
    auto block_products = [&](int bb) {
      const double* f0 = frag + bb * BS;
      const double* f1 = f0 + 4 * RS;
      const double a0 = f0[0], a1 = f1[0];
      const double b0 = f0[PG::COL_B], b1 = f1[PG::COL_B];
      dmma(cAA, a0, a0); dmma(cAA, a1, a1);
      dmma(cAB, a0, b0); dmma(cAB, a1, b1);
      if (EPASS) { dmma(cBB, b0, b0); dmma(cBB, b1, b1); }
      if (RIG) {
        const double x0 = f0[PG::COL_X], x1 = f1[PG::COL_X];
        dmma(cAX, a0, x0); dmma(cAX, a1, x1);
        if (EPASS) {
          dmma(cBX, b0, x0); dmma(cBX, b1, x1);
          dmma(cXX, x0, x0); dmma(cXX, x1, x1);
        }
      }
      if (EPASS) {
        // cross block W = J_own^T J_other of this observation block (rows own, columns other)
        const double t0 = f0[PG::COL_C], t1 = f1[PG::COL_C];
        double cW[2] = {0.0, 0.0};
        dmma(cW, a0, t0); dmma(cW, a1, t1);
        if (lane < 24 && (lane & 3) < 3)
          *reinterpret_cast<double2*>(a.W + ((int64_t)ch.start + it + bb) * 36 + (lane >> 2) * 6 + 2 * (lane & 3)) =
              make_double2(cW[0], cW[1]);
      }
    };
    // a full group (every group of a chunk but its last) runs as straight-line code, so that the fragment
    // loads of the next blocks can be issued ahead of the current block's MMAs
    if (ch.count - it >= BPW) {
#pragma unroll
      for (int bb = 0; bb < BPW; ++bb) block_products(bb);
    } else {
#pragma unroll 1
      for (int bb = 0; bb < ch.count - it; ++bb) block_products(bb);
    }
    __syncwarp();
  }

  // ---- chunk epilogue: the accumulator fragments are the partial (element (m, n) of a tile at m * 8 + n = 2 * lane + i)
  double2* out = reinterpret_cast<double2*>(a.partials + (size_t)chunk_id * PART) + lane;
  if (EPASS) {
    out[TE_AA * 32] = make_double2(cAA[0], cAA[1]);
    out[TE_AB * 32] = make_double2(cAB[0], cAB[1]);
    out[TE_BB * 32] = make_double2(cBB[0], cBB[1]);
    if (RIG) {
      out[TE_AX * 32] = make_double2(cAX[0], cAX[1]);
      out[TE_BX * 32] = make_double2(cBX[0], cBX[1]);
      out[TE_XX * 32] = make_double2(cXX[0], cXX[1]);
    }
    if (LOSS) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cost_acc += __shfl_xor_sync(0xffffffffu, cost_acc, o);
    }
    if (lane == 0) a.partials[(size_t)chunk_id * PART + PG::TILES_E * 64] = cost_acc;
  } else {
    out[TF_AA * 32] = make_double2(cAA[0], cAA[1]);
    out[TF_AB * 32] = make_double2(cAB[0], cAB[1]);
    if (RIG) out[TF_AX * 32] = make_double2(cAX[0], cAX[1]);
  }
}

template <bool RIG, bool EPASS, bool OWN_IS_VIEW, bool LOSS, Lens L>
__global__ void __launch_bounds__(PassGeom<RIG>::WARPS * 32, K2_MIN_CTAS<RIG, EPASS>)
assemble_kernel(const AssembleArgs a) {
  assemble_body<RIG, EPASS, OWN_IS_VIEW, LOSS, L, false>(a, threadIdx.x);
}

// the same with the corners of the corner layout
template <bool RIG, bool EPASS, bool OWN_IS_VIEW, bool LOSS, Lens L>
__global__ void __launch_bounds__(PassGeom<RIG>::WARPS * 32, K2_MIN_CTAS<RIG, EPASS>)
assemble_target_kernel(const AssembleArgs a) {
  assemble_body<RIG, EPASS, OWN_IS_VIEW, LOSS, L, true>(a, threadIdx.x);
}

template <bool RIG, bool EPASS, bool OWN_IS_VIEW, bool LOSS, Lens L, bool TARGET>
static void launch_assemble_t(const AssembleArgs& a, cudaStream_t s) {
  using PG = PassGeom<RIG>;
  if (a.n_chunks == 0) return;
  const size_t smem = PG::WARPS * WarpSmem<RIG, EPASS>::TOTAL * sizeof(double);
  void (*k)(AssembleArgs);
  if constexpr (TARGET) k = assemble_target_kernel<RIG, EPASS, OWN_IS_VIEW, LOSS, L>;
  else k = assemble_kernel<RIG, EPASS, OWN_IS_VIEW, LOSS, L>;
  static SmemOptIn optin;   // one per template instantiation
  optin.ensure(k, smem);
  const int grid = ceil_div(a.n_chunks, PG::WARPS);
  k<<<grid, PG::WARPS * 32, smem, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

template <bool LOSS, Lens L, bool TARGET = false>
static void launch_assemble_l(bool rig, bool epass, bool own_is_view, const AssembleArgs& a, cudaStream_t s) {
  const int sel = (rig ? 4 : 0) | (epass ? 2 : 0) | (own_is_view ? 1 : 0);
  switch (sel) {
    case 0: launch_assemble_t<false, false, false, LOSS, L, TARGET>(a, s); break;
    case 1: launch_assemble_t<false, false, true, LOSS, L, TARGET>(a, s); break;
    case 2: launch_assemble_t<false, true, false, LOSS, L, TARGET>(a, s); break;
    case 3: launch_assemble_t<false, true, true, LOSS, L, TARGET>(a, s); break;
    case 4: launch_assemble_t<true, false, false, LOSS, L, TARGET>(a, s); break;
    case 5: launch_assemble_t<true, false, true, LOSS, L, TARGET>(a, s); break;
    case 6: launch_assemble_t<true, true, false, LOSS, L, TARGET>(a, s); break;
    default: launch_assemble_t<true, true, true, LOSS, L, TARGET>(a, s); break;
  }
}

}  // namespace rcc
