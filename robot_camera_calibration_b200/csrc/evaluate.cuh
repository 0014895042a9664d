// K1 and K6 kernel templates (see evaluate.cu for the design).  Included by evaluate.cu, which instantiates them with
// the square of each marker's size, and by evaluate_target.cu, which instantiates them with the corners of a corner
// layout (chunk.cuh: TARGET), so that the two sets compile in parallel.  One body per kernel serves both entry points:
// evaluate_body.cuh (evaluate_kernel, evaluate_target_kernel) and materialise_body.cuh (materialise_kernel,
// materialise_target_kernel).
#pragma once

#include "chunk.cuh"
#include "common.cuh"
#include "kernels.h"
#include "model.cuh"

namespace rcc {

constexpr int EVAL_THREADS = 256;
constexpr int EVAL_CTAS_PER_SM = 2;   // 128 registers x 256 threads

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
  int slot;       // TARGET: layout slot of the block
  int o;          // caller position of the block
  double2 px;
  bool on;
};

// K6: residual / cost evaluation without Jacobians (LM gain ratio, Evaluate() without jacobians).
// Persistent warps, a group of 8 blocks per warp iteration, the next group's indices and pixels in flight.
template <bool RIG, Lens L>
__global__ void __launch_bounds__(EVAL_THREADS, EVAL_CTAS_PER_SM) evaluate_kernel(const EvalArgs a) {
  constexpr bool TARGET = false;
#include "evaluate_body.cuh"
}

// the same with the corners of the corner layout
template <bool RIG, Lens L>
__global__ void __launch_bounds__(EVAL_THREADS, EVAL_CTAS_PER_SM) evaluate_target_kernel(const EvalArgs a) {
  constexpr bool TARGET = true;
#include "evaluate_body.cuh"
}

template <bool RIG, Lens L, bool TARGET>
static void launch_evaluate_t(const EvalArgs& a, cudaStream_t s) {
  if constexpr (TARGET) evaluate_target_kernel<RIG, L><<<eval_grid(a.n), EVAL_THREADS, 0, s>>>(a);
  else evaluate_kernel<RIG, L><<<eval_grid(a.n), EVAL_THREADS, 0, s>>>(a);
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
  using Poses = ChunkPoses<RIG, OWN_IS_VIEW, EvalArgs, false>;
#include "materialise_body.cuh"
}

// the same with the corners of the corner layout
template <bool RIG, bool OWN_IS_VIEW, Lens L>
__global__ void __launch_bounds__(MAT_WARPS * 32, 3) materialise_target_kernel(const EvalArgs a) {
  using Poses = ChunkPoses<RIG, OWN_IS_VIEW, EvalArgs, true>;
#include "materialise_body.cuh"
}

template <bool RIG, bool OWN_IS_VIEW, Lens L, bool TARGET>
static void launch_materialise_t(const EvalArgs& a, cudaStream_t s) {
  const size_t smem = (size_t)MAT_WARPS * MatSmem<RIG>::TOTAL * sizeof(double);
  void (*k)(EvalArgs);
  if constexpr (TARGET) k = materialise_target_kernel<RIG, OWN_IS_VIEW, L>;
  else k = materialise_kernel<RIG, OWN_IS_VIEW, L>;
  static SmemOptIn optin;
  optin.ensure(k, smem);
  k<<<ceil_div(a.n_chunks, MAT_WARPS), MAT_WARPS * 32, smem, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

template <Lens L, bool TARGET>
static void launch_evaluate_l(bool rig, bool want_jac, const EvalArgs& a, cudaStream_t s) {
  if (want_jac) {
    if (rig) {
      if (a.own_is_view) launch_materialise_t<true, true, L, TARGET>(a, s);
      else launch_materialise_t<true, false, L, TARGET>(a, s);
    } else {
      if (a.own_is_view) launch_materialise_t<false, true, L, TARGET>(a, s);
      else launch_materialise_t<false, false, L, TARGET>(a, s);
    }
    return;
  }
  if (rig) launch_evaluate_t<true, L, TARGET>(a, s);
  else launch_evaluate_t<false, L, TARGET>(a, s);
}

// every instantiation of one corner source (evaluate.cu: the square, evaluate_target.cu: the corner layout)
template <bool TARGET>
static void launch_evaluate_any(bool rig, bool want_jac, int lens, const EvalArgs& a, cudaStream_t s) {
  if (lens == LENS_PER_CAMERA) {
    if (want_jac) throw Error(RCC_BAD_ARG, "K1 takes one lens per launch");
    if (rig) launch_evaluate_t<true, LENS_PER_CAMERA, TARGET>(a, s);
    else launch_evaluate_t<false, LENS_PER_CAMERA, TARGET>(a, s);
  } else if (lens == LENS_EQUIDISTANT) launch_evaluate_l<LENS_EQUIDISTANT, TARGET>(rig, want_jac, a, s);
  else launch_evaluate_l<LENS_RADTAN, TARGET>(rig, want_jac, a, s);
}
}  // namespace rcc
