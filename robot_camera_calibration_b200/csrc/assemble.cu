// K2 -- fused reprojection residual + analytic Jacobian + Gauss-Newton normal
// equation assembly.  The Jacobian never reaches HBM.
//
// Replaces (SURVEY.md 8a rows a1, a8): the Ceres cost-functor evaluation and the
// linearisation / J^T J builder that the reference's missing optimiser stage
// would run between camera_pose.cpp (initial guesses) and opt_visualization.cpp.
//
// Work decomposition.  Observation blocks are sorted by the 6-dof block that
// "owns" the pass (the eliminated set in the E pass, the kept set in the F
// pass) and cut into chunks that share (own block, camera).  One warp walks one
// chunk, 8 observation blocks per iteration:
//   phase 1  lane 4b+t evaluates corner t of block b (2 residual rows, all
//            Jacobian column groups) and stages the rows in shared memory
//            (column tiles of 8, see kernels.h);
//   phase 2  for every block the warp forms  tile_I^T tile_J  over the block's
//            8 residual rows with FP64 tensor-core MMAs (mma.sync.m8n8k4.f64,
//            two k-steps).  DMMA issues at the FP64 DFMA rate on B200
//            (tools/ubench/dmma_rate.cu: 37.1 TFLOP/s either way) but takes one
//            operand register per lane instead of 12 and keeps an 8x8
//            accumulator in 2 registers per lane, so the phase is bound by the
//            FP64 pipe instead of by shared-memory operand traffic.
// The chunk sums stay in the MMA accumulators and leave the warp once per chunk
// as coalesced 16-byte stores; the per-block cross tile J_own^T J_other (the
// Schur off-diagonal block W) is written straight to HBM.  finalize_* reduce the
// chunk partials in a fixed order (deterministic, no FP64 atomics).
#include "assemble.cuh"

namespace rcc {

void launch_assemble(bool rig, bool epass, bool own_is_view, int lens, const AssembleArgs& a, cudaStream_t s) {
  if (a.corners) {
    if (lens == LENS_EQUIDISTANT) launch_assemble_target_equidistant(rig, epass, own_is_view, a, s);
    else launch_assemble_target(rig, epass, own_is_view, a, s);
  } else if (lens == LENS_EQUIDISTANT) launch_assemble_equidistant(rig, epass, own_is_view, a, s);
  else if (a.loss != 0) launch_assemble_l<true, LENS_RADTAN>(rig, epass, own_is_view, a, s);
  else launch_assemble_l<false, LENS_RADTAN>(rig, epass, own_is_view, a, s);
}

// ---------------------------------------------------------------------------
// finalize_side: one warp per own block sums its chunk partials in chunk order.
// output (r, j): row r of the own block; j < 6 -> H_oo[r][j], j == 6 -> g_o[r],
// j >= 7 -> H_os[r][shared parameter j - 7] (kept per camera).
// ---------------------------------------------------------------------------
template <bool RIG, bool EPASS>
__device__ __forceinline__ void finalize_side_body(const FinalizeSideArgs& a, int i) {
  // one WARP per own block i; lane l sums outputs l, l + 32, ... over the block's chunks in chunk order
  using PG = PassGeom<RIG>;
  constexpr int SP = PG::SP, NJ = 7 + SP;
  constexpr int PART = EPASS ? PG::PART_E : PG::PART_F;
  constexpr int T_AX = EPASS ? (int)TE_AX : (int)TF_AX;
  const int lane = threadIdx.x & 31;
  if (i >= a.n_own) return;
  double* hos = a.Hos + (size_t)i * 6 * a.n_shared;
  const int c0 = a.chunk_ptr[i], c1 = a.chunk_ptr[i + 1];
  const Chunk* __restrict__ chunks = a.chunks;
  const int cam0 = (c0 < c1) ? chunks[c0].cam : 0;
  const bool one_cam = (c0 >= c1) || chunks[c1 - 1].cam == cam0;   // chunks of a block are sorted by camera
  if (!(one_cam && a.n_shared == SP)) {   // some camera columns of H_os stay empty
    for (int k = lane; k < 6 * a.n_shared; k += 32) hos[k] = 0.0;
    __syncwarp();
  }
  for (int o = lane; o < 6 * NJ; o += 32) {
    const int r = o / NJ, j = o - r * NJ;
    // element of the chunk partial this output sums
    int src;
    if (j < 6) src = TE_AA * 64 + r * 8 + j;
    else if (j == 6) src = TE_AB * 64 + r * 8 + 7;
    else if (j < 9) src = TE_AA * 64 + r * 8 + (j - 1);       // fx fy: columns 6, 7 of tile A
    else if (j < 16) src = TE_AB * 64 + r * 8 + (j - 9);      // cx .. k3: columns 0..6 of tile B
    else src = T_AX * 64 + r * 8 + (j - 16);                  // rig extrinsics
    const double* __restrict__ part = a.partials + src;
    double total = 0.0, per_cam = 0.0;
    int cam = cam0;
    for (int cb = c0; cb < c1; cb += 8) {
      // independent loads of up to 8 chunks first, then the ordered sums
      double v[8];
      int cm[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int c = min(cb + u, c1 - 1);
        v[u] = part[(size_t)c * PART];
        cm[u] = one_cam ? cam0 : chunks[c].cam;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (cb + u < c1) {
          if (cm[u] != cam) {
            if (j >= 7) hos[r * a.n_shared + cam * SP + (j - 7)] = per_cam;
            per_cam = 0.0;
            cam = cm[u];
          }
          total += v[u];
          per_cam += v[u];
        }
      }
    }
    if (j >= 7) {
      if (c0 < c1) hos[r * a.n_shared + cam * SP + (j - 7)] = per_cam;
      else if (one_cam && a.n_shared == SP) hos[r * a.n_shared + (j - 7)] = 0.0;   // unobserved block
    }
    if (j < 6) a.Hoo[(size_t)i * 36 + r * 6 + j] = total;
    if (j == 6) a.go[(size_t)i * 6 + r] = total;
  }
}

// ---------------------------------------------------------------------------
// finalize_shared: shared x shared block, gradient and cost per camera, all from
// the E-pass partials.  Stage 1: CTA (slice, camera) sums its share of the
// camera's chunk list for every partial element (fixed order).  Stage 2: the
// last stage-1 CTA of a camera to finish sums the n_slices partials in slice
// order and scatters them into H_ss / g_s / cost.
// ---------------------------------------------------------------------------
template <bool RIG>
__device__ __forceinline__ void finalize_shared_final_body(const FinalizeSharedArgs& a, int cam, double* tot);

template <bool RIG>
__device__ __forceinline__ void finalize_shared_partial_body(const FinalizeSharedArgs& a, int slice, int cam) {
  // warp w of the CTA takes chunks lo + w, lo + w + 8, ... of the slice; lane l keeps elements l, l + 32, ...
  // of the partial in registers; the 8 warp sums are then added in warp order.
  constexpr int PART = PassGeom<RIG>::PART_E, NR = (PART + 31) / 32;
  __shared__ double red[8][PART];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int32_t* __restrict__ list = a.cam_chunks_e + a.cam_ptr_e[cam];
  const double* __restrict__ part = a.part_e;
  const int n = a.cam_ptr_e[cam + 1] - a.cam_ptr_e[cam];
  const int per = (n + a.n_slices - 1) / a.n_slices;
  const int lo = slice * per, hi = min(n, lo + per);
  double acc[NR];
#pragma unroll
  for (int j = 0; j < NR; ++j) acc[j] = 0.0;
  // chunk ids of the warp first (one load per lane), so that the partial loads below do not wait on them
  for (int c0 = lo + warp; c0 < hi; c0 += 8 * 32) {
    const int cmine = c0 + 8 * lane;
    const int id_lane = (cmine < hi) ? list[cmine] : 0;
    const int cnt = min(32, (hi - c0 + 7) / 8);
#pragma unroll 4
    for (int i = 0; i < cnt; ++i) {
      const double* src = part + (size_t)__shfl_sync(0xffffffffu, id_lane, i) * PART;
#pragma unroll
      for (int j = 0; j < NR; ++j)
        if (lane + 32 * j < PART) acc[j] += src[lane + 32 * j];
    }
  }
#pragma unroll
  for (int j = 0; j < NR; ++j)
    if (lane + 32 * j < PART) red[warp][lane + 32 * j] = acc[j];
  __syncthreads();
  for (int k = threadIdx.x; k < PART; k += blockDim.x) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][k];
    a.scratch[((size_t)cam * a.n_slices + slice) * PART + k] = s;
  }
  // the last slice of the camera to arrive runs the second stage (fixed summation order: slice 0, 1, ...)
  __shared__ int is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int done = atomicAdd(a.done_count + cam, 1);
    is_last = (done == a.n_slices - 1);
    if (is_last) a.done_count[cam] = 0;   // ready for the next launch
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    finalize_shared_final_body<RIG>(a, cam, &red[0][0]);
  }
}

// element of the E-pass partial that holds the product of shared parameters i <= j (j == SP: the residual column)
template <bool RIG>
__device__ __forceinline__ int shared_src(int i, int j) {
  constexpr int SP = PassGeom<RIG>::SP;
  if (i < 2) {
    if (j < 2) return TE_AA * 64 + (6 + i) * 8 + 6 + j;
    if (j < 9) return TE_AB * 64 + (6 + i) * 8 + (j - 2);
    if (j == SP) return TE_AB * 64 + (6 + i) * 8 + 7;
    return TE_AX * 64 + (6 + i) * 8 + (j - 9);
  }
  if (i < 9) {
    if (j < 9) return TE_BB * 64 + (i - 2) * 8 + (j - 2);
    if (j == SP) return TE_BB * 64 + (i - 2) * 8 + 7;
    return TE_BX * 64 + (i - 2) * 8 + (j - 9);
  }
  if (j == SP) return TE_BX * 64 + 7 * 8 + (i - 9);   // residual row of tile B times the extrinsic columns
  return TE_XX * 64 + (i - 9) * 8 + (j - 9);
}

// second stage, run by the last first-stage CTA of a camera to finish (see finalize_fused_kernel)
template <bool RIG>
__device__ __forceinline__ void finalize_shared_final_body(const FinalizeSharedArgs& a, int cam, double* tot) {
  constexpr int SP = PassGeom<RIG>::SP, PART = PassGeom<RIG>::PART_E;
  const int tid = threadIdx.x;
  const int ns = a.n_shared;
  double* H = a.Hss;
  const int base = cam * SP;
  for (int k = tid; k < SP * ns; k += blockDim.x) H[(size_t)base * ns + k] = 0.0;
  for (int k = tid; k < PART; k += blockDim.x) {
    double s = 0.0;
    const double* src = a.scratch + (size_t)cam * a.n_slices * PART + k;
#pragma unroll 32
    for (int sl = 0; sl < a.n_slices; ++sl) s += __ldcg(src + (size_t)sl * PART);
    tot[k] = s;
  }
  __syncthreads();
  for (int k = tid; k < SP * (SP + 1); k += blockDim.x) {
    const int i = k / (SP + 1), j = k - i * (SP + 1);
    if (j == SP) {
      a.gs[base + i] = tot[shared_src<RIG>(i, SP)];
    } else {
      const double v = (i <= j) ? tot[shared_src<RIG>(i, j)] : tot[shared_src<RIG>(j, i)];
      H[(size_t)(base + i) * ns + base + j] = v;
    }
  }
  if (tid == 0) a.cost2_cam[cam] = a.robust ? tot[PassGeom<RIG>::TILES_E * 64] : tot[TE_BB * 64 + 7 * 8 + 7];
}

// one launch for the three independent reductions, longest CTAs first: the (slice, camera) first stage of
// finalize_shared, then the F side (many chunks per kept block), then the E side
constexpr int FIN_OWN_PER_CTA = 8;   // finalize_side: one warp per own block
template <bool RIG>
__global__ void __launch_bounds__(256) finalize_fused_kernel(const FinalizeSideArgs e, const FinalizeSideArgs f,
                                                             const FinalizeSharedArgs sh) {
  int i = blockIdx.x;
  const int warp = threadIdx.x >> 5;
  if (i < sh.n_slices * sh.n_cam) {
    finalize_shared_partial_body<RIG>(sh, i % sh.n_slices, i / sh.n_slices);
    return;
  }
  i -= sh.n_slices * sh.n_cam;
  const int f_ctas = (f.n_own + FIN_OWN_PER_CTA - 1) / FIN_OWN_PER_CTA;
  if (i < f_ctas) {
    finalize_side_body<RIG, false>(f, i * FIN_OWN_PER_CTA + warp);
    return;
  }
  finalize_side_body<RIG, true>(e, (i - f_ctas) * FIN_OWN_PER_CTA + warp);
}

void launch_finalize(bool rig, const FinalizeSideArgs& e, const FinalizeSideArgs& f, const FinalizeSharedArgs& sh,
                     cudaStream_t s) {
  const int grid = ceil_div(e.n_own, FIN_OWN_PER_CTA) + ceil_div(f.n_own, FIN_OWN_PER_CTA) + sh.n_slices * sh.n_cam;
  if (rig) finalize_fused_kernel<true><<<grid, 256, 0, s>>>(e, f, sh);
  else finalize_fused_kernel<false><<<grid, 256, 0, s>>>(e, f, sh);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
__global__ void expand_poses_kernel(const double* __restrict__ views, int n_views, double* __restrict__ view_x,
                                    const double* __restrict__ markers, const double* __restrict__ sizes,
                                    int n_markers, double* __restrict__ marker_x,
                                    const double* __restrict__ shared, int n_cam, int sp, double* __restrict__ ext_x) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_views) {
    expand_pose(views + (size_t)i * 6, view_x + (size_t)i * POSEX);
  } else if (i < n_views + n_markers) {
    const int j = i - n_views;
    expand_marker_pose(markers + (size_t)j * 6, marker_x + (size_t)j * POSEX);
    marker_x[(size_t)j * POSEX + PX_HS] = 0.5 * sizes[j];  // half tag size rides in the record's padding
  } else if (i < n_views + n_markers + n_cam && sp == 15) {
    const int j = i - n_views - n_markers;
    expand_pose(shared + (size_t)j * sp + 9, ext_x + (size_t)j * POSEX);
  }
}

void launch_expand_poses(const double* views, int n_views, double* view_x, const double* markers,
                         const double* sizes, int n_markers, double* marker_x, const double* shared, int n_cam, int sp,
                         double* ext_x, cudaStream_t s) {
  const int n = n_views + n_markers + n_cam;
  expand_poses_kernel<<<ceil_div(n, 128), 128, 0, s>>>(views, n_views, view_x, markers, sizes, n_markers, marker_x, shared,
                                                       n_cam, sp, ext_x);
  RCC_CUDA(cudaGetLastError());
}

}  // namespace rcc
