// Internal interface between the host-side problem object (problem.cu) and the
// CUDA kernels (assemble.cu, evaluate.cu, schur.cu).  Not part of the C ABI.
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace rcc {

// ---------------------------------------------------------------------------
// Geometry of the fused linearise+assemble kernel (K2).
//
// Every lane of a warp evaluates one tag corner (8 observation blocks x 4
// corners per warp iteration) and stages its two Jacobian rows in shared
// memory.  A staged row is cut into column tiles of 8:
//   E pass:  A = [O(6) fx fy]  B = [cx cy k1 k2 p1 p2 k3 | r]  X = [ext(6) - -] (rig)  C = [T(6) - -]
//   F pass:  A = [O(6) fx fy]  B = [cx cy k1 k2 p1 p2 k3 | r]  X = [ext(6) - -] (rig)
// O = d r / d own block (the block the pass is segmented by), T = d r / d other
// block, r = residual.  The products  tile_I^T tile_J  over the 8 residual rows
// of a block are FP64 tensor-core MMAs (mma.sync.m8n8k4.f64, k = residual row):
//   E pass accumulates AA AB BB [AX BX XX] over the chunk and emits AC (the
//   Schur off-diagonal block W = O^T T) per observation block;
//   F pass accumulates AA AB [AX].
// AA = [OO O.s01; . s01.s01], AB = [O.s2-8 g_O; s01.s2-8 g_s01], BB = [s2-8.s2-8 g_s2-8; . sum r^2].
// ---------------------------------------------------------------------------
template <bool RIG>
struct PassGeom {
  static constexpr int BPW = 8;               // observation blocks per warp iteration
  static constexpr int SP = RIG ? 15 : 9;     // shared parameters per camera
  static constexpr int WARPS = 4;             // warps (= chunks) per CTA
  // staged row stride in doubles: == 4 or 12 (mod 16) makes the MMA fragment loads (lane -> row lane%4,
  // column lane/4) hit 32 distinct banks per half-warp, and the 16-byte row stores of the 4 corner lanes
  // of a block land in 4 different bank groups
  static constexpr int RS_E = RIG ? 36 : 28;
  static constexpr int RS_F = RIG ? 28 : 20;
  static constexpr int COL_B = 8, COL_X = 16, COL_C = RIG ? 24 : 16;
  static constexpr int TILES_E = RIG ? 6 : 3;  // accumulated 8x8 tiles per chunk
  static constexpr int TILES_F = RIG ? 3 : 2;
  static constexpr int PART_E = TILES_E * 64 + 8;  // doubles per chunk partial; tail slot 0 = robust cost
  static constexpr int PART_F = TILES_F * 64;
};
enum TileE : int { TE_AA = 0, TE_AB = 1, TE_BB = 2, TE_AX = 3, TE_BX = 4, TE_XX = 5 };
enum TileF : int { TF_AA = 0, TF_AB = 1, TF_AX = 2 };

// one chunk of a pass: `count` consecutive sorted observation blocks that share
// the own block index and the camera
struct Chunk {
  int32_t own;
  int32_t cam;
  int32_t start;
  int32_t count;
};

struct AssembleArgs {
  // sorted observation blocks of this pass
  const int32_t* oth;     // [n] index of the other 6-dof block
  const double* pix;      // [n*8]
  const Chunk* chunks;    // [n_chunks]
  int32_t n_chunks;       // chunks this launch covers
  const int32_t* chunk_list;  // optional: the launch covers chunks chunk_list[0 .. n_chunks) instead of 0 .. n_chunks
  // parameters
  const double* view_x;   // expanded poses [n_views*24]
  const double* marker_x; // [n_markers*24]
  const double* ext_x;    // [n_cam*24] (rig)
  const double* shared;   // [n_cam*SP]
  // outputs
  double* partials;       // [n_chunks * PART_E|PART_F]: 8x8 tiles, element (m, n) at m * 8 + n
  double* W;              // [n*36] (E pass only) row-major 6x6: rows own, cols other
  int32_t* fail_flag;     // set to 1 on depth <= 0 / non-finite residual
  int32_t loss;           // 0 trivial, 1 Huber, 2 Cauchy (per tag residual block)
  double loss_a2;         // squared loss scale
};

// K2: fused residual + Jacobian + J^T J tiles.  own_is_view tells which pose
// table the segment owner indexes.
void launch_assemble(bool rig, bool epass, bool own_is_view, const AssembleArgs& a, cudaStream_t s);

// per-own-block reduction of the chunk partials
struct FinalizeSideArgs {
  const double* partials;
  const Chunk* chunks;
  const int32_t* chunk_ptr;  // [n_own+1] chunks of own block i
  int32_t n_own;
  int32_t n_shared;          // n_cam * SP
  double* Hoo;               // [n_own*36]
  double* go;                // [n_own*6]
  double* Hos;               // [n_own*6*n_shared]  (zeroed by the kernel)
};

// per-camera reduction of the shared x shared tiles, gradient and cost
struct FinalizeSharedArgs {
  const double* part_e;         // the shared x shared tiles all come from the E pass
  const int32_t* cam_chunks_e;  // chunk ids grouped by camera
  const int32_t* cam_ptr_e;     // [n_cam+1]
  int32_t n_cam;
  int32_t n_shared;
  double* Hss;                  // [n_shared*n_shared] block diagonal (zeroed by the kernel)
  double* gs;                   // [n_shared]
  double* cost2_cam;            // [n_cam] sum r^2 per camera
  double* scratch;              // [n_cam * n_slices * PART_E] first-stage partial tiles
  int32_t* done_count;          // [n_cam] first-stage CTAs finished (zero between launches)
  int32_t robust;               // 1: cost = tail slot (sum rho), else BB[7][7] (sum r^2)
  int32_t n_slices;             // first-stage CTAs per camera (fin_slices)
};
// First-stage CTAs per camera of finalize_shared: enough that the first stage of all cameras together puts two
// CTAs on every SM (one camera would otherwise read its E-pass partials through a fraction of the GPU), and at
// least 64.
inline int fin_slices(int n_sm, int n_cam) {
  const int per_cam = (2 * n_sm + n_cam - 1) / n_cam;
  return per_cam > 64 ? per_cam : 64;
}
// E side, F side and both stages of the shared reduction in one launch
void launch_finalize(bool rig, const FinalizeSideArgs& e, const FinalizeSideArgs& f, const FinalizeSharedArgs& sh,
                     cudaStream_t s);

// pose expansion: rvec,t -> R, Jr, t
void launch_expand_poses(const double* views, int n_views, double* view_x, const double* markers,
                         const double* sizes, int n_markers, double* marker_x, const double* shared, int n_cam, int sp,
                         double* ext_x, cudaStream_t s);

// ---------------------------------------------------------------------------
// K1 / K6: materialised evaluation and cost-only evaluation
// ---------------------------------------------------------------------------
struct EvalArgs {
  int64_t n;
  const int32_t* view_idx;  // [n] per sorted block
  const int32_t* marker_idx;
  const int32_t* cam;
  const int32_t* orig;      // caller position of sorted block
  const double* pix;
  const double* view_x;
  const double* marker_x;
  const double* ext_x;
  const double* shared;
  // outputs (caller order; any may be null)
  double* residuals;        // [n*8]
  double* jac_intr;         // [n*8*4]
  double* jac_dist;         // [n*8*5]
  double* jac_view;         // [n*8*6]
  double* jac_marker;       // [n*8*6]
  double* jac_ext;          // [n*8*6]
  double* cost2_partials;   // [grid] sum rho(||r_block||^2) per CTA
  int32_t* fail_flag;
  int32_t loss;
  double loss_a2;
  // chunk view of the same E-sorted blocks (materialising kernel: one warp per chunk)
  const Chunk* chunks;
  int32_t n_chunks;
  const int32_t* oth;       // [n] other 6-dof block of each sorted block (own block comes from the chunk)
  int32_t own_is_view;
};
int eval_grid(int64_t n);   // CTAs launch_evaluate / launch_cost will use
void launch_evaluate(bool rig, bool want_jac, const EvalArgs& a, cudaStream_t s);
// number of cost partials launch_evaluate writes (want_jac: one per chunk; else one per CTA)
int eval_partials(bool want_jac, const EvalArgs& a);
void launch_cost(bool rig, const EvalArgs& a, cudaStream_t s);
// deterministic sum of n doubles -> out[0] (single CTA)
void launch_sum(const double* in, int64_t n, double* out, double scale, cudaStream_t s);

// ---------------------------------------------------------------------------
// K3: Schur complement
// ---------------------------------------------------------------------------
// LM damping of one parameter from its diag(J^T J) entry h (Ceres: D^2 = clamp(diag) / radius).  With Jacobi
// scaling the clamp applies to the scaled column, s = 1 / (1 + sqrt(h)), and the result is mapped back to the
// unscaled parameter:  clamp(s^2 h) / (radius s^2).
__host__ __device__ inline double lm_diagonal(double h, double radius, double min_diag, double max_diag, int jacobi) {
  if (!jacobi) return fmin(fmax(h, min_diag), max_diag) / radius;
  const double s = 1.0 / (1.0 + sqrt(fmax(h, 0.0)));
  return fmin(fmax(h * s * s, min_diag), max_diag) / (radius * s * s);
}

struct SchurPrepArgs {
  int32_t n_e;
  int32_t n_shared;
  int32_t n_bb;                  // border blocks per E block: ceil((n_shared+1)/6)
  const double* Hee;             // [n_e*36]
  const double* ge;              // [n_e*6]
  const double* Hes;             // [n_e*6*n_shared]
  const uint8_t* e_const;        // [n_e]
  const int32_t* row_ptr;        // [n_e+1] pairs of row e
  const int32_t* pair_mptr;      // [n_pairs+1]
  const int32_t* pair_members;   // sorted-observation positions
  const int32_t* row_pos0;       // [n_e] first sorted position of row e when its pairs have one member each at
                                 // consecutive positions (then W of pair p0+i is W[row_pos0 + i]); -1 otherwise
  const double* W;               // [n_obs*36]
  double radius, min_diag, max_diag;
  int32_t jacobi;                // LM diagonal on the Jacobi-scaled columns (lm_diagonal())
  double* Linv;                  // [n_e*36] row-major lower-triangular inverse of chol(Hee + D)
  double* Y;                     // [n_pairs*36] column-major 6x6 blocks  L^-1 W
  double* Yb;                    // [n_e*n_bb*36] column-major blocks L^-1 [Hes | ge | 0]
  double* d2e;                   // [n_e*6] damping actually applied
  int32_t* pivot_fail;           // nullable: set to 1 when a free block's pivot of chol(Hee + D) is not positive
                                 // (the factorisation clamps it to 1e-300 and carries on)
};
void launch_schur_prep(const SchurPrepArgs& a, cudaStream_t s);

// Column tiling of the block-sparse SYRK: the kept blocks are cut into sub-tiles of SYRK_SUBTILE consecutive
// blocks (the granularity of tile_ptr; one warp each), and one CTA of schur_syrk_kernel covers a column tile of
// SYRK_CTA_SUBTILES neighbouring sub-tiles.
constexpr int SYRK_SUBTILE = 32;
constexpr int SYRK_CTA_SUBTILES = 2;

struct SchurSyrkArgs {
  int32_t n_f, n_e;
  int32_t n_shared, n_bb;
  int32_t n_tiles;               // ceil(n_f / SYRK_SUBTILE) sub-tiles
  int32_t ld;                    // row stride of S
  int32_t n_ctas;                // entries of cta_list
  const int32_t* col_ptr;        // [n_f+1]
  const int32_t* col_pair;       // pair ids of column f, ascending e
  const int32_t* pair_e;         // [n_pairs]
  const int32_t* pair_f;         // [n_pairs]
  const int32_t* tile_ptr;       // [n_e*(n_tiles+1)]
  const int32_t* cta_list;       // [n_ctas][2] (f, column tile) of schur_syrk_kernel, heaviest first
  const double* Y;
  const double* Yb;
  const double* Hff;             // [n_f*36]
  const double* gf;              // [n_f*6]
  const double* Hfs;             // [n_f*6*n_shared]
  double* S;                     // [(n + extra rows) * ld]
};
void launch_schur_syrk(const SchurSyrkArgs& a, cudaStream_t s);     // kept x kept blocks (upper triangle)
void launch_schur_border(const SchurSyrkArgs& a, cudaStream_t s);   // kept x [shared | rhs] strip

struct SchurSharedArgs {
  int32_t n_e, n_f, n_shared, n_bb, ld;
  const double* Yb;
  const double* Hss;
  const double* gs;
  double* scratch;               // [SHARED_SLICES * (6 n_bb)^2]
  double* S;
};
constexpr int SHARED_SLICES = 128;
void launch_schur_shared(const SchurSharedArgs& a, cudaStream_t s);

// extra rows appended to S for the all-reduce: [hdiag (n) | gF (n) | scalars (8)]
struct ReducedTailArgs {
  int32_t n_f, n_shared, ld;
  const double* Hff;
  const double* gf;
  const double* Hss;
  const double* gs;
  const double* cost2_cam;  // [n_cam]
  int32_t n_cam;
  double* S;                // tail starts at S + n*ld
};
void launch_reduced_tail(const ReducedTailArgs& a, cudaStream_t s);

struct MaskArgs {
  int32_t n, ld;
  double radius, min_diag, max_diag;
  int32_t jacobi;
  const int32_t* const_idx;  // reduced-system indices held constant
  int32_t n_const;
  double* S;                 // damping added to the diagonal, constants masked
  double* rhs;               // [n]  = -b  (solve S x = rhs)
  double* d2f;               // [n] damping applied (0 on constants)
  double* gF;                // [n] masked gradient copy
};
void launch_mask_damp(const MaskArgs& a, cudaStream_t s);

struct BacksubArgs {
  int32_t n_e, n_f, n_shared, n_bb;
  const int32_t* row_ptr;
  const int32_t* pair_f;
  const double* Y;
  const double* Yb;
  const double* Linv;
  const double* ge;
  const double* d2e;
  const double* delta_F;  // [6 n_f + n_shared]
  const double* x_e;      // current E parameters [n_e*6]
  const int32_t* e_count; // observations per E block on this rank
  double* delta_e;        // [n_e*6]
  double* partials;       // [n_e*4]: mcc, |d|^2, |x|^2, 0 per E block
};
void launch_backsub(const BacksubArgs& a, cudaStream_t s);

// Parameter covariance from the inverse of the undamped reduced system.  Sinv: S^-1 in the row-major upper triangle
// of the reduced buffer (rows and columns of constants zero).  Partner k of row e is pair row_ptr[e] + k (its kept
// block f, record Y) for k < m_e, and border block k - m_e (shared columns 6 (k - m_e) ..., record Yb, the g_e and
// pad columns left out) after it.
struct CovArgs {
  int32_t n_e, n_f, n_shared, n_bb;
  int32_t n, ld;                 // reduced size 6 n_f + n_shared, row stride of the buffer
  const int32_t* row_ptr;
  const int32_t* pair_f;
  const double* Y;               // undamped schur_prep outputs
  const double* Yb;
  const double* Linv;
  const double* Sinv;
  double* cov_e;                 // [n_e*36] row-major
  double* cov_f;                 // [n_f*36] row-major
  double* cov_s;                 // [n_shared*n_shared] row-major
};
// Cov(e) = L_e^-T (I + Y_e S^-1 Y_e^T) L_e^-1 for every eliminated block (Y_e = the 6 x n row of partners)
void launch_cov_eliminated(const CovArgs& a, cudaStream_t s);
// the kept 6 x 6 diagonal blocks and the shared block of S^-1, both triangles filled
void launch_cov_kept(const CovArgs& a, cudaStream_t s);

// Cross-covariance blocks (rcc_ba_covariance_blocks).  A side of a pair is an eliminated block e, whose items are its
// K_e = m_e + n_bb partners (records as in CovArgs), or a kept or shared block: one item, the identity record on its
// reduced columns [g, g + w).  Each pair is canonicalised on the host so that side b has at least as many items as
// side a, and the kernel computes X = sum_{k in a} sum_{l in b} C_ak S^-1[k, l] C_bl^T; then
//     Cov(a, b) = delta_ab L_a^-T L_a^-1 + P_a X P_b^T,   P = -L_e^-T for an eliminated side, I otherwise.
struct CovPairDesc {
  int32_t e_a, e_b;              // eliminated block of side a / b, or -1 for a kept or shared block
  int32_t g_a, w_a, g_b, w_b;    // kept or shared side: first reduced index and width (4, 5 or 6)
  int32_t item0, n_items;        // its work items [item0, item0 + n_items) of its launch, in summation order
  int32_t rows, cols;            // Cov(a, b) is rows x cols (6 for an eliminated side)
  int32_t transpose;             // 1: the request was (b, a), written as the cols x rows transpose
  int32_t pad;
};
// one work item: items [k0, k0 + COV_PAIR_CHUNK) of side a against the tile [l0, l0 + 32) of side b
struct CovPairItem { int32_t pair, k0, l0; };
constexpr int COV_PAIR_CHUNK = 256;
struct CovPairsArgs {
  CovArgs m;                     // sizes, partner lists, Y / Yb / Linv and S^-1 (its outputs unused)
  const CovPairDesc* pairs;      // every requested pair; this launch covers [pair_begin, pair_begin + n_pairs)
  const CovPairItem* items;      // the items of those pairs (item0 counts from here)
  int32_t pair_begin, n_pairs, n_items;
  double* partial;               // [n_items*36]: X of each item, row-major 6 x 6
  double* out;                   // [all pairs*36]: Cov of each request at the start of its 36-double slot
};
// partials of every item, then each pair's sum over its items in item order and the output (no atomics)
void launch_cov_pairs(const CovPairsArgs& a, cudaStream_t s);

// F-side model-cost-change / norms: out[0..2] = mcc_F, |dF|^2, |xF|^2
void launch_f_stats(const double* gF, const double* d2f, const double* delta_F, const double* x_f, const double* x_s,
                    int32_t n_f, int32_t n_shared, double* out3, cudaStream_t s);
// reduce the per-E-block partials: out[0..2]
void launch_e_stats(const double* partials, int32_t n_e, double* out3, cudaStream_t s);

// a column band of the reduced buffer for the overlapped reduction: rows [0, min(n_rows, c1)), columns
// [max(row, c0), c1) of each row (the live part of the upper triangle inside the band), rows back to back in `packed`
size_t packed_band_doubles(int32_t n_rows, int32_t c0, int32_t c1);
void launch_pack_band(double* S, int32_t ld, int32_t n_rows, int32_t c0, int32_t c1, double* packed, bool to_packed,
                      cudaStream_t s);
// x_new = x + delta (6-dof blocks and shared block)
void launch_apply(const double* x, const double* d, double* out, int64_t n, cudaStream_t s);
// make a symmetric full matrix out of the upper triangle (parity read-back only)
void launch_symmetrize(double* S, int32_t n, int32_t ld, cudaStream_t s);
// caller's pixel blocks (T = double, int32_t or int16_t) -> both sorted FP64 layouts, for sorted blocks g in [0, n):
// e_pix[g] = (double) src[orig ? orig[g] : g] and f_pix[f_inv[g]] = e_pix[g].  src == nullptr: e_pix already holds
// the blocks (an FP64 upload copied straight into it) and is only read, never written again.  src must not alias
// e_pix or f_pix otherwise.  Called on a piece of the sorted order, e_pix and f_inv point at the piece's first block.
template <typename T>
void launch_load_pixels(const T* src, const int32_t* orig, double* e_pix, const int32_t* f_inv, double* f_pix,
                        int64_t n, cudaStream_t s);
// write a scratch buffer (L2 flush)
void launch_fill(double* p, int64_t n, double v, cudaStream_t s);
// FP64 FMA throughput microbenchmark kernel; returns number of FMAs issued
double launch_fp64_peak(int iters, double* sink, cudaStream_t s);

}  // namespace rcc
