// Host-side problem object behind the opaque C handle.
#pragma once

#include <cublas_v2.h>
#include <cusolverDn.h>
#include <nccl.h>

#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "dense.h"
#include "kernels.h"

namespace rcc {

enum Stage : int {
  ST_EXPAND = 0, ST_ASSEMBLE_E, ST_ASSEMBLE_F, ST_FINALIZE, ST_SCHUR_PREP, ST_SCHUR_SYRK, ST_SCHUR_SHARED,
  ST_ALLREDUCE, ST_MASK, ST_CHOLESKY, ST_BACKSUB, ST_COST, ST_EVALUATE, ST_H2D, ST_INVERSE, ST_COVARIANCE,
  ST_COV_EXTRACT, ST_COUNT
};
const char* stage_name(int s);

struct StageTimer {
  struct Pending { int stage; cudaEvent_t a, b; };
  bool on = false;
  std::vector<Pending> pending;
  std::vector<cudaEvent_t> pool;
  double ms[ST_COUNT] = {0};
  int64_t launches[ST_COUNT] = {0};
  cudaEvent_t get();
  void begin(int stage, cudaStream_t s);
  void end(cudaStream_t s);
  void collect();  // requires the stream to be synchronised
  void reset();
  ~StageTimer();
};

}  // namespace rcc

struct rcc_ba_problem {
  rcc_ba_options opt{};
  bool rig = false;
  int sp = 9, n_cam = 1, n_shared = 9;
  int fin_slices = 64;   // first-stage CTAs per camera of the shared-parameter finalize (kernels.h: fin_slices)
  bool elim_view = true;
  int n_views = 0, n_markers = 0, n_e = 0, n_f = 0;
  int n_bb = 2, n_red = 0, ld = 0;
  int64_t n_obs = 0, n_pairs = 0;
  int n_tiles = 1, n_syrk_ctas = 0;
  // overlapped reduction (multi-rank): the SYRK work list is cut into groups of column tiles; group g covers the
  // CTAs [syrk_grp_cta[g], syrk_grp_cta[g+1]) and the columns [syrk_grp_col[g], syrk_grp_col[g+1]) of S
  static constexpr int SYRK_GROUPS = 8;
  int n_syrk_groups = 1;
  int syrk_grp_cta[SYRK_GROUPS + 1] = {0};
  int syrk_grp_col[SYRK_GROUPS + 1] = {0};
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t ev_grp[SYRK_GROUPS + 1] = {nullptr};
  bool reduced_in_schur = false;     // S already holds the sum over the ranks (rcc_ba_schur did the all-reduce)
  int n_chunks_e = 0, n_chunks_f = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  // fork/join side stream: small kernels that only depend on the previous stage run beside the big one
  cudaStream_t side_stream = nullptr, side_stream2 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // piecewise pixel upload (rcc_ba_update_pixels when the caller order is the E-sorted order): the H2D
  // copy runs on the side stream in PIX_PIECES pieces cut at chunk boundaries, and the next linearize
  // starts the E pass of a piece as soon as that piece has landed
  static constexpr int PIX_PIECES = 8;
  // from this many observation blocks on, an upload is cut into PIX_PIECES pieces (below: 4) and linearize runs the
  // F pass of each piece as it lands; below it, four more launches cost more than they hide
  static constexpr int64_t LARGE_UPLOAD_BLOCKS = 4000000;
  bool pix_identity = false;         // e_orig is the identity permutation
  bool pix_pending = false;          // pieces in flight on the copy streams (each piece also scatters itself into f_pix)
  int piece_chunk[PIX_PIECES + 1] = {0};
  int64_t piece_block[PIX_PIECES + 1] = {0};
  cudaEvent_t ev_piece[PIX_PIECES] = {nullptr};
  std::string err;
  int64_t launch_count = 0;

  // parameters: current (x) and candidate (xc)
  rcc::DBuf<double> views, markers, sizes, shared, views_c, markers_c, shared_c;
  rcc::DBuf<double> view_x, marker_x, ext_x, view_xc, marker_xc, ext_xc;
  bool expanded_valid = false;
  std::vector<uint8_t> c_view, c_marker, c_intr, c_dist, c_ext;
  bool const_dirty = true;

  // observation blocks, E-sorted and F-sorted
  rcc::DBuf<int32_t> e_own, e_oth, e_cam, e_orig, f_oth, f_inv, e_chunk_ptr, f_chunk_ptr;   // f_inv: E-sorted -> F-sorted position
  rcc::DBuf<double> e_pix, f_pix;
  rcc::DBuf<char> staging;           // caller's pixels on the device, of any element type, before launch_load_pixels
  rcc::DBuf<rcc::Chunk> e_chunks, f_chunks;
  rcc::DBuf<int32_t> cam_chunks_e, cam_ptr_e, cam_chunks_f, cam_ptr_f;
  rcc::DBuf<int32_t> f_piece_list;   // F-pass chunk ids grouped by upload piece
  int f_piece_ptr[PIX_PIECES + 1] = {0};
  std::vector<int32_t> row_ptr_h;    // row_ptr on the host (rcc_ba_covariance_blocks plans its work from it)
  rcc::DBuf<int32_t> row_ptr, pair_e, pair_f, pair_mptr, pair_members, row_pos0, col_ptr, col_pair, tile_ptr, syrk_ctas, e_count;
  rcc::DBuf<uint8_t> e_const;

  // linearisation products
  rcc::DBuf<double> fin_scratch, part_e, part_f, W, Hee, ge, Hes, Hff, gf, Hfs, Hss, gs, cost2_cam;
  // Schur / step
  rcc::DBuf<double> Linv, Y, Yb, d2e, S, shared_scratch, rhs, d2f, gFm, delta_F, delta_e, bs_partials, stats;
  rcc::DBuf<int32_t> const_idx, fail_flag, fin_done;
  int n_const = 0;
  double radius_used = 0.0;
  // evaluation outputs
  rcc::DBuf<double> o_res, o_ji, o_jd, o_jv, o_jm, o_jx, cost_partials, scalar;

  cusolverDnHandle_t solver = nullptr;
  cublasHandle_t blas = nullptr;
  rcc::DBuf<double> potrf_work, packed_S;   // packed_S: the packed column bands of the overlapped reduction (multi-rank)
  rcc::DBuf<int> dev_info;
  int potrf_lwork = 0;
  // rcc_ba_covariance: the eliminated / kept / shared blocks, diag(S) before the factorisation, and the status words
  // [potrf info, potri info, H_ee pivot, S pivot]
  rcc::DBuf<double> cov_e, cov_f, cov_s, cov_diag;
  rcc::DBuf<int32_t> cov_info;
  // rcc_ba_covariance_blocks: the canonical pairs, their work items, the items' partials and the outputs
  rcc::DBuf<rcc::CovPairDesc> cov_desc;
  rcc::DBuf<rcc::CovPairItem> cov_items;
  rcc::DBuf<double> cov_partial, cov_out;

  // reduced solve: 0 = cusolverDnDpotrf replicated on every rank, 1 = dense.cu on this rank, 2 = dense.cu with the
  // block columns distributed over the ranks (RCC_CHOLESKY = cusolver | own | dist | auto)
  int chol_mode = -1;                    // -1: not resolved yet
  rcc::DBuf<double> trsv_inv;            // K5d: inverses of the 32 x 32 diagonal blocks of the factor
  rcc::DBuf<int> trsv_flags;
  rcc::CholDriver chol;

  ncclComm_t comm = nullptr;
  int rank = 0, n_ranks = 1;

  bool have_obs = false, linearized = false, schur_done = false, step_ready = false, cand_ready = false;
  double min_diag = 1e-6, max_diag = 1e32;
  int jacobi = 0;                    // Jacobi column scaling of the LM diagonal
  int loss = 0;
  double loss_scale = 1.0;
  rcc::StageTimer timer;
  rcc::DBuf<double> flush_buf;

  // pinned host scratch for small read-backs
  double* h_pinned = nullptr;
  // pinned staging slots for parameter uploads: the setters copy the caller's buffer here and return
  // without a stream synchronisation; a slot is reused only after its previous H2D copy has completed
  struct HostSlot { void* p = nullptr; size_t cap = 0; cudaEvent_t ev = nullptr; bool busy = false; };
  HostSlot hslot[5];

  ~rcc_ba_problem();
};
