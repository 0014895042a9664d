/* rcc_ba.h -- C ABI of the B200-native bundle-adjustment hot path.
 *
 * Drop-in boundary (SURVEY.md 8b): the path sits where the reference's missing
 * "Milestone 3" optimiser would call Ceres -- between the initial guesses that
 * real_preprocessing/src/camera_pose.cpp:83-129 writes and the reader at
 * real_preprocessing/src/opt_visualization.cpp:46-66,118-138.  The contract it
 * replaces is Ceres's public evaluation interface
 *     bool CostFunction::Evaluate(double const* const* parameters,
 *                                 double* residuals, double** jacobians) const
 * (not in /root/reference -- the snapshot holds no optimiser; stated from the
 * published Ceres API, unverified here) plus the linear-algebra that follows it
 * inside Ceres (normal equations, Schur complement, LM step).
 *
 * Rules: extern "C", opaque handle, plain pointers and sizes, int status
 * return, no exceptions or C++ types across the boundary.  The caller owns
 * every host buffer (copied in/out synchronously); the library owns all device
 * memory.  One handle = one CUDA device + one stream; a handle is not
 * thread-safe, distinct handles are independent.  There is no CPU fallback:
 * every compute entry point fails with RCC_CUDA_ERROR when no sm_100 device is
 * usable.
 *
 * Parameter blocks (FP64), conventions cited to camera_pose.cpp:
 *   intr[4] = fx fy cx cy   (K[0] K[4] K[2] K[5], :61-62)
 *   dist[5] = k1 k2 p1 p2 k3 (:39,63-64)
 *   view[6] = Rodrigues rvec, t of world_T_camera (:88-98)   [rig: world_T_body]
 *   marker[6] = rvec, t of world_T_target (:111-121)
 *   ext[6]  = rvec, t of body_T_cam   (rig model only; not in the reference)
 * Observation block = one tag in one frame = 4 corners (bl br tr tl,
 * :123-126) = 8 residuals  u0 v0 u1 v1 u2 v2 u3 v3  (corner_detections.cpp:34-37).
 */
#ifndef RCC_BA_H
#define RCC_BA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rcc_ba_problem rcc_ba_problem; /* opaque */

enum rcc_status {
  RCC_OK = 0,
  RCC_BAD_ARG = 1,
  RCC_CUDA_ERROR = 2,
  RCC_NCCL_ERROR = 3,
  RCC_EVAL_FAILED = 4, /* non-finite residual or corner behind the camera (== Ceres Evaluate()==false) */
  RCC_NOT_SPD = 5,     /* reduced system not positive definite */
  RCC_NOT_READY = 6,   /* call order violated (e.g. schur before linearize) */
  RCC_SOLVER_ERROR = 7
};

enum rcc_model { RCC_MODEL_SINGLE = 0, RCC_MODEL_RIG = 1 };
enum rcc_eliminate { RCC_ELIM_AUTO = 0, RCC_ELIM_VIEWS = 1, RCC_ELIM_MARKERS = 2 };
enum rcc_loss { RCC_LOSS_TRIVIAL = 0, RCC_LOSS_HUBER = 1, RCC_LOSS_CAUCHY = 2 };
enum rcc_block_kind { RCC_BLOCK_VIEW = 0, RCC_BLOCK_MARKER = 1, RCC_BLOCK_INTR = 2, RCC_BLOCK_DIST = 3, RCC_BLOCK_EXT = 4 };

typedef struct {
  int32_t model;      /* rcc_model */
  int32_t n_views;    /* views (single) or body poses (rig) */
  int32_t n_markers;
  int32_t n_cameras;
  int64_t n_obs_blocks;
  int32_t device;     /* CUDA device ordinal */
  int32_t eliminate;  /* rcc_eliminate: which 6-dof block set the Schur complement removes */
} rcc_ba_options;

typedef struct {
  int32_t max_iterations;         /* 50 */
  double initial_radius;          /* 1e4   (Ceres initial_trust_region_radius) */
  double max_radius;              /* 1e16 */
  double min_relative_decrease;   /* 1e-3 */
  double function_tolerance;      /* 1e-6 */
  double gradient_tolerance;      /* 1e-10 */
  double parameter_tolerance;     /* 1e-8 */
  double min_diagonal;            /* 1e-6 */
  double max_diagonal;            /* 1e32 */
  int32_t verbose;
  int32_t jacobi_scaling;         /* 1 (Ceres default): the LM diagonal is formed on the Jacobian with columns scaled by
                                   * 1 / (1 + ||column||), i.e. min/max_diagonal clamp s^2 diag(J^T J) instead of
                                   * diag(J^T J); the step is returned in unscaled parameters */
} rcc_lm_options;

typedef struct {
  int32_t iterations;             /* LM iterations run (accepted + rejected) */
  int32_t accepted;
  int32_t termination;            /* 0 max-iter, 1 function tol, 2 gradient tol, 3 parameter tol, 4 failure */
  double initial_cost;
  double final_cost;
  double final_gradient_max;
  double final_radius;
  double total_ms;                /* device time of the whole solve */
  double linearize_ms, schur_ms, allreduce_ms, solve_ms, backsub_ms, cost_ms; /* per-stage device time, summed */
} rcc_lm_summary;

/* ---- lifetime ---------------------------------------------------------- */
int rcc_ba_create(const rcc_ba_options* opt, rcc_ba_problem** out);
void rcc_ba_destroy(rcc_ba_problem* p);
const char* rcc_ba_last_error(const rcc_ba_problem* p); /* never NULL */
void rcc_lm_default_options(rcc_lm_options* o);
/* library / build info: returns a static string "rcc_ba <version> sm_100a ..." */
const char* rcc_ba_version(void);
/* use the caller's CUDA stream (a cudaStream_t cast to void*) instead of the handle's own */
int rcc_ba_set_stream(rcc_ba_problem* p, void* cuda_stream);

/* ---- problem setup (host AoS in, Ceres-style contiguous double[k] blocks) ----
 * The parameter setters copy the caller's array into an internal pinned slot and return without a stream
 * synchronisation: the array may be reused as soon as the call returns. */
int rcc_ba_set_intrinsics(rcc_ba_problem* p, const double* intr /*n_cam x 4*/, const double* dist /*n_cam x 5*/);
int rcc_ba_set_rig_extrinsics(rcc_ba_problem* p, const double* ext /*n_cam x 6*/);
int rcc_ba_set_view_poses(rcc_ba_problem* p, const double* views /*n_views x 6*/);
int rcc_ba_set_marker_poses(rcc_ba_problem* p, const double* markers /*n_markers x 6*/);
int rcc_ba_set_marker_sizes(rcc_ba_problem* p, const double* sizes /*n_markers*/);
/* cam_idx may be NULL (all camera 0).  pixels: n_obs_blocks x 8.  Sorts the blocks
 * by eliminated-block owner and builds the segment / chunk / Schur index tables. */
int rcc_ba_set_observations(rcc_ba_problem* p, const int32_t* view_idx, const int32_t* marker_idx,
                            const int32_t* cam_idx, const double* pixels);
/* replace the pixel coordinates only (same indices, caller order).  Asynchronous: `pixels` must stay
 * valid until the next call that returns results (linearize with a cost pointer, evaluate, any getter).
 * When the caller order is the sorted order (blocks listed per eliminated block) the copy runs on a side
 * streams in 8 pieces (each piece also lands in the second sorted copy) and the next rcc_ba_linearize starts the E pass of a piece as soon as it has landed:
 * call the parameter setters BEFORE update_pixels so that they do not queue behind it.  Otherwise: one
 * H2D copy plus a device-side permutation into the sorted layouts. */
int rcc_ba_update_pixels(rcc_ba_problem* p, const double* pixels /*n_obs_blocks x 8*/);
/* Integer pixel corners -- the reference's own observation format: corner_detections.cpp:53-54 truncates the
 * detector's corners to int before writing them, camera_pose.cpp:135-142 parses them back with .as<int>().
 * 16 bits are lossless for any image up to 32 767 px; the conversion to FP64 happens on the device, so an update
 * ships 16 bytes per tag over PCIe instead of 64 and the results are bit-identical to the FP64 entry points
 * fed with the same integers.  Same ordering / asynchrony contract as rcc_ba_update_pixels. */
int rcc_ba_set_observations_i16(rcc_ba_problem* p, const int32_t* view_idx, const int32_t* marker_idx,
                                const int32_t* cam_idx, const int16_t* pixels /*n_obs_blocks x 8*/);
int rcc_ba_set_observations_i32(rcc_ba_problem* p, const int32_t* view_idx, const int32_t* marker_idx,
                                const int32_t* cam_idx, const int32_t* pixels /*n_obs_blocks x 8*/);
int rcc_ba_update_pixels_i16(rcc_ba_problem* p, const int16_t* pixels /*n_obs_blocks x 8*/);
/* hold a parameter block constant (the gauge: world tag, camera_pose.cpp:71-80) */
int rcc_ba_set_constant(rcc_ba_problem* p, int32_t block_kind, int32_t index, int32_t is_constant);

/* robust loss rho(s) on s = ||r||^2 of each tag's 8-residual block (Ceres LossFunction semantics:
 * HuberLoss(scale) / CauchyLoss(scale), scale in pixels); the reported cost becomes 0.5 * sum rho(s) */
int rcc_ba_set_loss(rcc_ba_problem* p, int32_t loss, double scale);

int rcc_ba_get_intrinsics(rcc_ba_problem* p, double* intr, double* dist);
int rcc_ba_get_rig_extrinsics(rcc_ba_problem* p, double* ext);
int rcc_ba_get_view_poses(rcc_ba_problem* p, double* views);
int rcc_ba_get_marker_poses(rcc_ba_problem* p, double* markers);

/* ---- cost functor evaluation (materialise mode, Ceres Evaluate layout) ----
 * Outputs are in the caller's observation order.  Any pointer may be NULL.
 *   residuals   : n_obs_blocks x 8
 *   jac_intr    : n_obs_blocks x 8 x 4   row-major per block  (= jacobians[0])
 *   jac_dist    : n_obs_blocks x 8 x 5                        (= jacobians[1])
 *   jac_view    : n_obs_blocks x 8 x 6                        (= jacobians[2])
 *   jac_marker  : n_obs_blocks x 8 x 6                        (= jacobians[3])
 *   jac_ext     : n_obs_blocks x 8 x 6   (rig only)           (= jacobians[4])
 * Returns RCC_EVAL_FAILED (outputs still written) if any corner has depth <= 0
 * or a non-finite residual. */
int rcc_ba_evaluate(rcc_ba_problem* p, int32_t want_jacobians, double* cost, double* residuals,
                    double* jac_intr, double* jac_dist, double* jac_view, double* jac_marker, double* jac_ext);
/* same kernel, outputs stay in device memory (timed by bench.py); cost may be NULL */
int rcc_ba_evaluate_device(rcc_ba_problem* p, int32_t want_jacobians, double* cost);

/* ---- normal equations, Schur complement, LM step ------------------------- */
/* residual + Jacobian + J^T J / J^T r blocks, fused (no Jacobian in HBM) */
int rcc_ba_linearize(rcc_ba_problem* p, double* cost /*may be NULL: no host sync*/);
/* damped Schur complement into the reduced system.  With a communicator attached (rcc_ba_comm_init) this is a
 * COLLECTIVE call: the ranks' partial systems are summed band by band behind the computation, and the reduced system
 * every rank holds on return is the sum over all ranks.  Uses the LM diagonal bounds and the Jacobi-scaling flag of
 * the last rcc_ba_solve / rcc_ba_set_lm_diagonal (defaults 1e-6, 1e32, no scaling). */
int rcc_ba_schur(rcc_ba_problem* p, double radius);
int rcc_ba_set_lm_diagonal(rcc_ba_problem* p, double min_diagonal, double max_diagonal, int32_t jacobi_scaling);
/* constant mask + Cholesky (distributed over the ranks for large systems) + back-substitution.
 * model_cost_change may be NULL. */
int rcc_ba_solve_step(rcc_ba_problem* p, double* model_cost_change, double* step_norm, double* x_norm);
/* cost at x + step (all-reduced over ranks) */
int rcc_ba_candidate_cost(rcc_ba_problem* p, double* cost);
int rcc_ba_accept_step(rcc_ba_problem* p);
/* whole Levenberg-Marquardt loop */
int rcc_ba_solve(rcc_ba_problem* p, const rcc_lm_options* opt, rcc_lm_summary* summary);

/* Parameter covariance at the current parameters (ceres::Covariance semantics):
 *   C = (J^T J)^-1 of the UNDAMPED Gauss-Newton system, J the same loss-weighted Jacobian the LM step uses (Huber /
 *   Cauchy applied: Ceres's apply_loss_function = true).  C is not scaled by a residual variance: a caller whose
 *   pixel noise has standard deviation sigma multiplies by sigma^2.  Rows and columns of constant blocks (the gauge,
 *   rcc_ba_set_constant) are exactly zero; every other entry is the entry of the inverse of J^T J restricted to the
 *   free parameters.  Marginal blocks (rcc_ba_covariance_blocks gives any pair of blocks), row-major, in the
 *   caller's block index order whichever set is eliminated; any pointer may be NULL:
 *     cov_shared  n_shared x n_shared   per camera fx fy cx cy k1 k2 p1 p2 k3 [ext 6], cross-camera terms included
 *     cov_views   n_views x 6 x 6
 *     cov_markers n_markers x 6 x 6
 * Returns RCC_NOT_SPD when J^T J restricted to the free parameters is not positive definite (an unobserved block, no
 * gauge held constant): a non-positive pivot of an eliminated block's H_ee or of the reduced system, or a reduced-
 * system pivot below 1e-10 of its diagonal entry.  Single rank only: with a communicator of several ranks attached
 * it returns RCC_BAD_ARG.  Afterwards the handle is linearised at the current point and the reduced system has been
 * consumed: call rcc_ba_schur again before rcc_ba_solve_step (rcc_ba_solve does). */
int rcc_ba_covariance(rcc_ba_problem* p, double* cov_shared, double* cov_views, double* cov_markers);

/* Cross-covariance blocks of (J^T J)^-1 for any pairs of parameter blocks (ceres::Covariance::Compute with a list of
 * block pairs), same semantics, conditions and after-state as rcc_ba_covariance: the undamped, loss-weighted system,
 * not scaled by a residual variance, exactly zero wherever a constant block is involved.
 *   pairs  n_pairs x 4 int32: kind_a, index_a, kind_b, index_b  (rcc_block_kind; index = view, marker or camera)
 *   out    n_pairs x 36: Cov(a, b) row-major size(a) x size(b) (Ceres GetCovarianceBlock layout) at the start of
 *          its 36-double slot, the rest of the slot zero.  size: view/marker/ext 6, intr 4, dist 5.
 * Cov(b, a) is exactly the transpose of Cov(a, b), and a pair's block does not depend on the other pairs of the request
 * or on its position there; two calls give bitwise equal results.  RCC_BAD_ARG (checked before any device work) for an
 * unknown kind, an index out of range, RCC_BLOCK_EXT on the single-camera model, n_pairs < 0, a NULL pairs or out
 * with n_pairs > 0, or a communicator of several ranks; n_pairs == 0 returns RCC_OK at once.  RCC_NOT_SPD and
 * RCC_EVAL_FAILED as for rcc_ba_covariance. */
int rcc_ba_covariance_blocks(rcc_ba_problem* p, int64_t n_pairs, const int32_t* pairs, double* out);

/* ---- read-backs for parity tests (host buffers; any may be NULL) -------- */
typedef struct {
  int32_t eliminated_is_view; /* 1: E = views, F = markers ; 0: E = markers, F = views */
  int32_t n_e, n_f;           /* number of eliminated / kept 6-dof blocks */
  int32_t n_shared;           /* n_cameras * (9 | 15) */
  int32_t n_reduced;          /* 6 n_f + n_shared */
  int32_t ld_reduced;         /* leading dimension (row stride) of the reduced matrix */
  int64_t n_pairs;            /* distinct (e,f) pairs */
} rcc_ba_dims;
int rcc_ba_get_dims(rcc_ba_problem* p, rcc_ba_dims* d);
/* J^T J / J^T r blocks after rcc_ba_linearize (undamped, constants not masked):
 *   Hee  n_e x 6 x 6      ge  n_e x 6      Hes  n_e x 6 x n_shared
 *   Hff  n_f x 6 x 6      gf  n_f x 6      Hfs  n_f x 6 x n_shared
 *   Hss  n_shared x n_shared (block diagonal per camera)   gs  n_shared
 *   W    n_obs_blocks x 6 x 6 (= J_e^T J_f per block, caller's observation order) */
int rcc_ba_get_normal_blocks(rcc_ba_problem* p, double* Hee, double* ge, double* Hes, double* Hff, double* gf,
                             double* Hfs, double* Hss, double* gs, double* W);
/* reduced system after rcc_ba_schur (summed over the ranks when a communicator is attached):
 * S n_reduced x n_reduced row-major, both triangles filled; b n_reduced */
int rcc_ba_get_reduced_system(rcc_ba_problem* p, double* S, double* b);
/* a rectangular window of the same matrix without materialising it on the host (n_reduced = 30 009 is 7.2 GB):
 * out[i * n_cols + j] = S[row0 + i][col0 + j] for 0 <= row0 + i < n_reduced and 0 <= col0 + j <= n_reduced, where
 * column n_reduced is the right-hand side b (so a window that ends at col0 + n_cols == n_reduced + 1 carries b) */
int rcc_ba_get_reduced_block(rcc_ba_problem* p, int32_t row0, int32_t n_rows, int32_t col0, int32_t n_cols, double* out);
/* last step: d_e n_e x 6, d_f n_f x 6, d_shared n_shared */
int rcc_ba_get_step(rcc_ba_problem* p, double* d_e, double* d_f, double* d_shared);

/* ---- multi-GPU: one handle per rank, observations sharded by eliminated-block
 * owner, one all-reduce of the reduced system per LM iteration ------------- */
#define RCC_COMM_ID_BYTES 128
int rcc_comm_get_unique_id(char id[RCC_COMM_ID_BYTES]);             /* rank 0 calls, then broadcasts */
int rcc_ba_comm_init(rcc_ba_problem* p, const char id[RCC_COMM_ID_BYTES], int32_t rank, int32_t n_ranks);

/* ---- measurement -------------------------------------------------------- */
/* per-stage device time (CUDA events on the handle's stream) accumulated since
 * the last reset.  names: "expand","assemble_e","assemble_f","finalize","schur_prep",
 * "schur_syrk","schur_shared","allreduce","mask","cholesky","backsub","cost","evaluate","h2d",
 * "inverse","covariance","cov_extract" (the last three: rcc_ba_covariance) */
int rcc_ba_profile_enable(rcc_ba_problem* p, int32_t on);
int rcc_ba_profile_reset(rcc_ba_problem* p);
int rcc_ba_profile_get(rcc_ba_problem* p, const char* stage, double* total_ms, int64_t* launches);
/* number of kernel launches issued by this handle since creation */
int64_t rcc_ba_launch_count(const rcc_ba_problem* p);
/* block until all work queued on the handle's stream has finished */
int rcc_ba_synchronize(rcc_ba_problem* p);
/* writes >= bytes to a scratch buffer to evict L2 between timed iterations */
int rcc_ba_flush_l2(rcc_ba_problem* p);
/* The dense Cholesky of the reduced solve on its own (tests, timing): factors in place the n x n SPD matrix whose
 * LOWER triangle is stored column-major with leading dimension ld (even, > n + extra_rows) in DEVICE memory dA;
 * rows n .. n+extra_rows-1 ride along as bordered right-hand sides (they come back multiplied by L^-T from the
 * right, i.e. as forward-substituted vectors).  use_cusolver != 0 runs cusolverDnDpotrf instead (the comparator;
 * extra_rows must be 0).  info: 0 or 1 + the first column with a non-positive pivot; ms: device time. */
int rcc_dense_potrf(int32_t device, double* dA, int32_t n, int32_t ld, int32_t extra_rows, int32_t use_cusolver,
                    int32_t* info, double* ms);
/* The back-substitution of the reduced solve on its own: L^T x = r in place (dx holds r on entry, x on return), L as
 * left by rcc_dense_potrf.  use_cublas != 0 runs cublasDtrsv instead (the comparator). */
int rcc_dense_trsv(int32_t device, const double* dA, int32_t n, int32_t ld, double* dx, int32_t use_cublas, double* ms);
/* FP64 FMA microbenchmark for the roofline denominator: returns TFLOP/s */
int rcc_fp64_peak_tflops(int32_t device, double* tflops);

/* ---- batched PnP initialiser (SURVEY 8f-2; camera_pose.cpp:132-173) ------
 * For n tags: minimise the reprojection error of the 4 corners over cam_T_tag
 * (6 dof), the job cv::solvePnP(..., CV_ITERATIVE) does at camera_pose.cpp:163.
 *   shared9 : fx fy cx cy k1 k2 p1 p2 k3 ;  sizes n ; pixels n x 8
 *   cam_T_tag (in/out) n x 6 : initial guess in (all-zero => planar homography
 *   initialisation), refined pose out ; final_cost n (may be NULL; -1 = failed) */
int rcc_pnp_batch(int32_t device, int64_t n, const double* shared9, const double* sizes, const double* pixels,
                  double* cam_T_tag, double* final_cost, int32_t max_iterations);

#ifdef __cplusplus
}
#endif
#endif /* RCC_BA_H */
