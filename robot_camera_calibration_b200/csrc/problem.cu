// Host side of the hot path: problem object, index construction, the
// Levenberg-Marquardt driver and the extern "C" boundary (include/rcc_ba.h).
//
// Stands where the reference's missing optimiser stage ("Milestone 3", between
// real_preprocessing/src/camera_pose.cpp and opt_visualization.cpp) would drive
// Ceres: ceres::Problem construction -> set_observations/set_constant,
// Problem::Evaluate -> rcc_ba_evaluate, ceres::Solve -> rcc_ba_solve.
#include "problem.h"
#include "model.cuh"

#include <nvtx3/nvToolsExt.h>   // header-only NVTX 3: ranges are no-ops unless a profiler is attached
#include <omp.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <numeric>
#include <tuple>
#include <type_traits>

using namespace rcc;

#define RCC_STR2(x) #x
#define RCC_STR(x) RCC_STR2(x)

namespace rcc {

static const char* kStageNames[ST_COUNT] = {"expand", "assemble_e", "assemble_f", "finalize", "schur_prep",
                                            "schur_syrk", "schur_shared", "allreduce", "mask", "cholesky",
                                            "backsub", "cost", "evaluate", "h2d", "inverse", "covariance",
                                            "cov_extract"};
const char* stage_name(int s) { return (s >= 0 && s < ST_COUNT) ? kStageNames[s] : "?"; }

cudaEvent_t StageTimer::get() {
  if (!pool.empty()) {
    cudaEvent_t e = pool.back();
    pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  RCC_CUDA(cudaEventCreate(&e));
  return e;
}
void StageTimer::begin(int stage, cudaStream_t s) {
  launches[stage]++;
  if (!on) return;
  Pending p{stage, get(), get()};
  RCC_CUDA(cudaEventRecord(p.a, s));
  pending.push_back(p);
}
void StageTimer::end(cudaStream_t s) {
  if (!on) return;
  RCC_CUDA(cudaEventRecord(pending.back().b, s));
}
void StageTimer::collect() {
  for (auto& p : pending) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, p.a, p.b) == cudaSuccess) ms[p.stage] += t;
    pool.push_back(p.a);
    pool.push_back(p.b);
  }
  pending.clear();
}
void StageTimer::reset() {
  collect();
  for (int i = 0; i < ST_COUNT; ++i) {
    ms[i] = 0;
    launches[i] = 0;
  }
}
StageTimer::~StageTimer() {
  for (auto& p : pending) {
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
  }
  for (auto e : pool) cudaEventDestroy(e);
}

// one pipeline stage: CUDA-event timing (rcc_ba_profile_*), launch accounting and an NVTX range named after the
// stage (K0 expand ... K6 cost), so that a timeline tool shows the same stages the profile API reports
struct Scoped {
  rcc_ba_problem* P;
  Scoped(rcc_ba_problem* p, int stage, int n_launch) : P(p) {
    nvtxRangePushA(stage_name(stage));
    P->timer.begin(stage, P->stream);
    P->launch_count += n_launch;
  }
  ~Scoped() {
    P->timer.end(P->stream);
    nvtxRangePop();
  }
};

}  // namespace rcc

rcc_ba_problem::~rcc_ba_problem() {
  chol.destroy();
  if (comm) ncclCommDestroy(comm);
  if (solver) cusolverDnDestroy(solver);
  if (blas) cublasDestroy(blas);
  if (h_pinned) cudaFreeHost(h_pinned);
  for (auto& hs : hslot) {
    if (hs.p) cudaFreeHost(hs.p);
    if (hs.ev) cudaEventDestroy(hs.ev);
  }
  if (own_stream && stream) cudaStreamDestroy(stream);
  if (comm_stream) cudaStreamDestroy(comm_stream);
  for (auto e : ev_grp)
    if (e) cudaEventDestroy(e);
  if (side_stream) cudaStreamDestroy(side_stream);
  if (side_stream2) cudaStreamDestroy(side_stream2);
  if (ev_fork) cudaEventDestroy(ev_fork);
  if (ev_join) cudaEventDestroy(ev_join);
  for (auto e : ev_piece)
    if (e) cudaEventDestroy(e);
}

typedef rcc_ba_problem P_t;
typedef rcc_ba_problem::Run Run;

#define RCC_NCCL(expr)                                                                                         \
  do {                                                                                                         \
    ncclResult_t _r = (expr);                                                                                  \
    if (_r != ncclSuccess) throw Error(RCC_NCCL_ERROR, std::string(#expr) + ": " + ncclGetErrorString(_r));   \
  } while (0)
#define RCC_BLAS(expr)                                                                             \
  do {                                                                                             \
    cublasStatus_t _r = (expr);                                                                    \
    if (_r != CUBLAS_STATUS_SUCCESS)                                                               \
      throw Error(RCC_SOLVER_ERROR, std::string(#expr) + ": cublas status " + std::to_string((int)_r)); \
  } while (0)
#define RCC_SOLVER(expr)                                                                              \
  do {                                                                                                \
    cusolverStatus_t _r = (expr);                                                                     \
    if (_r != CUSOLVER_STATUS_SUCCESS)                                                                \
      throw Error(RCC_SOLVER_ERROR, std::string(#expr) + ": cusolver status " + std::to_string((int)_r)); \
  } while (0)

static void sync(P_t* P) {
  RCC_CUDA(cudaStreamSynchronize(P->stream));
  if (P->pix_pending) {
    // a piecewise rcc_ba_update_pixels is still reading the caller's buffer on the copy streams and the main
    // stream has not joined them yet: the header promises the buffer is free once a getter / synchronize returns
    RCC_CUDA(cudaStreamSynchronize(P->side_stream));
    RCC_CUDA(cudaStreamSynchronize(P->side_stream2));
  }
}

// caller buffer -> internal pinned slot (waits for the slot's previous H2D copy, normally long done)
enum { HS_VIEWS = 0, HS_MARKERS, HS_INTR, HS_DIST, HS_EXT };
static void* stage_in(P_t* P, int slot, const void* src, size_t bytes) {
  auto& hs = P->hslot[slot];
  if (hs.busy) {
    RCC_CUDA(cudaEventSynchronize(hs.ev));
    hs.busy = false;
  }
  if (bytes > hs.cap) {
    if (hs.p) RCC_CUDA(cudaFreeHost(hs.p));
    hs.p = nullptr;
    RCC_CUDA(cudaMallocHost(&hs.p, bytes));
    hs.cap = bytes;
  }
  if (!hs.ev) RCC_CUDA(cudaEventCreateWithFlags(&hs.ev, cudaEventDisableTiming));
  memcpy(hs.p, src, bytes);
  return hs.p;
}
static void stage_issued(P_t* P, int slot) {
  RCC_CUDA(cudaEventRecord(P->hslot[slot].ev, P->stream));
  P->hslot[slot].busy = true;
}

static double* x_e(P_t* P, bool cand = false) {
  return P->elim_view ? (cand ? P->views_c.p : P->views.p) : (cand ? P->markers_c.p : P->markers.p);
}
static double* x_f(P_t* P, bool cand = false) {
  return P->elim_view ? (cand ? P->markers_c.p : P->markers.p) : (cand ? P->views_c.p : P->views.p);
}

// ---------------------------------------------------------------------------
// index construction
// ---------------------------------------------------------------------------
static std::vector<int32_t> sort_by_owner(const int32_t* own, const int32_t* oth, const int32_t* cam, int64_t n,
                                          int n_own, std::vector<int32_t>& seg_ptr) {
  seg_ptr.assign((size_t)n_own + 1, 0);
  for (int64_t i = 0; i < n; ++i) seg_ptr[own[i] + 1]++;
  for (int i = 0; i < n_own; ++i) seg_ptr[i + 1] += seg_ptr[i];
  std::vector<int32_t> perm((size_t)n), cur(seg_ptr.begin(), seg_ptr.end() - 1);
  for (int64_t i = 0; i < n; ++i) perm[cur[own[i]]++] = (int32_t)i;
#pragma omp parallel for schedule(dynamic, 64)
  for (int s = 0; s < n_own; ++s) {
    std::sort(perm.begin() + seg_ptr[s], perm.begin() + seg_ptr[s + 1], [&](int32_t a, int32_t b) {
      if (cam[a] != cam[b]) return cam[a] < cam[b];
      if (oth[a] != oth[b]) return oth[a] < oth[b];
      return a < b;
    });
  }
  return perm;
}

// group_of (optional): a group id per sorted position, non-decreasing inside a (own, camera) run; chunks never
// straddle a group boundary (the upload pieces of the F pass)
static void make_chunks(const std::vector<int32_t>& perm, const std::vector<int32_t>& seg_ptr, const int32_t* cam,
                        int n_own, int bpw, int ch_max, std::vector<Chunk>& chunks, std::vector<int32_t>& chunk_ptr,
                        const std::vector<int32_t>* group_of = nullptr) {
  chunks.clear();
  chunk_ptr.assign((size_t)n_own + 1, 0);
  for (int s = 0; s < n_own; ++s) {
    int i = seg_ptr[s];
    const int end = seg_ptr[s + 1];
    while (i < end) {
      const int c = cam[perm[i]];
      int j = i;
      while (j < end && cam[perm[j]] == c && (!group_of || (*group_of)[j] == (*group_of)[i])) ++j;
      const int len = j - i;
      const int nch = (len + ch_max - 1) / ch_max;
      int per = (len + nch - 1) / nch;
      per = ((per + bpw - 1) / bpw) * bpw;
      for (int k = i; k < j; k += per) chunks.push_back(Chunk{s, c, k, std::min(per, j - k)});
      i = j;
    }
    chunk_ptr[s + 1] = (int32_t)chunks.size();
  }
}

// counting sort of the ids 0 .. n by key(id) < n_groups: group g is list[ptr[g] .. ptr[g+1]), ascending
template <typename Key>
static void group_by(size_t n, int n_groups, Key key, std::vector<int32_t>& list, std::vector<int32_t>& ptr) {
  ptr.assign((size_t)n_groups + 1, 0);
  for (size_t i = 0; i < n; ++i) ptr[key(i) + 1]++;
  for (int g = 0; g < n_groups; ++g) ptr[g + 1] += ptr[g];
  list.resize(n);
  std::vector<int32_t> cur(ptr.begin(), ptr.end() - 1);
  for (size_t i = 0; i < n; ++i) list[cur[key(i)]++] = (int32_t)i;
}

static void cam_lists(const std::vector<Chunk>& chunks, int n_cam, std::vector<int32_t>& list,
                      std::vector<int32_t>& ptr) {
  group_by(chunks.size(), n_cam, [&](size_t c) { return chunks[c].cam; }, list, ptr);
}

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
}

// the lens every camera has, or LENS_PER_CAMERA when they differ
static int handle_lens(const P_t* P) {
  for (int32_t l : P->cam_lens)
    if (l != P->cam_lens[0]) return LENS_PER_CAMERA;
  return P->cam_lens[0];
}

// The K2 and K1 runs (problem.h: Run) from the chunk records, the upload pieces and the cameras' lenses.  A pass, or
// each upload piece of it, is launched once per lens among its chunks, in lens order, the ids ascending; a run whose
// ids form a contiguous range needs no id list.  With one lens for every camera a pass or a piece is one run, even
// without chunks (launch_assemble then returns at once; the run still counts as a launch); an upload piece without E
// chunks has no runs, and neither has any piece unless the caller order is the E-sorted order (pix_identity).
static void plan_launches(P_t* P) {
  if (!P->have_obs) return;
  const int common = handle_lens(P);
  std::vector<int32_t> ids, list, ptr;
  auto plan = [&](const std::vector<Chunk>& chunks, int n_groups, auto group_of, std::vector<Run>* runs) {
    group_by(chunks.size(), n_groups * N_LENSES,
             [&](size_t c) { return group_of(c) * N_LENSES + P->cam_lens[chunks[c].cam]; }, list, ptr);
    for (int g = 0; g < n_groups; ++g) {
      runs[g].clear();
      for (int l = 0; l < N_LENSES; ++l) {
        const int lo = ptr[g * N_LENSES + l], n = ptr[g * N_LENSES + l + 1] - lo;
        if (n == 0 && l != common) continue;
        const bool listed = n > 0 && list[lo + n - 1] - list[lo] != n - 1;
        runs[g].push_back(Run{l, listed ? (int)ids.size() : n > 0 ? list[lo] : 0, n, listed});
        if (listed) ids.insert(ids.end(), list.begin() + lo, list.begin() + lo + n);
      }
    }
  };
  constexpr int NP = rcc_ba_problem::PIX_PIECES;
  if (P->pix_identity) {
    std::vector<int32_t> e_piece(P->e_chunks_h.size());
    for (int k = 0; k < NP; ++k)
      for (int c = P->piece_chunk[k]; c < P->piece_chunk[k + 1]; ++c) e_piece[c] = k;
    plan(P->e_chunks_h, NP, [&](size_t c) { return e_piece[c]; }, P->piece_runs_e);
    plan(P->f_chunks_h, NP, [&](size_t c) { return P->f_chunk_piece_h[c]; }, P->piece_runs_f);
  }
  for (int k = 0; k < NP; ++k)
    if (!P->pix_identity || P->piece_chunk[k + 1] <= P->piece_chunk[k]) {
      P->piece_runs_e[k].clear();
      P->piece_runs_f[k].clear();
    }
  plan(P->f_chunks_h, 1, [](size_t) { return 0; }, &P->runs_f);
  plan(P->e_chunks_h, 1, [](size_t) { return 0; }, &P->runs_e);
  // K1: the E runs as positions of `list` (the E chunk ids in lens order); a copy of the records unless that order
  // is the chunk order
  bool copy = false;
  for (size_t i = 0; i < list.size(); ++i) copy |= list[i] != (int32_t)i;
  P->runs_k1 = P->runs_e;
  for (int i = 0, pos = 0; i < (int)P->runs_k1.size(); pos += P->runs_k1[i++].count) {
    P->runs_k1[i].first = pos;
    P->runs_k1[i].listed = copy;
  }
  cudaStream_t s = P->stream;
  if (copy) {
    std::vector<Chunk> recs(list.size());
    for (size_t i = 0; i < list.size(); ++i) recs[i] = P->e_chunks_h[list[i]];
    P->k1_chunks.upload(recs, s);
  } else {
    P->k1_chunks.release();
  }
  P->run_ids.upload(ids, s);
  RCC_CUDA(cudaStreamSynchronize(s));
}

static void build_indices(P_t* P, const int32_t* view_idx, const int32_t* marker_idx, const int32_t* cam_idx) {
  const int64_t n = P->n_obs;
  RCC_REQUIRE(n < (int64_t)2000000000 / 36 * 8, RCC_BAD_ARG, "too many observation blocks for 32-bit indexing");
  RCC_CUDA(cudaStreamSynchronize(P->side_stream));   // a piecewise pixel upload may still target the old buffers
  RCC_CUDA(cudaStreamSynchronize(P->side_stream2));
  P->pix_pending = false;
  std::vector<int32_t> cam_zero;
  if (!cam_idx) {
    cam_zero.assign((size_t)n, 0);
    cam_idx = cam_zero.data();
  }
  for (int64_t i = 0; i < n; ++i) {
    RCC_REQUIRE(view_idx[i] >= 0 && view_idx[i] < P->n_views, RCC_BAD_ARG, "view index out of range");
    RCC_REQUIRE(marker_idx[i] >= 0 && marker_idx[i] < P->n_markers, RCC_BAD_ARG, "marker index out of range");
    RCC_REQUIRE(cam_idx[i] >= 0 && cam_idx[i] < P->n_cam, RCC_BAD_ARG, "camera index out of range");
  }
  const int32_t* e_of = P->elim_view ? view_idx : marker_idx;
  const int32_t* f_of = P->elim_view ? marker_idx : view_idx;
  const int bpw = P->rig ? PassGeom<true>::BPW : PassGeom<false>::BPW;
  const int ch_max = std::max(bpw, env_int("RCC_CHUNK", 64));
  cudaStream_t s = P->stream;

  // ---- E pass order
  std::vector<int32_t> seg_e, seg_f;
  std::vector<int32_t> perm_e = sort_by_owner(e_of, f_of, cam_idx, n, P->n_e, seg_e);
  std::vector<Chunk> chunks;
  std::vector<int32_t> chunk_ptr, list, ptr;
  make_chunks(perm_e, seg_e, cam_idx, P->n_e, bpw, ch_max, chunks, chunk_ptr);
  P->n_chunks_e = (int)chunks.size();
  P->e_chunks.upload(chunks, s);
  P->e_chunks_h = chunks;
  P->e_chunk_ptr.upload(chunk_ptr, s);
  cam_lists(chunks, P->n_cam, list, ptr);
  P->cam_chunks_e.upload(list, s);
  P->cam_ptr_e.upload(ptr, s);
  {
    std::vector<int32_t> own((size_t)n), oth((size_t)n), cam((size_t)n);
#pragma omp parallel for
    for (int64_t i = 0; i < n; ++i) {
      const int32_t o = perm_e[i];
      own[i] = e_of[o];
      oth[i] = f_of[o];
      cam[i] = cam_idx[o];
    }
    P->e_own.upload(own, s);
    P->e_oth.upload(oth, s);
    P->e_cam.upload(cam, s);
    P->e_orig.upload(perm_e, s);
    RCC_CUDA(cudaStreamSynchronize(s));
  }
  {
    // caller order == E-sorted order (observations listed per eliminated block, the usual case):
    // update_pixels can then copy straight into e_pix, piece by piece, cut at chunk boundaries
    bool ident = true;
    for (int64_t i = 0; i < n && ident; ++i) ident = perm_e[i] == (int32_t)i;
    P->pix_identity = ident && n > 0;
    P->pix_pending = false;
    // pieces are cut at eliminated-block boundaries: 8 for large uploads (what is left after the copy is the work
    // of the last piece: keep it short), 4 for small ones, where a piece must still be worth a launch
    const int np = n >= rcc_ba_problem::LARGE_UPLOAD_BLOCKS ? rcc_ba_problem::PIX_PIECES : 4;
    P->piece_chunk[0] = 0;
    P->piece_block[0] = 0;
    int e_cut = 0;
    for (int k = 1; k <= rcc_ba_problem::PIX_PIECES; ++k) {
      const int64_t want = n * std::min(k, np) / np;
      while (e_cut < P->n_e && seg_e[e_cut] < want) ++e_cut;      // first eliminated block starting at or after `want`
      if (k >= np) e_cut = P->n_e;
      P->piece_block[k] = seg_e[e_cut];
      P->piece_chunk[k] = chunk_ptr[e_cut];
    }
  }
  {
    std::vector<int32_t> cnt((size_t)P->n_e);
    for (int e = 0; e < P->n_e; ++e) cnt[e] = seg_e[e + 1] - seg_e[e];
    P->e_count.upload(cnt, s);
  }

  // ---- F pass order
  std::vector<int32_t> perm_f = sort_by_owner(f_of, e_of, cam_idx, n, P->n_f, seg_f);
  {
    // F-pass chunks never straddle an upload piece: the F pass of a piece can then run as soon as the piece has
    // landed, like its E pass (rows are sorted by eliminated block inside a camera run, pieces are ranges of them)
    std::vector<int32_t> piece_of_e((size_t)P->n_e, 0), group((size_t)n, 0);
    if (P->pix_identity) {
      for (int k = 0, e = 0; k < rcc_ba_problem::PIX_PIECES; ++k)
        for (; e < P->n_e && seg_e[e] < P->piece_block[k + 1]; ++e) piece_of_e[e] = k;
#pragma omp parallel for
      for (int64_t i = 0; i < n; ++i) group[i] = piece_of_e[e_of[perm_f[i]]];
    }
    make_chunks(perm_f, seg_f, cam_idx, P->n_f, bpw, ch_max, chunks, chunk_ptr, P->pix_identity ? &group : nullptr);
    P->f_chunk_piece_h.resize(chunks.size());
    for (size_t c = 0; c < chunks.size(); ++c) P->f_chunk_piece_h[c] = group[chunks[c].start];
  }
  P->n_chunks_f = (int)chunks.size();
  P->f_chunks.upload(chunks, s);
  P->f_chunks_h = chunks;
  P->f_chunk_ptr.upload(chunk_ptr, s);
  cam_lists(chunks, P->n_cam, list, ptr);
  P->cam_chunks_f.upload(list, s);
  P->cam_ptr_f.upload(ptr, s);
  {
    std::vector<int32_t> oth((size_t)n);
#pragma omp parallel for
    for (int64_t i = 0; i < n; ++i) oth[i] = e_of[perm_f[i]];
    P->f_oth.upload(oth, s);
    // E-sorted position -> F-sorted position (the pixel loader scatters every E-sorted block into f_pix)
    std::vector<int32_t> e_pos_of_caller((size_t)n), f_inv((size_t)n);
#pragma omp parallel for
    for (int64_t i = 0; i < n; ++i) e_pos_of_caller[perm_e[i]] = (int32_t)i;
#pragma omp parallel for
    for (int64_t i = 0; i < n; ++i) f_inv[e_pos_of_caller[perm_f[i]]] = (int32_t)i;
    P->f_inv.upload(f_inv, s);
    RCC_CUDA(cudaStreamSynchronize(s));
  }

  // ---- distinct (e,f) pairs in (e,f) order, members = E-sorted positions
  std::vector<int32_t> row_ptr((size_t)P->n_e + 1, 0), pair_e, pair_f, pair_mptr, members;
  pair_e.reserve((size_t)n);
  pair_f.reserve((size_t)n);
  pair_mptr.reserve((size_t)n + 1);
  members.reserve((size_t)n);
  {
    std::vector<std::pair<int32_t, int32_t>> tmp;
    for (int e = 0; e < P->n_e; ++e) {
      tmp.clear();
      for (int pos = seg_e[e]; pos < seg_e[e + 1]; ++pos) tmp.emplace_back(f_of[perm_e[pos]], pos);
      if (P->n_cam > 1) std::sort(tmp.begin(), tmp.end());
      for (size_t k = 0; k < tmp.size(); ++k) {
        if (k == 0 || tmp[k].first != tmp[k - 1].first) {
          pair_e.push_back(e);
          pair_f.push_back(tmp[k].first);
          pair_mptr.push_back((int32_t)members.size());
        }
        members.push_back(tmp[k].second);
      }
      row_ptr[e + 1] = (int32_t)pair_e.size();
    }
    pair_mptr.push_back((int32_t)members.size());
  }
  P->n_pairs = (int64_t)pair_e.size();
  {
    // rows whose pairs have exactly one member each, at consecutive sorted positions (every row of a
    // single-camera problem): schur_prep then needs no per-pair index loads
    std::vector<int32_t> row_pos0((size_t)std::max(P->n_e, 1), -1);
#pragma omp parallel for schedule(static)
    for (int e = 0; e < P->n_e; ++e) {
      const int p0 = row_ptr[e], p1 = row_ptr[e + 1];
      if (p1 <= p0) continue;
      const int first = members[pair_mptr[p0]];
      bool ok = true;
      for (int p = p0; p < p1 && ok; ++p)
        ok = (pair_mptr[p + 1] - pair_mptr[p] == 1) && (members[pair_mptr[p]] == first + (p - p0));
      if (ok) row_pos0[e] = first;
    }
    P->row_pos0.upload(row_pos0, s);
  }
  P->row_ptr.upload(row_ptr, s);
  P->row_ptr_h = row_ptr;
  P->pair_e.upload(pair_e, s);
  P->pair_f.upload(pair_f, s);
  P->pair_mptr.upload(pair_mptr, s);
  P->pair_members.upload(members, s);

  // ---- column structure (pairs of kept block f, ascending e)
  std::vector<int32_t> col_ptr((size_t)P->n_f + 1, 0), col_pair((size_t)P->n_pairs);
  {
    for (int64_t p = 0; p < P->n_pairs; ++p) col_ptr[pair_f[p] + 1]++;
    for (int f = 0; f < P->n_f; ++f) col_ptr[f + 1] += col_ptr[f];
    std::vector<int32_t> cur(col_ptr.begin(), col_ptr.end() - 1);
    for (int64_t p = 0; p < P->n_pairs; ++p) col_pair[cur[pair_f[p]]++] = (int32_t)p;
    P->col_ptr.upload(col_ptr, s);
    P->col_pair.upload(col_pair, s);
    RCC_CUDA(cudaStreamSynchronize(s));
  }
  // ---- column sub-tiles of the Schur SYRK: tile_ptr[e][J] = first pair of row e with f >= SYRK_SUBTILE J
  P->n_tiles = (P->n_f + SYRK_SUBTILE - 1) / SYRK_SUBTILE;
  {
    const int nt = P->n_tiles;
    std::vector<int32_t> tile_ptr((size_t)P->n_e * (nt + 1));
#pragma omp parallel for schedule(static)
    for (int e = 0; e < P->n_e; ++e) {
      int p = row_ptr[e];
      const int end = row_ptr[e + 1];
      for (int J = 0; J <= nt; ++J) {
        const int fmin = J * SYRK_SUBTILE;
        while (p < end && pair_f[p] < fmin) ++p;
        tile_ptr[(size_t)e * (nt + 1) + J] = (J == nt) ? end : p;
      }
    }
    P->tile_ptr.upload(tile_ptr, s);
    // work list of the SYRK: one CTA per (block row f, column tile J on or right of the diagonal),
    // column tile major so that co-resident CTAs read the same columns of Y (L2 locality; a
    // heaviest-first order was measured slower on cfg4 for that reason)
    const int ctw = SYRK_SUBTILE * SYRK_CTA_SUBTILES;   // kept blocks per column tile
    const int nct = (nt + SYRK_CTA_SUBTILES - 1) / SYRK_CTA_SUBTILES;
    std::vector<int64_t> order;
    for (int J = 0; J < nct; ++J)
      for (int f = 0; f < std::min(P->n_f, (J + 1) * ctw); ++f) order.push_back((int64_t)f * nct + J);
    std::vector<int32_t> cta_list(2 * order.size());
    for (size_t i = 0; i < order.size(); ++i) {
      cta_list[2 * i] = (int32_t)(order[i] / nct);
      cta_list[2 * i + 1] = (int32_t)(order[i] % nct);
    }
    P->n_syrk_ctas = (int)order.size();
    {
      // groups of column tiles with about equal CTA counts; few groups when the reduced system is small (each group
      // is one all-reduce: below ~64 MB per group the launch latency would outweigh what the overlap hides)
      const size_t bytes = (size_t)P->n_red * P->n_red * 4;          // upper triangle in bytes
      int G = (int)std::min<size_t>(rcc_ba_problem::SYRK_GROUPS, std::max<size_t>(1, bytes / ((size_t)64 << 20)));
      if (env_int("RCC_SYRK_GROUPS", 0) > 0) G = std::min((int)rcc_ba_problem::SYRK_GROUPS, env_int("RCC_SYRK_GROUPS", 0));   // tests
      G = std::max(1, std::min(G, nct));
      P->n_syrk_groups = G;
      P->syrk_grp_cta[0] = 0;
      P->syrk_grp_col[0] = 0;
      int64_t cum = 0;
      int g = 1;
      for (int J = 0; J < nct && g < G; ++J) {
        cum += std::min(P->n_f, (J + 1) * ctw);
        if (cum * G >= (int64_t)order.size() * g) {
          P->syrk_grp_cta[g] = (int)cum;
          P->syrk_grp_col[g] = std::min(6 * P->n_f, (J + 1) * ctw * 6);
          ++g;
        }
      }
      for (; g <= rcc_ba_problem::SYRK_GROUPS; ++g) {               // the last real group ends at the end; the rest are empty
        P->syrk_grp_cta[g] = (int)order.size();
        P->syrk_grp_col[g] = 6 * P->n_f;
      }
    }
    if (cta_list.empty()) cta_list.assign(2, 0);
    P->syrk_ctas.upload(cta_list, s);
    RCC_CUDA(cudaStreamSynchronize(s));
  }

  // ---- buffers that scale with the observations
  P->e_pix.alloc((size_t)n * 8);
  P->f_pix.alloc((size_t)n * 8);
  P->part_e.alloc((size_t)P->n_chunks_e * (P->rig ? PassGeom<true>::PART_E : PassGeom<false>::PART_E));
  P->part_f.alloc((size_t)P->n_chunks_f * (P->rig ? PassGeom<true>::PART_F : PassGeom<false>::PART_F));
  P->W.alloc((size_t)n * 36);
  P->Y.alloc((size_t)std::max<int64_t>(P->n_pairs, 1) * 36);
  P->cost_partials.alloc((size_t)std::max(std::max(1, eval_grid(n)), P->n_chunks_e) + P->n_prior_parts);
  RCC_CUDA(cudaStreamSynchronize(s));
  P->have_obs = true;
  P->n_slots = 0;   // new observations clear the corner layout
  P->linearized = P->schur_done = P->step_ready = P->cand_ready = false;
  plan_launches(P);
}

static void refresh_constants(P_t* P) {
  if (!P->const_dirty) return;
  const std::vector<uint8_t>& ce = P->elim_view ? P->c_view : P->c_marker;
  const std::vector<uint8_t>& cf = P->elim_view ? P->c_marker : P->c_view;
  P->e_const.upload(ce, P->stream);
  std::vector<int32_t> idx;
  for (int f = 0; f < P->n_f; ++f)
    if (cf[f])
      for (int k = 0; k < 6; ++k) idx.push_back(6 * f + k);
  for (int c = 0; c < P->n_cam; ++c) {
    const int b = 6 * P->n_f + c * P->sp;
    if (P->c_intr[c]) for (int k = 0; k < 4; ++k) idx.push_back(b + k);
    if (P->c_dist[c]) for (int k = 4; k < 9; ++k) idx.push_back(b + k);
    else if (P->cam_lens[c] == LENS_EQUIDISTANT) idx.push_back(b + 8);   // the reserved distortion slot
    if (P->rig && P->c_ext[c]) for (int k = 9; k < 15; ++k) idx.push_back(b + k);
  }
  P->n_const = (int)idx.size();
  if (idx.empty()) idx.push_back(0);
  P->const_idx.upload(idx, P->stream);
  sync(P);
  P->const_dirty = false;
}

// ---------------------------------------------------------------------------
// pipeline stages
// ---------------------------------------------------------------------------
static void ensure_expanded(P_t* P) {
  if (P->expanded_valid) return;
  Scoped t(P, ST_EXPAND, 1);
  launch_expand_poses(P->views.p, P->n_views, P->view_x.p, P->markers.p, P->sizes.p, P->n_markers, P->marker_x.p, P->shared.p,
                      P->n_cam, P->sp, P->ext_x.p, P->stream);
  P->expanded_valid = true;
}

// after a piecewise update_pixels: wait for the last piece (every piece has scattered itself into f_pix)
static void ensure_pixels(P_t* P) {
  if (!P->pix_pending) return;
  for (int k = 0; k < rcc_ba_problem::PIX_PIECES; ++k) RCC_CUDA(cudaStreamWaitEvent(P->stream, P->ev_piece[k], 0));
  P->pix_pending = false;
}

// K2 over one run of a pass; a.chunks and a.partials are the whole pass's
static void assemble_run(P_t* P, bool epass, AssembleArgs a, const Run& r) {
  const int part = epass ? (P->rig ? PassGeom<true>::PART_E : PassGeom<false>::PART_E)
                         : (P->rig ? PassGeom<true>::PART_F : PassGeom<false>::PART_F);
  if (r.listed) {
    a.chunk_list = P->run_ids.p + r.first;
  } else {
    a.chunks += r.first;
    a.partials += (size_t)r.first * part;
  }
  a.n_chunks = r.count;
  launch_assemble(P->rig, epass, epass ? P->elim_view : !P->elim_view, r.lens, a, P->stream);
  P->launch_count += 1;
}

// the priors evaluated at the current or the candidate parameters; H and g are the linearisation's blocks (used by
// launch_prior(true, ...) only)
static PriorArgs prior_args(P_t* P, bool cand, double* cost2) {
  PriorArgs a{};
  for (int t = 0; t <= PRIOR_KINDS; ++t) a.off[t] = P->prior_off[t];
  a.index = P->prior_index.p; a.mean = P->prior_mean.p; a.A = P->prior_A.p; a.AtA = P->prior_AtA.p;
  a.views = cand ? P->views_c.p : P->views.p;
  a.markers = cand ? P->markers_c.p : P->markers.p;
  a.shared = cand ? P->shared_c.p : P->shared.p;
  a.sp = P->sp; a.n_shared = P->n_shared; a.elim_view = P->elim_view ? 1 : 0;
  a.Hee = P->Hee.p; a.ge = P->ge.p; a.Hff = P->Hff.p; a.gf = P->gf.p; a.Hss = P->Hss.p; a.gs = P->gs.p;
  a.cost2 = cost2;
  return a;
}

static void do_linearize(P_t* P) {
  RCC_REQUIRE(P->have_obs, RCC_NOT_READY, "set_observations has not been called");
  ensure_expanded(P);
  RCC_CUDA(cudaMemsetAsync(P->fail_flag.p, 0, sizeof(int32_t), P->stream));
  AssembleArgs e{};
  e.view_x = P->view_x.p;
  e.marker_x = P->marker_x.p;
  e.ext_x = P->ext_x.p;
  e.shared = P->shared.p;
  e.fail_flag = P->fail_flag.p;
  e.loss = P->loss;
  e.loss_a2 = P->loss_scale * P->loss_scale;
  AssembleArgs f = e;
  e.oth = P->e_oth.p;
  e.pix = P->e_pix.p;
  e.chunks = P->e_chunks.p;
  e.partials = P->part_e.p;
  e.W = P->W.p;
  f.oth = P->f_oth.p;
  f.pix = P->f_pix.p;
  f.chunks = P->f_chunks.p;
  f.partials = P->part_f.p;
  if (P->n_slots > 0) {   // the target instantiations, for every run of plan_launches
    e.corners = f.corners = P->corners.p;
    e.slot = P->e_slot.p;
    f.slot = P->f_slot.p;
  }
  bool f_done = false;
  {
    Scoped t(P, ST_ASSEMBLE_E, 0);
    if (P->pix_pending) {
      // pixels are still arriving on the side stream: the E pass of a piece starts when the piece has landed,
      // and so does its F pass on large uploads (the piece scattered itself into f_pix, and no F chunk straddles
      // pieces)
      f_done = P->n_obs >= rcc_ba_problem::LARGE_UPLOAD_BLOCKS;
      for (int k = 0; k < rcc_ba_problem::PIX_PIECES; ++k) {
        RCC_CUDA(cudaStreamWaitEvent(P->stream, P->ev_piece[k], 0));
        for (const Run& r : P->piece_runs_e[k]) assemble_run(P, true, e, r);
        if (f_done)
          for (const Run& r : P->piece_runs_f[k]) assemble_run(P, false, f, r);
      }
    } else {
      for (const Run& r : P->runs_e) assemble_run(P, true, e, r);
    }
  }
  ensure_pixels(P);
  if (!f_done) {
    Scoped t(P, ST_ASSEMBLE_F, 0);
    for (const Run& r : P->runs_f) assemble_run(P, false, f, r);
  }
  {
    Scoped t(P, ST_FINALIZE, P->n_prior_parts > 0 ? 2 : 1);
    FinalizeSideArgs fe{P->part_e.p, P->e_chunks.p, P->e_chunk_ptr.p, P->n_e, P->n_shared, P->Hee.p, P->ge.p, P->Hes.p};
    FinalizeSideArgs ff{P->part_f.p, P->f_chunks.p, P->f_chunk_ptr.p, P->n_f, P->n_shared, P->Hff.p, P->gf.p, P->Hfs.p};
    FinalizeSharedArgs fs{P->part_e.p, P->cam_chunks_e.p, P->cam_ptr_e.p, P->n_cam, P->n_shared, P->Hss.p, P->gs.p,
                          P->cost2_cam.p, P->fin_scratch.p, P->fin_done.p, P->loss != 0 ? 1 : 0, P->fin_slices};
    launch_finalize(P->rig, fe, ff, fs, P->stream);
    // the priors add into the finalized blocks; their cost partials follow the cameras' in cost2_cam
    if (P->n_prior_parts > 0) launch_prior(true, prior_args(P, false, P->cost2_cam.p + P->n_cam), P->stream);
  }
  P->linearized = true;
  P->schur_done = P->step_ready = P->cand_ready = false;
}

// pivot_fail (device, nullable): set when a free eliminated block's pivot of chol(H_ee + D_e) is not positive
static void do_schur(P_t* P, double radius, int32_t* pivot_fail = nullptr) {
  RCC_REQUIRE(P->linearized, RCC_NOT_READY, "linearize has not been called");
  bool eager = false;
  RCC_REQUIRE(radius > 0, RCC_BAD_ARG, "radius must be positive");
  refresh_constants(P);
  P->radius_used = radius;
  {
    Scoped t(P, ST_SCHUR_PREP, 1);
    SchurPrepArgs a{};
    a.n_e = P->n_e; a.n_shared = P->n_shared; a.n_bb = P->n_bb;
    a.Hee = P->Hee.p; a.ge = P->ge.p; a.Hes = P->Hes.p; a.e_const = P->e_const.p;
    a.row_ptr = P->row_ptr.p; a.pair_mptr = P->pair_mptr.p; a.pair_members = P->pair_members.p; a.row_pos0 = P->row_pos0.p; a.W = P->W.p;
    a.radius = radius; a.min_diag = P->min_diag; a.max_diag = P->max_diag; a.jacobi = P->jacobi;
    a.Linv = P->Linv.p; a.Y = P->Y.p; a.Yb = P->Yb.p; a.d2e = P->d2e.p;
    a.pivot_fail = pivot_fail;
    launch_schur_prep(a, P->stream);
  }
  {
    // the border strip, the shared x shared corner and the tail rows depend only on schur_prep:
    // they run on the side stream beside the block-sparse SYRK and join before the stage ends
    Scoped t(P, ST_SCHUR_SYRK, 5);
    SchurSyrkArgs a{};
    a.n_f = P->n_f; a.n_e = P->n_e; a.n_shared = P->n_shared; a.n_bb = P->n_bb;
    a.n_tiles = P->n_tiles; a.ld = P->ld;
    a.col_ptr = P->col_ptr.p; a.col_pair = P->col_pair.p; a.pair_e = P->pair_e.p; a.pair_f = P->pair_f.p;
    a.cta_list = P->syrk_ctas.p; a.n_ctas = P->n_syrk_ctas;
    a.tile_ptr = P->tile_ptr.p; a.Y = P->Y.p; a.Yb = P->Yb.p; a.Hff = P->Hff.p; a.gf = P->gf.p; a.Hfs = P->Hfs.p;
    a.S = P->S.p;
    RCC_CUDA(cudaEventRecord(P->ev_fork, P->stream));
    RCC_CUDA(cudaStreamWaitEvent(P->side_stream, P->ev_fork, 0));
    launch_schur_border(a, P->side_stream);
    SchurSharedArgs sh{P->n_e, P->n_f, P->n_shared, P->n_bb, P->ld, P->Yb.p, P->Hss.p, P->gs.p, P->shared_scratch.p,
                       P->S.p};
    launch_schur_shared(sh, P->side_stream);
    ReducedTailArgs r{P->n_f, P->n_shared, P->ld, P->Hff.p, P->gf.p, P->Hss.p, P->gs.p, P->cost2_cam.p,
                      P->n_cam + P->n_prior_parts, P->S.p};
    launch_reduced_tail(r, P->side_stream);
    RCC_CUDA(cudaEventRecord(P->ev_join, P->side_stream));
    eager = P->comm != nullptr && P->n_ranks > 1;
    if (!eager) {
      launch_schur_syrk(a, P->stream);
      RCC_CUDA(cudaStreamWaitEvent(P->stream, P->ev_join, 0));
    } else {
      // Several ranks: the sum over the ranks overlaps with the SYRK.  The work list is column-tile major, so a group
      // of column tiles = a band of columns of S is final as soon as its CTAs are done: the communication stream
      // packs the band's live part (upper triangle inside the band), all-reduces it and unpacks it while the main
      // stream computes the next band.  The border band (shared parameters, rhs) and the tail rows come last.
      const int n = P->n_red;
      const size_t tail = 2 * (size_t)n + 8;
      size_t need = packed_band_doubles(n, 6 * P->n_f, P->ld) + tail;
      for (int g = 0; g < P->n_syrk_groups; ++g) need += packed_band_doubles(n, P->syrk_grp_col[g], P->syrk_grp_col[g + 1]);
      P->packed_S.ensure(need);
      size_t off = 0;
      for (int g = 0; g < P->n_syrk_groups; ++g) {
        SchurSyrkArgs ag = a;
        ag.cta_list = P->syrk_ctas.p + 2 * (size_t)P->syrk_grp_cta[g];
        ag.n_ctas = P->syrk_grp_cta[g + 1] - P->syrk_grp_cta[g];
        launch_schur_syrk(ag, P->stream);
        RCC_CUDA(cudaEventRecord(P->ev_grp[g], P->stream));
        RCC_CUDA(cudaStreamWaitEvent(P->comm_stream, P->ev_grp[g], 0));
        const int c0 = P->syrk_grp_col[g], c1 = P->syrk_grp_col[g + 1];
        const size_t cnt = packed_band_doubles(n, c0, c1);
        if (cnt == 0) continue;
        launch_pack_band(P->S.p, P->ld, n, c0, c1, P->packed_S.p + off, true, P->comm_stream);
        RCC_NCCL(ncclAllReduce(P->packed_S.p + off, P->packed_S.p + off, cnt, ncclDouble, ncclSum, P->comm, P->comm_stream));
        launch_pack_band(P->S.p, P->ld, n, c0, c1, P->packed_S.p + off, false, P->comm_stream);
        off += cnt;
        P->launch_count += 3;
      }
      {
        RCC_CUDA(cudaStreamWaitEvent(P->comm_stream, P->ev_join, 0));
        const int c0 = 6 * P->n_f, c1 = P->ld;
        const size_t cnt = packed_band_doubles(n, c0, c1);
        double* pk = P->packed_S.p + off;
        launch_pack_band(P->S.p, P->ld, n, c0, c1, pk, true, P->comm_stream);
        RCC_CUDA(cudaMemcpyAsync(pk + cnt, P->S.p + (size_t)n * P->ld, tail * sizeof(double), cudaMemcpyDeviceToDevice,
                                 P->comm_stream));
        RCC_NCCL(ncclAllReduce(pk, pk, cnt + tail, ncclDouble, ncclSum, P->comm, P->comm_stream));
        launch_pack_band(P->S.p, P->ld, n, c0, c1, pk, false, P->comm_stream);
        RCC_CUDA(cudaMemcpyAsync(P->S.p + (size_t)n * P->ld, pk + cnt, tail * sizeof(double), cudaMemcpyDeviceToDevice,
                                 P->comm_stream));
        RCC_CUDA(cudaEventRecord(P->ev_grp[rcc_ba_problem::SYRK_GROUPS], P->comm_stream));
        P->launch_count += 2;
      }
    }
  }
  if (eager) {
    // what is left of the reduction once the last band has been computed
    Scoped t(P, ST_ALLREDUCE, 1);
    RCC_CUDA(cudaStreamWaitEvent(P->stream, P->ev_grp[rcc_ba_problem::SYRK_GROUPS], 0));
  }
  P->reduced_in_schur = eager;
  P->schur_done = true;
  P->step_ready = P->cand_ready = false;
}

// stats buffer layout (device, 16 doubles)
enum { SX_MCC_E = 0, SX_DN_E, SX_XN_E, SX_CAND2, SX_GMAX_E, SX_MCC_F, SX_DN_F, SX_XN_F, SX_GMAX_F, SX_COST2, SX_N };

__global__ void gmax_kernel(const double* __restrict__ g, const uint8_t* __restrict__ cst, int n_blocks,
                            double* __restrict__ out) {
  __shared__ double red[256];
  double m = 0.0;
  for (int i = threadIdx.x; i < n_blocks * 6; i += 256) {
    if (cst == nullptr || !cst[i / 6]) m = fmax(m, fabs(g[i]));
  }
  red[threadIdx.x] = m;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + o]);
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0];
}
__global__ void gmaxf_kernel(const double* __restrict__ g, int n, double* __restrict__ out) {
  __shared__ double red[256];
  double m = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) m = fmax(m, fabs(g[i]));
  red[threadIdx.x] = m;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + o]);
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0];
}
__global__ void copy_scalar_kernel(const double* src, double* dst) { dst[0] = src[0]; }
// pivot of the border row of the bordered Cholesky: anything larger than b^T S^-1 b keeps it positive
__global__ void set_border_pivot_kernel(double* p) { p[0] = 1e300; }
// rhs = -(L^-1 b): the border row of the factor (column n of the row-major buffer), negated for S x = -b
__global__ void extract_rhs_kernel(const double* __restrict__ S, int n, int ld, double* __restrict__ rhs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) rhs[i] = -S[(size_t)i * ld + n];
}

// which factorisation the reduced solve uses (RCC_CHOLESKY overrides; resolved once per handle and communicator)
static int cholesky_mode(P_t* P) {
  if (P->chol_mode >= 0) return P->chol_mode;
  const char* v = getenv("RCC_CHOLESKY");
  const std::string s = v ? v : "auto";
  const bool multi = P->comm != nullptr && P->n_ranks > 1;
  int mode;
  if (s == "cusolver") mode = 0;
  else if (s == "own") mode = 1;
  else if (s == "dist") mode = multi ? 2 : 1;
  else {
    // auto: with several ranks and a system large enough for its trailing update to dominate, the hand-written
    // factorisation distributed over the ranks; on one GPU it runs at 86 % of cusolverDnDpotrf's rate at n = 30 009
    // and loses to it below (panel latency of the 128-column steps), so a single rank calls the library
    // (measured, DESIGN.md section 6)
    const int n_min = env_int("RCC_CHOL_MIN_N", 6000);
    mode = (multi && P->n_red >= n_min) ? 2 : 0;
  }
  P->chol_mode = mode;
  return mode;
}

// Cholesky of the reduced system in place, by the method cholesky_mode() picks; dev_info[0] receives 0 or the first
// column with a non-positive pivot.  with_rhs: the (n+1) x (n+1) bordered matrix [[S, b], [b^T, big]], whose last row
// comes out as L^-1 b (see do_step); otherwise S alone.
static void factor_reduced(P_t* P, bool with_rhs) {
  const int n = P->n_red;
  const int mode = cholesky_mode(P);
  if (mode == 0) {
    if (with_rhs) set_border_pivot_kernel<<<1, 1, 0, P->stream>>>(P->S.p + (size_t)n * P->ld + n);
    RCC_SOLVER(cusolverDnDpotrf(P->solver, CUBLAS_FILL_MODE_LOWER, with_rhs ? n + 1 : n, P->S.p, P->ld,
                                P->potrf_work.p, P->potrf_lwork, P->dev_info.p));
  } else {
    // dense.cu: the right-hand side is row n of every panel (never a column), so no border pivot is needed.
    // mode 2: block column J is factored and updated by rank J % n_ranks, finished panels are broadcast in place.
    const int64_t before = P->chol.launches;
    chol_factor(P->S.p, n, P->ld, with_rhs ? n + 1 : n, P->rank, mode == 2 ? P->n_ranks : 1,
                mode == 2 ? P->comm : nullptr, P->stream, P->chol);
    P->launch_count += P->chol.launches - before;
    RCC_CUDA(cudaMemcpyAsync(P->dev_info.p, P->chol.info, sizeof(int), cudaMemcpyDeviceToDevice, P->stream));
  }
}

// all-reduce + damping/mask + Cholesky + back-substitution + candidate parameters
static void do_step(P_t* P) {
  RCC_REQUIRE(P->schur_done, RCC_NOT_READY, "schur has not been called");
  const int n = P->n_red;
  // several ranks: rcc_ba_schur has already summed S over the ranks, band by band, behind its SYRK
  RCC_REQUIRE(!P->comm || P->reduced_in_schur, RCC_NOT_READY, "reduced system not summed over the ranks");
  {
    Scoped t(P, ST_MASK, 3);
    MaskArgs m{n, P->ld, P->radius_used, P->min_diag, P->max_diag, P->jacobi, P->const_idx.p, P->n_const, P->S.p, P->rhs.p,
               P->d2f.p, P->gFm.p};
    launch_mask_damp(m, P->stream);
    copy_scalar_kernel<<<1, 1, 0, P->stream>>>(P->S.p + (size_t)n * P->ld + 2 * n, P->stats.p + SX_COST2);
  }
  {
    // Bordered factorisation: the rhs already sits in column n of the row-major upper triangle, i.e. in row n
    // of the column-major lower triangle cuSOLVER sees.  Factoring the (n+1) x (n+1) matrix [[S, b], [b^T, big]]
    // leaves y = L^-1 b in that row -- the forward substitution comes out of potrf for free -- and one
    // triangular solve L^T x = -y remains (cusolverDnDpotrs would run two).
    Scoped t(P, ST_CHOLESKY, 4);
    factor_reduced(P, true);
    extract_rhs_kernel<<<ceil_div(n, 256), 256, 0, P->stream>>>(P->S.p, n, P->ld, P->rhs.p);
    RCC_CUDA(cudaGetLastError());
    // hand-written back-substitution (dense.cu K5d) where it is the faster one: 0.49 / 0.98 / 2.63 ms against
    // cublasDtrsv's 0.59 / 1.16 / 3.08 ms at n = 6 030 / 12 060 / 30 009, but 0.25 against 0.23 ms at n = 3 009 (the
    // hand-off between the 128-row blocks costs ~10 us each).  RCC_TRSV = own | cublas overrides.
    const char* tv = getenv("RCC_TRSV");
    const bool own_trsv = tv ? std::string(tv) == "own" : n >= 4500;
    if (own_trsv) {
      P->trsv_inv.ensure(chol_trsv_workspace_doubles(n));
      P->trsv_flags.ensure((size_t)chol_trsv_flags(n));
      chol_trsv(P->S.p, P->ld, n, P->rhs.p, P->trsv_inv.p, P->trsv_flags.p, P->stream);
      RCC_CUDA(cudaMemcpyAsync(P->dev_info.p + 1, P->trsv_flags.p + chol_trsv_flags(n) - 1, sizeof(int),
                               cudaMemcpyDeviceToDevice, P->stream));
      P->launch_count += 2;
    } else {
      RCC_BLAS(cublasDtrsv(P->blas, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_T, CUBLAS_DIAG_NON_UNIT, n, P->S.p, P->ld,
                           P->rhs.p, 1));
    }
  }
  {
    Scoped t(P, ST_BACKSUB, 8);
    BacksubArgs b{};
    b.n_e = P->n_e; b.n_f = P->n_f; b.n_shared = P->n_shared; b.n_bb = P->n_bb;
    b.row_ptr = P->row_ptr.p; b.pair_f = P->pair_f.p; b.Y = P->Y.p; b.Yb = P->Yb.p; b.Linv = P->Linv.p;
    b.ge = P->ge.p; b.d2e = P->d2e.p; b.delta_F = P->rhs.p; b.x_e = x_e(P); b.e_count = P->e_count.p;
    b.delta_e = P->delta_e.p; b.partials = P->bs_partials.p;
    launch_backsub(b, P->stream);
    launch_e_stats(P->bs_partials.p, P->n_e, P->stats.p + SX_MCC_E, P->stream);
    gmax_kernel<<<1, 256, 0, P->stream>>>(P->ge.p, P->e_const.p, P->n_e, P->stats.p + SX_GMAX_E);
    launch_f_stats(P->gFm.p, P->d2f.p, P->rhs.p, x_f(P), P->shared.p, P->n_f, P->n_shared, P->stats.p + SX_MCC_F,
                   P->stream);
    gmaxf_kernel<<<1, 256, 0, P->stream>>>(P->gFm.p, n, P->stats.p + SX_GMAX_F);
    // candidate x + delta
    launch_apply(x_e(P), P->delta_e.p, x_e(P, true), (int64_t)P->n_e * 6, P->stream);
    launch_apply(x_f(P), P->rhs.p, x_f(P, true), (int64_t)P->n_f * 6, P->stream);
    launch_apply(P->shared.p, P->rhs.p + (size_t)6 * P->n_f, P->shared_c.p, P->n_shared, P->stream);
    RCC_CUDA(cudaGetLastError());
  }
  P->schur_done = false;  // S now holds the Cholesky factor
  P->step_ready = true;
  P->cand_ready = false;
}

// ---------------------------------------------------------------------------
// parameter covariance (rcc_ba_covariance)
// ---------------------------------------------------------------------------
// A free parameter whose Cholesky pivot keeps less than this fraction of its diagonal entry is taken as undetermined:
// J^T J without a gauge held constant factors in FP64 with pivots of about +-1e-11 of their diagonal there instead of
// an exact zero, while the determined problems of the test scenes keep 1e-4 or more.
constexpr double COV_MIN_PIVOT = 1e-10;

__global__ void save_diag_kernel(const double* __restrict__ S, int n, int ld, double* __restrict__ d) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] = S[(size_t)i * ld + i];
}
__global__ void pivot_check_kernel(const double* __restrict__ L, int n, int ld, const double* __restrict__ d,
                                   int32_t* flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double l = L[(size_t)i * ld + i];
  if (!(l * l >= COV_MIN_PIVOT * d[i])) *flag = 1;
}
// the mask left a unit diagonal on every constant parameter, which the inverse keeps: zero it
__global__ void zero_const_diag_kernel(double* S, int ld, const int32_t* __restrict__ idx, int n_const) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_const) S[(size_t)idx[i] * ld + idx[i]] = 0.0;
}

enum { CI_POTRF = 0, CI_POTRI, CI_HEE_PIVOT, CI_S_PIVOT, CI_N };

static void require_single_rank(P_t* P) {
  RCC_REQUIRE(!(P->comm && P->n_ranks > 1), RCC_BAD_ARG,
              "covariance is computed on a single rank only; this handle has a communicator of several ranks");
}

// The part every covariance call shares: linearise, the undamped reduced system with the constants masked, its
// factorisation with the pivot checks, and potri.  Leaves S^-1 in the upper triangle of P->S, with a unit diagonal
// still on the constant parameters (zero_const_diag clears it).
static void covariance_inverse(P_t* P) {
  const int n = P->n_red;
  cudaStream_t s = P->stream;
  P->cov_info.ensure(CI_N);
  RCC_CUDA(cudaMemsetAsync(P->cov_info.p, 0, CI_N * sizeof(int32_t), s));
  do_linearize(P);
  // an infinite radius makes every LM diagonal exactly zero (lm_diagonal divides by it): the undamped system
  do_schur(P, INFINITY, P->cov_info.p + CI_HEE_PIVOT);
  {
    Scoped t(P, ST_MASK, P->n_const > 0 ? 2 : 1);
    MaskArgs m{n, P->ld, INFINITY, P->min_diag, P->max_diag, P->jacobi, P->const_idx.p, P->n_const, P->S.p, P->rhs.p,
               P->d2f.p, P->gFm.p};
    launch_mask_damp(m, s);
  }
  P->schur_done = P->step_ready = P->cand_ready = false;   // S is about to become the factor, then the inverse
  P->cov_diag.ensure((size_t)n);
  {
    Scoped t(P, ST_CHOLESKY, 4);
    save_diag_kernel<<<ceil_div(n, 256), 256, 0, s>>>(P->S.p, n, P->ld, P->cov_diag.p);
    factor_reduced(P, false);
    pivot_check_kernel<<<ceil_div(n, 256), 256, 0, s>>>(P->S.p, n, P->ld, P->cov_diag.p, P->cov_info.p + CI_S_PIVOT);
    RCC_CUDA(cudaMemcpyAsync(P->cov_info.p + CI_POTRF, P->dev_info.p, sizeof(int), cudaMemcpyDeviceToDevice, s));
    RCC_CUDA(cudaGetLastError());
  }
  int32_t* hi = reinterpret_cast<int32_t*>(P->h_pinned + 32);
  RCC_CUDA(cudaMemcpyAsync(hi, P->cov_info.p, CI_N * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  RCC_CUDA(cudaMemcpyAsync(hi + CI_N, P->fail_flag.p, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  sync(P);
  if (hi[CI_N]) throw Error(RCC_EVAL_FAILED, "evaluation failed: corner behind the camera or non-finite residual");
  if (hi[CI_HEE_PIVOT])
    throw Error(RCC_NOT_SPD, "J^T J is not positive definite: an eliminated block's H_ee has a non-positive pivot");
  if (hi[CI_POTRF] != 0 || hi[CI_S_PIVOT])
    throw Error(RCC_NOT_SPD, "J^T J is not positive definite: the reduced system has a non-positive or vanishing pivot"
                             " (potrf info " + std::to_string(hi[CI_POTRF]) + ")");
  {
    Scoped t(P, ST_INVERSE, 1);
    int lwork = 0;
    RCC_SOLVER(cusolverDnDpotri_bufferSize(P->solver, CUBLAS_FILL_MODE_LOWER, n, P->S.p, P->ld, &lwork));
    P->potrf_work.ensure((size_t)std::max(lwork, P->potrf_lwork));
    RCC_SOLVER(cusolverDnDpotri(P->solver, CUBLAS_FILL_MODE_LOWER, n, P->S.p, P->ld, P->potrf_work.p, lwork,
                                P->cov_info.p + CI_POTRI));
  }
}

// one launch when there are constants (counted by the caller's Scoped)
static void zero_const_diag(P_t* P) {
  if (P->n_const > 0)
    zero_const_diag_kernel<<<ceil_div(P->n_const, 256), 256, 0, P->stream>>>(P->S.p, P->ld, P->const_idx.p,
                                                                              P->n_const);
}

static CovArgs cov_args(P_t* P) {
  CovArgs c{};
  c.n_e = P->n_e; c.n_f = P->n_f; c.n_shared = P->n_shared; c.n_bb = P->n_bb; c.n = P->n_red; c.ld = P->ld;
  c.row_ptr = P->row_ptr.p; c.pair_f = P->pair_f.p; c.Y = P->Y.p; c.Yb = P->Yb.p; c.Linv = P->Linv.p; c.Sinv = P->S.p;
  c.cov_e = P->cov_e.p; c.cov_f = P->cov_f.p; c.cov_s = P->cov_s.p;
  return c;
}

// after the caller's downloads: wait for them and report a failed potri
static void covariance_finish(P_t* P) {
  int32_t* hi = reinterpret_cast<int32_t*>(P->h_pinned + 32);
  RCC_CUDA(cudaMemcpyAsync(hi, P->cov_info.p, CI_N * sizeof(int32_t), cudaMemcpyDeviceToHost, P->stream));
  sync(P);
  if (hi[CI_POTRI] != 0)
    throw Error(RCC_NOT_SPD, "inverse of the reduced system: potri info " + std::to_string(hi[CI_POTRI]));
}

static void do_covariance(P_t* P, double* cov_shared, double* cov_views, double* cov_markers) {
  require_single_rank(P);
  cudaStream_t s = P->stream;
  covariance_inverse(P);
  P->cov_e.ensure((size_t)P->n_e * 36);
  P->cov_f.ensure((size_t)P->n_f * 36);
  P->cov_s.ensure((size_t)P->n_shared * P->n_shared);
  const CovArgs c = cov_args(P);
  {
    Scoped t(P, ST_COVARIANCE, P->n_const > 0 ? 2 : 1);
    zero_const_diag(P);
    launch_cov_eliminated(c, s);
  }
  {
    Scoped t(P, ST_COV_EXTRACT, 1);
    launch_cov_kept(c, s);
  }
  double* ce = P->elim_view ? cov_views : cov_markers;
  double* cf = P->elim_view ? cov_markers : cov_views;
  if (ce) P->cov_e.download(ce, (size_t)P->n_e * 36, s);
  if (cf) P->cov_f.download(cf, (size_t)P->n_f * 36, s);
  if (cov_shared) P->cov_s.download(cov_shared, (size_t)P->n_shared * P->n_shared, s);
  covariance_finish(P);
}

// A launch of the pair kernels covers whole pairs and at most about this many work items (36 doubles of partials
// each), so that the scratch stays bounded however many pairs one call requests.
constexpr int64_t COV_PAIR_BATCH_ITEMS = 1 << 20;

static void do_covariance_blocks(P_t* P, int64_t n_pairs, const int32_t* pairs, double* out) {
  RCC_REQUIRE(n_pairs >= 0 && n_pairs <= INT32_MAX / 36, RCC_BAD_ARG, "n_pairs out of range");
  RCC_REQUIRE(n_pairs == 0 || (pairs && out), RCC_BAD_ARG, "null pointer");
  require_single_rank(P);
  // a side of a pair: an eliminated block (e >= 0, K partners) or a kept or shared block (reduced columns [g, g + w))
  struct Side { int e, g, w, K; };
  auto side = [&](int32_t kind, int32_t index) -> Side {
    int count = 0;
    switch (kind) {
      case RCC_BLOCK_VIEW: count = P->n_views; break;
      case RCC_BLOCK_MARKER: count = P->n_markers; break;
      case RCC_BLOCK_INTR: case RCC_BLOCK_DIST: count = P->n_cam; break;
      case RCC_BLOCK_EXT:
        RCC_REQUIRE(P->rig, RCC_BAD_ARG, "RCC_BLOCK_EXT needs the rig model");
        count = P->n_cam;
        break;
      default: throw Error(RCC_BAD_ARG, "unknown block kind " + std::to_string(kind));
    }
    RCC_REQUIRE(index >= 0 && index < count, RCC_BAD_ARG, "block index out of range");
    if (kind == RCC_BLOCK_VIEW || kind == RCC_BLOCK_MARKER) {
      if ((kind == RCC_BLOCK_VIEW) == P->elim_view) return Side{index, 0, 6, 0};
      return Side{-1, 6 * index, 6, 1};
    }
    const int g = 6 * P->n_f + P->sp * index;
    if (kind == RCC_BLOCK_INTR) return Side{-1, g, 4, 1};
    if (kind == RCC_BLOCK_DIST) return Side{-1, g + 4, 5, 1};
    return Side{-1, g + 9, 6, 1};
  };
  std::vector<Side> sa((size_t)n_pairs), sb((size_t)n_pairs);
  for (int64_t p = 0; p < n_pairs; ++p) {
    sa[p] = side(pairs[4 * p], pairs[4 * p + 1]);
    sb[p] = side(pairs[4 * p + 2], pairs[4 * p + 3]);
  }
  if (n_pairs == 0) return;
  RCC_REQUIRE(P->have_obs && (int64_t)P->row_ptr_h.size() == (int64_t)P->n_e + 1, RCC_NOT_READY,
              "observations have not been set");
  for (int64_t p = 0; p < n_pairs; ++p)
    for (Side* x : {&sa[p], &sb[p]})
      if (x->e >= 0) x->K = P->row_ptr_h[x->e + 1] - P->row_ptr_h[x->e] + P->n_bb;

  // canonical order: side b has the more items (ties: the larger block), so that the lanes of an item run over the
  // long side; the request (b, a) is then written as the transpose of Cov(a, b)
  std::vector<CovPairDesc> desc((size_t)n_pairs);
  std::vector<CovPairItem> items;
  std::vector<int64_t> batch_pair{0}, batch_item{0};
  auto key = [](const Side& x) { return std::make_tuple(x.K, x.e >= 0, x.e >= 0 ? x.e : x.g); };
  for (int64_t p = 0; p < n_pairs; ++p) {
    Side a = sa[p], b = sb[p];
    const bool swap = key(a) > key(b);
    if (swap) std::swap(a, b);
    const int64_t n_items = (int64_t)ceil_div(a.K, COV_PAIR_CHUNK) * ceil_div(b.K, 32);
    if ((int64_t)items.size() - batch_item.back() + n_items > COV_PAIR_BATCH_ITEMS && p > batch_pair.back()) {
      batch_pair.push_back(p);
      batch_item.push_back((int64_t)items.size());
    }
    CovPairDesc& d = desc[p];
    d.e_a = a.e; d.e_b = b.e; d.g_a = a.g; d.w_a = a.w; d.g_b = b.g; d.w_b = b.w;
    d.item0 = (int32_t)((int64_t)items.size() - batch_item.back());
    d.n_items = (int32_t)n_items;
    d.rows = a.w; d.cols = b.w; d.transpose = swap ? 1 : 0;
    for (int k0 = 0; k0 < a.K; k0 += COV_PAIR_CHUNK)
      for (int l0 = 0; l0 < b.K; l0 += 32) items.push_back(CovPairItem{(int32_t)p, k0, l0});
  }
  batch_pair.push_back(n_pairs);
  batch_item.push_back((int64_t)items.size());
  const int n_batches = (int)batch_pair.size() - 1;

  cudaStream_t s = P->stream;
  covariance_inverse(P);
  int64_t max_items = 0;
  for (int b = 0; b < n_batches; ++b) max_items = std::max(max_items, batch_item[b + 1] - batch_item[b]);
  P->cov_desc.upload(desc.data(), desc.size(), s);
  P->cov_items.upload(items.data(), items.size(), s);
  P->cov_partial.ensure((size_t)max_items * 36);
  P->cov_out.ensure((size_t)n_pairs * 36);
  CovPairsArgs c{};
  c.m = cov_args(P);
  c.pairs = P->cov_desc.p;
  c.partial = P->cov_partial.p;
  c.out = P->cov_out.p;
  {
    Scoped t(P, ST_COVARIANCE, (P->n_const > 0 ? 1 : 0) + 2 * n_batches);
    zero_const_diag(P);
    for (int b = 0; b < n_batches; ++b) {
      c.items = P->cov_items.p + batch_item[b];
      c.pair_begin = (int32_t)batch_pair[b];
      c.n_pairs = (int32_t)(batch_pair[b + 1] - batch_pair[b]);
      c.n_items = (int32_t)(batch_item[b + 1] - batch_item[b]);
      launch_cov_pairs(c, s);
    }
  }
  P->cov_out.download(out, (size_t)n_pairs * 36, s);
  covariance_finish(P);
}

static EvalArgs eval_args(P_t* P, bool cand) {
  EvalArgs a{};
  a.n = P->n_obs;
  a.view_idx = P->elim_view ? P->e_own.p : P->e_oth.p;
  a.marker_idx = P->elim_view ? P->e_oth.p : P->e_own.p;
  a.cam = P->e_cam.p;
  a.orig = P->e_orig.p;
  a.pix = P->e_pix.p;
  a.view_x = cand ? P->view_xc.p : P->view_x.p;
  a.marker_x = cand ? P->marker_xc.p : P->marker_x.p;
  a.ext_x = cand ? P->ext_xc.p : P->ext_x.p;
  a.shared = cand ? P->shared_c.p : P->shared.p;
  a.cost2_partials = P->cost_partials.p;
  a.chunks = P->e_chunks.p;
  a.n_chunks = P->n_chunks_e;
  a.oth = P->e_oth.p;
  a.own_is_view = P->elim_view ? 1 : 0;
  a.fail_flag = P->fail_flag.p;
  a.loss = P->loss;
  a.loss_a2 = P->loss_scale * P->loss_scale;
  a.cam_equidistant = P->cam_equidistant;
  if (P->n_slots > 0) {   // the target instantiations of K1 and K6
    a.slot = P->e_slot.p;
    a.corners = P->corners.p;
  }
  return a;
}

static void do_candidate_cost(P_t* P) {
  RCC_REQUIRE(P->step_ready, RCC_NOT_READY, "solve_step has not been called");
  ensure_pixels(P);
  {
    Scoped t(P, ST_EXPAND, 1);
    launch_expand_poses(P->views_c.p, P->n_views, P->view_xc.p, P->markers_c.p, P->sizes.p, P->n_markers, P->marker_xc.p,
                        P->shared_c.p, P->n_cam, P->sp, P->ext_xc.p, P->stream);
  }
  {
    Scoped t(P, ST_COST, P->n_prior_parts > 0 ? 3 : 2);
    EvalArgs a = eval_args(P, true);
    a.fail_flag = P->fail_flag.p + 1;   // slot 1: candidate point (slot 0 keeps the linearisation point's flag)
    RCC_CUDA(cudaMemsetAsync(a.fail_flag, 0, sizeof(int32_t), P->stream));
    launch_cost(P->rig, handle_lens(P), a, P->stream);
    const int np = eval_grid(P->n_obs);
    if (P->n_prior_parts > 0) launch_prior(false, prior_args(P, true, P->cost_partials.p + np), P->stream);
    launch_sum(P->cost_partials.p, np + P->n_prior_parts, P->stats.p + SX_CAND2, 1.0, P->stream);
  }
  if (P->comm) {
    Scoped t(P, ST_ALLREDUCE, 2);
    RCC_NCCL(ncclAllReduce(P->stats.p + SX_MCC_E, P->stats.p + SX_MCC_E, 4, ncclDouble, ncclSum, P->comm, P->stream));
    RCC_NCCL(ncclAllReduce(P->stats.p + SX_GMAX_E, P->stats.p + SX_GMAX_E, 1, ncclDouble, ncclMax, P->comm, P->stream));
    // both fail flags (linearisation point, candidate point) must be seen by every rank
    RCC_NCCL(ncclAllReduce(P->fail_flag.p, P->fail_flag.p, 2, ncclInt32, ncclMax, P->comm, P->stream));
  }
  P->cand_ready = true;
}

struct StepScalars {
  double mcc, step_norm, x_norm, cand_cost, cur_cost, gmax;
  int potrf_info, fail, fail_lin;   // fail: candidate point; fail_lin: the point the system was linearised at
};

static StepScalars read_step_scalars(P_t* P) {
  double* h = P->h_pinned;
  RCC_CUDA(cudaMemcpyAsync(h, P->stats.p, SX_N * sizeof(double), cudaMemcpyDeviceToHost, P->stream));
  int* hi = reinterpret_cast<int*>(h + 16);
  RCC_CUDA(cudaMemcpyAsync(hi, P->dev_info.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, P->stream));
  RCC_CUDA(cudaMemcpyAsync(hi + 2, P->fail_flag.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, P->stream));
  sync(P);
  StepScalars s;
  s.mcc = h[SX_MCC_E] + h[SX_MCC_F];
  s.step_norm = std::sqrt(h[SX_DN_E] + h[SX_DN_F]);
  s.x_norm = std::sqrt(h[SX_XN_E] + h[SX_XN_F]);
  s.cand_cost = 0.5 * h[SX_CAND2];
  s.cur_cost = 0.5 * h[SX_COST2];
  s.gmax = std::max(h[SX_GMAX_E], h[SX_GMAX_F]);
  s.potrf_info = hi[0] != 0 ? hi[0] : (hi[1] != 0 ? -1 : 0);   // hi[1]: the back-substitution gave up waiting (never expected)
  s.fail_lin = hi[2];
  s.fail = hi[3];
  return s;
}

static void do_accept(P_t* P) {
  RCC_REQUIRE(P->step_ready, RCC_NOT_READY, "no step to accept");
  std::swap(P->views.p, P->views_c.p);
  std::swap(P->markers.p, P->markers_c.p);
  std::swap(P->shared.p, P->shared_c.p);
  if (P->cand_ready) {
    std::swap(P->view_x.p, P->view_xc.p);
    std::swap(P->marker_x.p, P->marker_xc.p);
    std::swap(P->ext_x.p, P->ext_xc.p);
    P->expanded_valid = true;
  } else {
    P->expanded_valid = false;
  }
  P->linearized = P->schur_done = P->step_ready = P->cand_ready = false;
}

static void do_solve(P_t* P, const rcc_lm_options& o, rcc_lm_summary& sum) {
  memset(&sum, 0, sizeof(sum));
  P->min_diag = o.min_diagonal;
  P->max_diag = o.max_diagonal;
  P->jacobi = o.jacobi_scaling ? 1 : 0;
  double radius = o.initial_radius, decrease = 2.0;
  bool need_lin = true;
  const bool was_on = P->timer.on;
  P->timer.reset();
  P->timer.on = true;
  cudaEvent_t e0 = P->timer.get(), e1 = P->timer.get();
  RCC_CUDA(cudaEventRecord(e0, P->stream));
  sum.termination = 0;
  double cost = 0.0;
  int it = 0;
  for (; it < o.max_iterations; ++it) {
    if (need_lin) do_linearize(P);
    do_schur(P, radius);
    do_step(P);
    do_candidate_cost(P);
    StepScalars s = read_step_scalars(P);
    cost = s.cur_cost;
    if (it == 0) sum.initial_cost = cost;
    sum.final_gradient_max = s.gmax;
    if (s.fail_lin || !std::isfinite(cost)) {
      // the current point itself cannot be evaluated (corner at depth <= 0, non-finite residual): H and g are
      // garbage, so stop -- Ceres returns FAILURE when the initial evaluation fails
      if (o.verbose) fprintf(stderr, "[rcc_ba] it %3d evaluation failed at the linearisation point\n", it);
      sum.termination = 4;
      break;
    }
    if (need_lin && s.gmax < o.gradient_tolerance) {
      sum.termination = 2;
      break;
    }
    const bool solved = (s.potrf_info == 0) && std::isfinite(s.step_norm);
    if (solved && s.step_norm <= o.parameter_tolerance * (s.x_norm + o.parameter_tolerance)) {
      sum.termination = 3;
      break;
    }
    const bool valid = solved && !s.fail && std::isfinite(s.cand_cost) && s.mcc > 0;
    const double rho = valid ? (cost - s.cand_cost) / s.mcc : -1.0;
    if (o.verbose)
      fprintf(stderr, "[rcc_ba] it %3d cost %.9e -> %.9e rho %.4f radius %.3e |g| %.3e |dx| %.3e%s\n", it, cost,
              s.cand_cost, rho, radius, s.gmax, s.step_norm, solved ? "" : " (factorisation failed)");
    if (valid && rho > o.min_relative_decrease) {
      do_accept(P);
      sum.accepted++;
      need_lin = true;
      radius = std::min(o.max_radius, radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * rho - 1.0, 3)));
      decrease = 2.0;
      const double dc = std::fabs(cost - s.cand_cost);
      cost = s.cand_cost;
      if (dc <= o.function_tolerance * std::fabs(s.cur_cost)) {
        sum.termination = 1;
        ++it;
        break;
      }
    } else {
      radius /= decrease;
      decrease *= 2.0;
      need_lin = false;
      P->step_ready = P->cand_ready = false;
      if (radius < 1e-32) {
        sum.termination = 4;
        break;
      }
    }
  }
  RCC_CUDA(cudaEventRecord(e1, P->stream));
  sync(P);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  P->timer.pool.push_back(e0);
  P->timer.pool.push_back(e1);
  P->timer.collect();
  sum.iterations = it;
  sum.final_cost = cost;
  sum.final_radius = radius;
  sum.total_ms = ms;
  const double* m = P->timer.ms;
  sum.linearize_ms = m[ST_EXPAND] + m[ST_ASSEMBLE_E] + m[ST_ASSEMBLE_F] + m[ST_FINALIZE];
  sum.schur_ms = m[ST_SCHUR_PREP] + m[ST_SCHUR_SYRK] + m[ST_SCHUR_SHARED];
  sum.allreduce_ms = m[ST_ALLREDUCE];
  sum.solve_ms = m[ST_MASK] + m[ST_CHOLESKY];
  sum.backsub_ms = m[ST_BACKSUB];
  sum.cost_ms = m[ST_COST];
  P->timer.on = was_on;
}

// ---------------------------------------------------------------------------
// extern "C" boundary
// ---------------------------------------------------------------------------
// caller's pixels (FP64 or integer, caller order) -> e_pix and f_pix
template <typename T>
static void load_pixels(P_t* P, const T* pixels, bool piecewise) {
  if (piecewise) {
    // caller order is the E-sorted order: copy on the side streams in pieces cut at chunk boundaries, FP64 straight
    // into e_pix; linearize overlaps its E pass with the pieces still in flight
    constexpr bool f64 = std::is_same<T, double>::value;
    if (!f64) P->staging.ensure((size_t)P->n_obs * 8 * sizeof(T));
    T* dst = f64 ? reinterpret_cast<T*>(P->e_pix.p) : reinterpret_cast<T*>(P->staging.p);
    Scoped t(P, ST_H2D, 0);
    RCC_CUDA(cudaEventRecord(P->ev_fork, P->stream));          // earlier readers of e_pix on the main stream
    RCC_CUDA(cudaStreamWaitEvent(P->side_stream, P->ev_fork, 0));
    RCC_CUDA(cudaStreamWaitEvent(P->side_stream2, P->ev_fork, 0));
    for (int k = 0; k < rcc_ba_problem::PIX_PIECES; ++k) {
      // pieces alternate between two streams: two copy engines in flight keep the link busier (48 -> 52 GB/s)
      cudaStream_t cs = (k & 1) ? P->side_stream2 : P->side_stream;
      const int64_t b0 = P->piece_block[k], b1 = P->piece_block[k + 1];
      if (b1 > b0) {
        RCC_CUDA(cudaMemcpyAsync(dst + b0 * 8, pixels + b0 * 8, (size_t)(b1 - b0) * 8 * sizeof(T),
                                 cudaMemcpyHostToDevice, cs));
        launch_load_pixels<T>(f64 ? nullptr : dst + b0 * 8, nullptr, P->e_pix.p + b0 * 8, P->f_inv.p + b0, P->f_pix.p,
                              b1 - b0, cs);
        P->launch_count += 1;
      }
      RCC_CUDA(cudaEventRecord(P->ev_piece[k], cs));
    }
    P->pix_pending = true;
  } else {
    const size_t bytes = (size_t)P->n_obs * 8 * sizeof(T);
    Scoped t(P, ST_H2D, P->n_obs > 0 ? 1 : 0);
    P->staging.ensure(bytes);
    if (bytes) RCC_CUDA(cudaMemcpyAsync(P->staging.p, pixels, bytes, cudaMemcpyHostToDevice, P->stream));
    launch_load_pixels<T>(reinterpret_cast<const T*>(P->staging.p), P->e_orig.p, P->e_pix.p, P->f_inv.p, P->f_pix.p,
                          P->n_obs, P->stream);
  }
}

template <typename T>
static void set_observations(P_t* P, const int32_t* view_idx, const int32_t* marker_idx, const int32_t* cam_idx,
                             const T* pixels) {
  RCC_REQUIRE(view_idx && marker_idx && pixels, RCC_BAD_ARG, "null pointer");
  build_indices(P, view_idx, marker_idx, cam_idx);
  load_pixels(P, pixels, false);
  RCC_CUDA(cudaStreamSynchronize(P->stream));
  P->staging.release();   // only needed again by a later update_pixels that goes through it
}

template <typename T>
static void update_pixels(P_t* P, const T* pixels) {
  RCC_REQUIRE(pixels, RCC_BAD_ARG, "null pointer");
  RCC_REQUIRE(P->have_obs, RCC_NOT_READY, "set_observations has not been called");
  load_pixels(P, pixels, P->pix_identity);
  P->linearized = P->schur_done = P->step_ready = P->cand_ready = false;
}

static thread_local std::string g_create_error;

// 6-wide column blocks of the dense border of the reduced system: the shared parameters and the right-hand side.
// The border kernels hold at most 128 columns (schur_border_kernel: SB_MAXPASS passes of 32).
static int64_t border_blocks(int64_t n_shared) { return (n_shared + 1 + 5) / 6; }

#define API_BEGIN(P)                                     \
  if (!(P)) return RCC_BAD_ARG;                          \
  try {                                                  \
    RCC_CUDA(cudaSetDevice((P)->opt.device));
#define API_END(P)                                       \
  }                                                      \
  catch (const Error& e) {                               \
    (P)->err = e.what();                                 \
    return e.status;                                     \
  }                                                      \
  catch (const std::exception& e) {                      \
    (P)->err = e.what();                                 \
    return RCC_BAD_ARG;                                  \
  }                                                      \
  return RCC_OK;

extern "C" {

const char* rcc_ba_version(void) { return "rcc_ba 0.1.0 sm_100a fp64 (cuda " RCC_STR(CUDART_VERSION) ")"; }

void rcc_lm_default_options(rcc_lm_options* o) {
  if (!o) return;
  o->max_iterations = 50;
  o->initial_radius = 1e4;
  o->max_radius = 1e16;
  o->min_relative_decrease = 1e-3;
  o->function_tolerance = 1e-6;
  o->gradient_tolerance = 1e-10;
  o->parameter_tolerance = 1e-8;
  o->min_diagonal = 1e-6;
  o->max_diagonal = 1e32;
  o->verbose = 0;
  o->jacobi_scaling = 1;
}

int rcc_ba_create(const rcc_ba_options* opt, rcc_ba_problem** out) {
  if (!opt || !out) return RCC_BAD_ARG;
  *out = nullptr;
  if (opt->n_views <= 0 || opt->n_markers <= 0 || opt->n_cameras <= 0 || opt->n_obs_blocks < 0 ||
      (opt->model != RCC_MODEL_SINGLE && opt->model != RCC_MODEL_RIG))
    return RCC_BAD_ARG;
  const int sp = opt->model == RCC_MODEL_RIG ? 15 : 9;
  if (border_blocks((int64_t)opt->n_cameras * sp) * 6 > 128) {
    g_create_error = "too many cameras: the shared border holds at most 125 parameters (8 rig or 13 single-model cameras)";
    fprintf(stderr, "[rcc_ba] create failed: %s\n", g_create_error.c_str());
    return RCC_BAD_ARG;
  }
  P_t* P = new P_t();
  try {
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
      throw Error(RCC_CUDA_ERROR, std::string("no CUDA device: ") + cudaGetErrorString(ce) +
                                      " (this library has no CPU fallback)");
    RCC_REQUIRE(opt->device >= 0 && opt->device < ndev, RCC_BAD_ARG, "device ordinal out of range");
    RCC_CUDA(cudaSetDevice(opt->device));
    cudaDeviceProp prop;
    RCC_CUDA(cudaGetDeviceProperties(&prop, opt->device));
    RCC_REQUIRE(prop.major == 10, RCC_CUDA_ERROR,
                std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                    "; this library carries sm_100a code only");
    P->opt = *opt;
    P->rig = opt->model == RCC_MODEL_RIG;
    P->sp = sp;
    P->n_cam = opt->n_cameras;
    P->n_shared = P->n_cam * P->sp;
    P->fin_slices = fin_slices(prop.multiProcessorCount, P->n_cam);
    P->n_views = opt->n_views;
    P->n_markers = opt->n_markers;
    P->n_obs = opt->n_obs_blocks;
    P->elim_view = opt->eliminate == RCC_ELIM_VIEWS || (opt->eliminate == RCC_ELIM_AUTO && opt->n_views >= opt->n_markers);
    P->n_e = P->elim_view ? P->n_views : P->n_markers;
    P->n_f = P->elim_view ? P->n_markers : P->n_views;
    P->n_bb = (int)border_blocks(P->n_shared);
    P->n_red = 6 * P->n_f + P->n_shared;
    P->ld = 6 * P->n_f + 6 * P->n_bb;
    RCC_REQUIRE((int64_t)P->n_red * P->ld < (int64_t)1 << 40, RCC_BAD_ARG, "reduced system too large");
    RCC_CUDA(cudaStreamCreateWithFlags(&P->stream, cudaStreamNonBlocking));
    P->own_stream = true;
    RCC_CUDA(cudaStreamCreateWithFlags(&P->side_stream, cudaStreamNonBlocking));
    RCC_CUDA(cudaStreamCreateWithFlags(&P->side_stream2, cudaStreamNonBlocking));
    RCC_CUDA(cudaEventCreateWithFlags(&P->ev_fork, cudaEventDisableTiming));
    RCC_CUDA(cudaEventCreateWithFlags(&P->ev_join, cudaEventDisableTiming));
    for (auto& e : P->ev_piece) RCC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    RCC_CUDA(cudaMallocHost(&P->h_pinned, 64 * sizeof(double)));
    cudaStream_t s = P->stream;
    P->views.alloc((size_t)P->n_views * 6); P->views.zero(s);
    P->views_c.alloc((size_t)P->n_views * 6); P->views_c.zero(s);
    P->markers.alloc((size_t)P->n_markers * 6); P->markers.zero(s);
    P->markers_c.alloc((size_t)P->n_markers * 6); P->markers_c.zero(s);
    P->sizes.alloc((size_t)P->n_markers); P->sizes.zero(s);
    P->shared.alloc((size_t)P->n_shared); P->shared.zero(s);
    P->shared_c.alloc((size_t)P->n_shared); P->shared_c.zero(s);
    P->view_x.alloc((size_t)P->n_views * POSEX); P->view_xc.alloc((size_t)P->n_views * POSEX);
    P->marker_x.alloc((size_t)P->n_markers * POSEX); P->marker_xc.alloc((size_t)P->n_markers * POSEX);
    P->ext_x.alloc((size_t)P->n_cam * POSEX); P->ext_xc.alloc((size_t)P->n_cam * POSEX);
    P->c_view.assign(P->n_views, 0); P->c_marker.assign(P->n_markers, 0);
    P->c_intr.assign(P->n_cam, 0); P->c_dist.assign(P->n_cam, 0); P->c_ext.assign(P->n_cam, 0);
    P->cam_lens.assign(P->n_cam, LENS_RADTAN);
    P->Hee.alloc((size_t)P->n_e * 36); P->ge.alloc((size_t)P->n_e * 6); P->Hes.alloc((size_t)P->n_e * 6 * P->n_shared);
    P->Hff.alloc((size_t)P->n_f * 36); P->gf.alloc((size_t)P->n_f * 6); P->Hfs.alloc((size_t)P->n_f * 6 * P->n_shared);
    P->fin_scratch.alloc((size_t)P->n_cam * P->fin_slices * PassGeom<true>::PART_E);
    P->fin_done.alloc((size_t)P->n_cam); P->fin_done.zero(s);
    P->Hss.alloc((size_t)P->n_shared * P->n_shared); P->gs.alloc((size_t)P->n_shared); P->cost2_cam.alloc(P->n_cam);
    P->Linv.alloc((size_t)P->n_e * 36); P->Yb.alloc((size_t)P->n_e * P->n_bb * 36); P->d2e.alloc((size_t)P->n_e * 6);
    P->S.alloc((size_t)(P->n_red + 3) * P->ld); P->S.zero(s);
    P->shared_scratch.alloc((size_t)SHARED_SLICES * (6 * P->n_bb) * (6 * P->n_bb));
    P->rhs.alloc(P->n_red); P->d2f.alloc(P->n_red); P->gFm.alloc(P->n_red);
    P->delta_e.alloc((size_t)P->n_e * 6); P->delta_e.zero(s);
    P->bs_partials.alloc((size_t)P->n_e * 4);
    P->stats.alloc(16); P->stats.zero(s);
    P->fail_flag.alloc(4); P->fail_flag.zero(s);
    P->dev_info.alloc(2); P->dev_info.zero(s);
    P->scalar.alloc(8);
    RCC_SOLVER(cusolverDnCreate(&P->solver));
    RCC_SOLVER(cusolverDnSetStream(P->solver, s));
    RCC_SOLVER(cusolverDnDpotrf_bufferSize(P->solver, CUBLAS_FILL_MODE_LOWER, P->n_red + 1, P->S.p, P->ld,
                                           &P->potrf_lwork));   // + the border row (see do_step)
    RCC_BLAS(cublasCreate(&P->blas));
    RCC_BLAS(cublasSetStream(P->blas, s));
    P->potrf_work.alloc((size_t)std::max(1, P->potrf_lwork));
    RCC_CUDA(cudaStreamSynchronize(s));
  } catch (const Error& e) {
    g_create_error = e.what();
    fprintf(stderr, "[rcc_ba] create failed: %s\n", e.what());
    int st = e.status;
    delete P;
    return st;
  }
  *out = P;
  return RCC_OK;
}

void rcc_ba_destroy(rcc_ba_problem* p) {
  if (!p) return;
  cudaSetDevice(p->opt.device);
  if (p->stream) cudaStreamSynchronize(p->stream);
  if (p->side_stream) cudaStreamSynchronize(p->side_stream);
  if (p->side_stream2) cudaStreamSynchronize(p->side_stream2);
  delete p;
}

const char* rcc_ba_last_error(const rcc_ba_problem* p) { return p ? p->err.c_str() : g_create_error.c_str(); }

int rcc_ba_set_stream(rcc_ba_problem* P, void* cuda_stream) {
  API_BEGIN(P)
  sync(P);
  if (P->own_stream && P->stream) cudaStreamDestroy(P->stream);
  P->stream = (cudaStream_t)cuda_stream;
  P->own_stream = false;
  RCC_SOLVER(cusolverDnSetStream(P->solver, P->stream));
  RCC_BLAS(cublasSetStream(P->blas, P->stream));
  API_END(P)
}

static void invalidate(P_t* P) {
  P->expanded_valid = false;
  P->linearized = P->schur_done = P->step_ready = P->cand_ready = false;
}

int rcc_ba_set_intrinsics(rcc_ba_problem* P, const double* intr, const double* dist) {
  API_BEGIN(P)
  RCC_REQUIRE(intr && dist, RCC_BAD_ARG, "null pointer");
  // strided scatter into the per-camera records [fx fy cx cy | k1 k2 p1 p2 k3 | ext]: no read-modify-write, no sync
  const size_t pitch = (size_t)P->sp * sizeof(double);
  const void* hi = stage_in(P, HS_INTR, intr, (size_t)P->n_cam * 4 * sizeof(double));
  RCC_CUDA(cudaMemcpy2DAsync(P->shared.p, pitch, hi, 4 * sizeof(double), 4 * sizeof(double), P->n_cam,
                             cudaMemcpyHostToDevice, P->stream));
  stage_issued(P, HS_INTR);
  const void* hd = stage_in(P, HS_DIST, dist, (size_t)P->n_cam * 5 * sizeof(double));
  RCC_CUDA(cudaMemcpy2DAsync(P->shared.p + 4, pitch, hd, 5 * sizeof(double), 5 * sizeof(double), P->n_cam,
                             cudaMemcpyHostToDevice, P->stream));
  stage_issued(P, HS_DIST);
  invalidate(P);
  API_END(P)
}

int rcc_ba_set_rig_extrinsics(rcc_ba_problem* P, const double* ext) {
  API_BEGIN(P)
  RCC_REQUIRE(ext, RCC_BAD_ARG, "null pointer");
  RCC_REQUIRE(P->rig, RCC_BAD_ARG, "extrinsics exist only in the rig model");
  const void* he = stage_in(P, HS_EXT, ext, (size_t)P->n_cam * 6 * sizeof(double));
  RCC_CUDA(cudaMemcpy2DAsync(P->shared.p + 9, (size_t)P->sp * sizeof(double), he, 6 * sizeof(double), 6 * sizeof(double),
                             P->n_cam, cudaMemcpyHostToDevice, P->stream));
  stage_issued(P, HS_EXT);
  invalidate(P);
  API_END(P)
}

int rcc_ba_set_view_poses(rcc_ba_problem* P, const double* views) {
  API_BEGIN(P)
  RCC_REQUIRE(views, RCC_BAD_ARG, "null pointer");
  Scoped t(P, ST_H2D, 0);
  const size_t bytes = (size_t)P->n_views * 6 * sizeof(double);
  RCC_CUDA(cudaMemcpyAsync(P->views.p, stage_in(P, HS_VIEWS, views, bytes), bytes, cudaMemcpyHostToDevice, P->stream));
  stage_issued(P, HS_VIEWS);
  invalidate(P);
  API_END(P)
}

int rcc_ba_set_marker_poses(rcc_ba_problem* P, const double* markers) {
  API_BEGIN(P)
  RCC_REQUIRE(markers, RCC_BAD_ARG, "null pointer");
  Scoped t(P, ST_H2D, 0);
  const size_t bytes = (size_t)P->n_markers * 6 * sizeof(double);
  RCC_CUDA(cudaMemcpyAsync(P->markers.p, stage_in(P, HS_MARKERS, markers, bytes), bytes, cudaMemcpyHostToDevice,
                           P->stream));
  stage_issued(P, HS_MARKERS);
  invalidate(P);
  API_END(P)
}

int rcc_ba_set_marker_sizes(rcc_ba_problem* P, const double* sizes) {
  API_BEGIN(P)
  RCC_REQUIRE(sizes, RCC_BAD_ARG, "null pointer");
  P->sizes.upload(sizes, (size_t)P->n_markers, P->stream);
  sync(P);
  invalidate(P);
  API_END(P)
}

int rcc_ba_set_observations(rcc_ba_problem* P, const int32_t* view_idx, const int32_t* marker_idx,
                            const int32_t* cam_idx, const double* pixels) {
  API_BEGIN(P)
  set_observations(P, view_idx, marker_idx, cam_idx, pixels);
  API_END(P)
}

int rcc_ba_update_pixels(rcc_ba_problem* P, const double* pixels) {
  API_BEGIN(P)
  update_pixels(P, pixels);
  API_END(P)
}

int rcc_ba_set_observations_i16(rcc_ba_problem* P, const int32_t* view_idx, const int32_t* marker_idx,
                                const int32_t* cam_idx, const int16_t* pixels) {
  API_BEGIN(P)
  set_observations(P, view_idx, marker_idx, cam_idx, pixels);
  API_END(P)
}

int rcc_ba_set_observations_i32(rcc_ba_problem* P, const int32_t* view_idx, const int32_t* marker_idx,
                                const int32_t* cam_idx, const int32_t* pixels) {
  API_BEGIN(P)
  set_observations(P, view_idx, marker_idx, cam_idx, pixels);
  API_END(P)
}

int rcc_ba_update_pixels_i16(rcc_ba_problem* P, const int16_t* pixels) {
  API_BEGIN(P)
  update_pixels(P, pixels);
  API_END(P)
}

int rcc_ba_set_constant(rcc_ba_problem* P, int32_t kind, int32_t index, int32_t is_constant) {
  API_BEGIN(P)
  std::vector<uint8_t>* v = nullptr;
  switch (kind) {
    case RCC_BLOCK_VIEW: v = &P->c_view; break;
    case RCC_BLOCK_MARKER: v = &P->c_marker; break;
    case RCC_BLOCK_INTR: v = &P->c_intr; break;
    case RCC_BLOCK_DIST: v = &P->c_dist; break;
    case RCC_BLOCK_EXT: v = &P->c_ext; break;
    default: throw Error(RCC_BAD_ARG, "unknown block kind");
  }
  RCC_REQUIRE(index >= 0 && index < (int)v->size(), RCC_BAD_ARG, "block index out of range");
  (*v)[index] = is_constant ? 1 : 0;
  P->const_dirty = true;
  P->schur_done = P->step_ready = P->cand_ready = false;
  API_END(P)
}

int rcc_ba_set_loss(rcc_ba_problem* P, int32_t loss, double scale) {
  API_BEGIN(P)
  RCC_REQUIRE(loss >= RCC_LOSS_TRIVIAL && loss <= RCC_LOSS_CAUCHY, RCC_BAD_ARG, "unknown loss");
  RCC_REQUIRE(loss == RCC_LOSS_TRIVIAL || scale > 0.0, RCC_BAD_ARG, "loss scale must be positive");
  P->loss = loss;
  P->loss_scale = scale;
  P->linearized = P->schur_done = P->step_ready = P->cand_ready = false;
  API_END(P)
}

// every check first: a refused call changes nothing
static void set_camera_lenses(P_t* P, const int32_t* lenses) {
  RCC_REQUIRE(lenses, RCC_BAD_ARG, "null pointer");
  for (int c = 0; c < P->n_cam; ++c)
    RCC_REQUIRE(lenses[c] == RCC_LENS_RADTAN || lenses[c] == RCC_LENS_EQUIDISTANT, RCC_BAD_ARG, "unknown lens");
  P->cam_lens.assign(lenses, lenses + P->n_cam);
  P->cam_equidistant = 0;
  for (int c = 0; c < P->n_cam; ++c)
    if (lenses[c] == RCC_LENS_EQUIDISTANT) P->cam_equidistant |= 1u << c;
  plan_launches(P);
  P->const_dirty = true;   // the reserved slot of an equidistant camera is held constant
  P->linearized = P->schur_done = P->step_ready = P->cand_ready = false;
}

int rcc_ba_set_lens(rcc_ba_problem* P, int32_t lens) {
  API_BEGIN(P)
  RCC_REQUIRE(lens == RCC_LENS_RADTAN || lens == RCC_LENS_EQUIDISTANT, RCC_BAD_ARG, "unknown lens");
  set_camera_lenses(P, std::vector<int32_t>((size_t)P->n_cam, lens).data());
  API_END(P)
}

int rcc_ba_set_camera_lenses(rcc_ba_problem* P, const int32_t* lenses) {
  API_BEGIN(P)
  set_camera_lenses(P, lenses);
  API_END(P)
}

// every check first: a refused call changes nothing
static void set_priors(P_t* P, int32_t kind, int64_t n, const int32_t* index, const double* mean, const double* sqrt_info) {
  int count = 0;
  switch (kind) {
    case RCC_BLOCK_VIEW: count = P->n_views; break;
    case RCC_BLOCK_MARKER: count = P->n_markers; break;
    case RCC_BLOCK_INTR: case RCC_BLOCK_DIST: count = P->n_cam; break;
    case RCC_BLOCK_EXT:
      RCC_REQUIRE(P->rig, RCC_BAD_ARG, "RCC_BLOCK_EXT needs the rig model");
      count = P->n_cam;
      break;
    default: throw Error(RCC_BAD_ARG, "unknown block kind " + std::to_string(kind));
  }
  RCC_REQUIRE(n >= 0, RCC_BAD_ARG, "n must not be negative");
  RCC_REQUIRE(n <= count, RCC_BAD_ARG, "more priors than blocks: an index out of range or repeated");
  RCC_REQUIRE(n == 0 || (index && mean && sqrt_info), RCC_BAD_ARG, "null pointer");
  const int k = prior_block_size(kind);
  std::vector<uint8_t> seen((size_t)count, 0);
  for (int64_t i = 0; i < n; ++i) {
    RCC_REQUIRE(index[i] >= 0 && index[i] < count, RCC_BAD_ARG, "prior block index out of range");
    RCC_REQUIRE(!seen[index[i]], RCC_BAD_ARG, "block " + std::to_string(index[i]) + " has two priors in one call");
    seen[index[i]] = 1;
    for (int j = 0; j < k; ++j) RCC_REQUIRE(std::isfinite(mean[i * k + j]), RCC_BAD_ARG, "non-finite prior mean");
    for (int j = 0; j < k * k; ++j)
      RCC_REQUIRE(std::isfinite(sqrt_info[i * k * k + j]), RCC_BAD_ARG, "non-finite prior sqrt_information");
  }
  std::vector<int32_t>& hi = P->prior_index_h[kind];
  std::vector<double>& hm = P->prior_mean_h[kind];
  std::vector<double>& ha = P->prior_A_h[kind];
  hi.assign(index, index + n);
  hm.assign((size_t)n * 6, 0.0);
  ha.assign((size_t)n * 36, 0.0);
  for (int64_t i = 0; i < n; ++i)
    for (int r = 0; r < k; ++r) {
      hm[i * 6 + r] = mean[i * k + r];
      for (int c = 0; c < k; ++c) ha[i * 36 + r * 6 + c] = sqrt_info[i * k * k + r * k + c];
    }
  std::vector<int32_t> idx;
  std::vector<double> mu, A;
  for (int t = 0; t < PRIOR_KINDS; ++t) {
    P->prior_off[t] = (int)idx.size();
    idx.insert(idx.end(), P->prior_index_h[t].begin(), P->prior_index_h[t].end());
    mu.insert(mu.end(), P->prior_mean_h[t].begin(), P->prior_mean_h[t].end());
    A.insert(A.end(), P->prior_A_h[t].begin(), P->prior_A_h[t].end());
  }
  const int total = (int)idx.size();
  P->prior_off[PRIOR_KINDS] = total;
  P->n_prior_parts = prior_grid(total);
  if (total > 0) {
    cudaStream_t s = P->stream;
    P->prior_index.upload(idx, s);
    P->prior_mean.upload(mu, s);
    P->prior_A.upload(A, s);
    P->prior_AtA.ensure((size_t)total * 36);
    Scoped t(P, ST_H2D, 1);
    launch_prior_gram(total, P->prior_A.p, P->prior_AtA.p, s);
  }
  // the cost partials of the priors follow the cameras' (linearisation) and K1's / K6's (evaluation, candidate cost)
  P->cost2_cam.ensure((size_t)P->n_cam + P->n_prior_parts);
  if (P->have_obs)
    P->cost_partials.ensure((size_t)std::max(std::max(1, eval_grid(P->n_obs)), P->n_chunks_e) + P->n_prior_parts);
  P->linearized = P->schur_done = P->step_ready = P->cand_ready = false;
}

int rcc_ba_set_priors(rcc_ba_problem* P, int32_t block_kind, int64_t n, const int32_t* index, const double* mean,
                      const double* sqrt_information) {
  API_BEGIN(P)
  set_priors(P, block_kind, n, index, mean, sqrt_information);
  API_END(P)
}

// every check first: a refused call changes nothing
static void set_corner_layout(P_t* P, int32_t n_slots, const double* corners, const int32_t* slot) {
  RCC_REQUIRE(n_slots >= 0, RCC_BAD_ARG, "n_slots must not be negative");
  RCC_REQUIRE(n_slots == 0 || (corners && slot), RCC_BAD_ARG, "null pointer");
  RCC_REQUIRE(P->have_obs, RCC_NOT_READY, "set_observations has not been called");
  const int64_t n = P->n_obs;
  if (n_slots > 0) {
    for (int64_t i = 0; i < (int64_t)n_slots * 8; ++i)
      RCC_REQUIRE(std::isfinite(corners[i]), RCC_BAD_ARG, "non-finite layout corner");
    for (int64_t i = 0; i < n; ++i)
      RCC_REQUIRE(slot[i] >= -1 && slot[i] < n_slots, RCC_BAD_ARG,
                  "layout slot " + std::to_string(slot[i]) + " of block " + std::to_string(i) + " out of range");
    cudaStream_t s = P->stream;
    P->corners.upload(corners, (size_t)n_slots * 8, s);
    P->slot_in.upload(slot, (size_t)n, s);
    P->e_slot.ensure((size_t)n);
    P->f_slot.ensure((size_t)n);
    Scoped t(P, ST_H2D, n > 0 ? 1 : 0);
    launch_sort_slots(P->slot_in.p, P->e_orig.p, P->f_inv.p, P->e_slot.p, P->f_slot.p, n, s);
  }
  P->n_slots = n_slots;
  P->linearized = P->schur_done = P->step_ready = P->cand_ready = false;
}

int rcc_ba_set_corner_layout(rcc_ba_problem* P, int32_t n_slots, const double* corners, const int32_t* slot) {
  API_BEGIN(P)
  set_corner_layout(P, n_slots, corners, slot);
  API_END(P)
}

int rcc_ba_get_intrinsics(rcc_ba_problem* P, double* intr, double* dist) {
  API_BEGIN(P)
  std::vector<double> h((size_t)P->n_shared);
  P->shared.download(h.data(), h.size(), P->stream);
  sync(P);
  for (int c = 0; c < P->n_cam; ++c) {
    if (intr) for (int k = 0; k < 4; ++k) intr[c * 4 + k] = h[(size_t)c * P->sp + k];
    if (dist) for (int k = 0; k < 5; ++k) dist[c * 5 + k] = h[(size_t)c * P->sp + 4 + k];
  }
  API_END(P)
}

int rcc_ba_get_rig_extrinsics(rcc_ba_problem* P, double* ext) {
  API_BEGIN(P)
  RCC_REQUIRE(ext && P->rig, RCC_BAD_ARG, "extrinsics exist only in the rig model");
  std::vector<double> h((size_t)P->n_shared);
  P->shared.download(h.data(), h.size(), P->stream);
  sync(P);
  for (int c = 0; c < P->n_cam; ++c)
    for (int k = 0; k < 6; ++k) ext[c * 6 + k] = h[(size_t)c * P->sp + 9 + k];
  API_END(P)
}

int rcc_ba_get_view_poses(rcc_ba_problem* P, double* views) {
  API_BEGIN(P)
  RCC_REQUIRE(views, RCC_BAD_ARG, "null pointer");
  P->views.download(views, (size_t)P->n_views * 6, P->stream);
  sync(P);
  API_END(P)
}

int rcc_ba_get_marker_poses(rcc_ba_problem* P, double* markers) {
  API_BEGIN(P)
  RCC_REQUIRE(markers, RCC_BAD_ARG, "null pointer");
  P->markers.download(markers, (size_t)P->n_markers * 6, P->stream);
  sync(P);
  API_END(P)
}

static int evaluate_impl(P_t* P, int want_j, double* cost, bool to_host, double* residuals, double* ji, double* jd,
                         double* jv, double* jm, double* jx) {
  RCC_REQUIRE(P->have_obs, RCC_NOT_READY, "set_observations has not been called");
  ensure_expanded(P);
  ensure_pixels(P);
  const size_t n = (size_t)P->n_obs;
  EvalArgs a = eval_args(P, false);
  const bool all = !to_host;  // device mode materialises everything
  if (all || residuals) { P->o_res.ensure(n * 8); a.residuals = P->o_res.p; }
  if (want_j) {
    if (all || ji) { P->o_ji.ensure(n * 32); a.jac_intr = P->o_ji.p; }
    if (all || jd) { P->o_jd.ensure(n * 40); a.jac_dist = P->o_jd.p; }
    if (all || jv) { P->o_jv.ensure(n * 48); a.jac_view = P->o_jv.p; }
    if (all || jm) { P->o_jm.ensure(n * 48); a.jac_marker = P->o_jm.p; }
    if (P->rig && (all || jx)) { P->o_jx.ensure(n * 48); a.jac_ext = P->o_jx.p; }
  }
  a.fail_flag = P->fail_flag.p + 2;   // slot 2: materialised evaluation
  RCC_CUDA(cudaMemsetAsync(a.fail_flag, 0, sizeof(int32_t), P->stream));
  {
    Scoped t(P, ST_EVALUATE, P->n_prior_parts > 0 ? 2 : 1);
    if (want_j) {
      // K1 once per run; outputs go to caller positions and the cost partials stay one per chunk, so the launches
      // are independent
      for (const Run& r : P->runs_k1) {
        EvalArgs b = a;
        b.chunks = (r.listed ? P->k1_chunks.p : P->e_chunks.p) + r.first;
        b.n_chunks = r.count;
        b.cost2_partials = a.cost2_partials + r.first;
        launch_evaluate(P->rig, true, r.lens, b, P->stream);
        P->launch_count += 1;
      }
    } else {
      launch_evaluate(P->rig, false, handle_lens(P), a, P->stream);
      P->launch_count += 1;
    }
    const int np = eval_partials(want_j != 0, a);
    if (P->n_prior_parts > 0) launch_prior(false, prior_args(P, false, P->cost_partials.p + np), P->stream);
    launch_sum(P->cost_partials.p, np + P->n_prior_parts, P->scalar.p, 0.5, P->stream);
  }
  int fail = 0;
  if (to_host) {
    if (residuals) P->o_res.download(residuals, n * 8, P->stream);
    if (want_j) {
      if (ji) P->o_ji.download(ji, n * 32, P->stream);
      if (jd) P->o_jd.download(jd, n * 40, P->stream);
      if (jv) P->o_jv.download(jv, n * 48, P->stream);
      if (jm) P->o_jm.download(jm, n * 48, P->stream);
      if (jx && P->rig) P->o_jx.download(jx, n * 48, P->stream);
    }
  }
  if (cost || to_host) {
    RCC_CUDA(cudaMemcpyAsync(P->h_pinned, P->scalar.p, sizeof(double), cudaMemcpyDeviceToHost, P->stream));
    RCC_CUDA(cudaMemcpyAsync(P->h_pinned + 1, P->fail_flag.p + 2, sizeof(int32_t), cudaMemcpyDeviceToHost, P->stream));
    sync(P);
    if (cost) *cost = P->h_pinned[0];
    fail = *reinterpret_cast<int32_t*>(P->h_pinned + 1);
  }
  return fail ? RCC_EVAL_FAILED : RCC_OK;
}

int rcc_ba_evaluate(rcc_ba_problem* P, int32_t want_j, double* cost, double* residuals, double* ji, double* jd,
                    double* jv, double* jm, double* jx) {
  int rc = RCC_OK;
  API_BEGIN(P)
  rc = evaluate_impl(P, want_j, cost, true, residuals, ji, jd, jv, jm, jx);
  if (rc == RCC_EVAL_FAILED) P->err = "evaluation failed: corner behind the camera or non-finite residual";
  if (rc != RCC_OK) return rc;
  API_END(P)
}

int rcc_ba_evaluate_device(rcc_ba_problem* P, int32_t want_j, double* cost) {
  int rc = RCC_OK;
  API_BEGIN(P)
  rc = evaluate_impl(P, want_j, cost, false, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
  if (rc != RCC_OK) return rc;
  API_END(P)
}

int rcc_ba_linearize(rcc_ba_problem* P, double* cost) {
  API_BEGIN(P)
  do_linearize(P);
  if (cost) {
    std::vector<double> c2((size_t)P->n_cam + P->n_prior_parts);   // the cameras', then the priors' cost
    int32_t fail = 0;
    P->cost2_cam.download(c2.data(), c2.size(), P->stream);
    RCC_CUDA(cudaMemcpyAsync(&fail, P->fail_flag.p, sizeof(int32_t), cudaMemcpyDeviceToHost, P->stream));
    sync(P);
    *cost = 0.5 * std::accumulate(c2.begin(), c2.end(), 0.0);
    if (fail) throw Error(RCC_EVAL_FAILED, "evaluation failed: corner behind the camera or non-finite residual");
  }
  API_END(P)
}

int rcc_ba_schur(rcc_ba_problem* P, double radius) {
  API_BEGIN(P)
  do_schur(P, radius);
  API_END(P)
}

int rcc_ba_set_lm_diagonal(rcc_ba_problem* P, double min_diagonal, double max_diagonal, int32_t jacobi_scaling) {
  API_BEGIN(P)
  RCC_REQUIRE(min_diagonal >= 0 && max_diagonal >= min_diagonal, RCC_BAD_ARG, "bad LM diagonal bounds");
  P->min_diag = min_diagonal;
  P->max_diag = max_diagonal;
  P->jacobi = jacobi_scaling ? 1 : 0;
  P->schur_done = P->step_ready = P->cand_ready = false;
  API_END(P)
}

int rcc_ba_solve_step(rcc_ba_problem* P, double* mcc, double* step_norm, double* x_norm) {
  API_BEGIN(P)
  do_step(P);
  if (P->comm) {
    RCC_NCCL(ncclAllReduce(P->stats.p + SX_MCC_E, P->stats.p + SX_MCC_E, 3, ncclDouble, ncclSum, P->comm, P->stream));
    RCC_NCCL(ncclAllReduce(P->stats.p + SX_GMAX_E, P->stats.p + SX_GMAX_E, 1, ncclDouble, ncclMax, P->comm, P->stream));
  }
  StepScalars s = read_step_scalars(P);
  if (mcc) *mcc = s.mcc;
  if (step_norm) *step_norm = s.step_norm;
  if (x_norm) *x_norm = s.x_norm;
  if (s.potrf_info != 0) throw Error(RCC_NOT_SPD, "reduced system is not positive definite (potrf info " +
                                                      std::to_string(s.potrf_info) + ")");
  API_END(P)
}

int rcc_ba_candidate_cost(rcc_ba_problem* P, double* cost) {
  API_BEGIN(P)
  RCC_REQUIRE(P->step_ready, RCC_NOT_READY, "solve_step has not been called");
  // the E-side sums were already all-reduced by solve_step; zero them so the
  // fused all-reduce inside do_candidate_cost cannot double count
  if (P->comm) {
    RCC_CUDA(cudaMemsetAsync(P->stats.p + SX_MCC_E, 0, 3 * sizeof(double), P->stream));
  }
  do_candidate_cost(P);
  StepScalars s = read_step_scalars(P);
  if (cost) *cost = s.cand_cost;
  if (s.fail) throw Error(RCC_EVAL_FAILED, "candidate point: corner behind the camera or non-finite residual");
  API_END(P)
}

int rcc_ba_accept_step(rcc_ba_problem* P) {
  API_BEGIN(P)
  do_accept(P);
  API_END(P)
}

int rcc_ba_solve(rcc_ba_problem* P, const rcc_lm_options* opt, rcc_lm_summary* summary) {
  API_BEGIN(P)
  rcc_lm_options o;
  if (opt) o = *opt;
  else rcc_lm_default_options(&o);
  rcc_lm_summary s;
  do_solve(P, o, s);
  if (summary) *summary = s;
  API_END(P)
}

int rcc_ba_covariance(rcc_ba_problem* P, double* cov_shared, double* cov_views, double* cov_markers) {
  API_BEGIN(P)
  do_covariance(P, cov_shared, cov_views, cov_markers);
  API_END(P)
}

int rcc_ba_covariance_blocks(rcc_ba_problem* P, int64_t n_pairs, const int32_t* pairs, double* out) {
  API_BEGIN(P)
  do_covariance_blocks(P, n_pairs, pairs, out);
  API_END(P)
}

int rcc_ba_get_dims(rcc_ba_problem* P, rcc_ba_dims* d) {
  API_BEGIN(P)
  RCC_REQUIRE(d, RCC_BAD_ARG, "null pointer");
  d->eliminated_is_view = P->elim_view ? 1 : 0;
  d->n_e = P->n_e;
  d->n_f = P->n_f;
  d->n_shared = P->n_shared;
  d->n_reduced = P->n_red;
  d->ld_reduced = P->ld;
  d->n_pairs = P->n_pairs;
  API_END(P)
}

int rcc_ba_get_normal_blocks(rcc_ba_problem* P, double* Hee, double* ge, double* Hes, double* Hff, double* gf,
                             double* Hfs, double* Hss, double* gs, double* W) {
  API_BEGIN(P)
  RCC_REQUIRE(P->linearized, RCC_NOT_READY, "linearize has not been called");
  cudaStream_t s = P->stream;
  if (Hee) P->Hee.download(Hee, (size_t)P->n_e * 36, s);
  if (ge) P->ge.download(ge, (size_t)P->n_e * 6, s);
  if (Hes) P->Hes.download(Hes, (size_t)P->n_e * 6 * P->n_shared, s);
  if (Hff) P->Hff.download(Hff, (size_t)P->n_f * 36, s);
  if (gf) P->gf.download(gf, (size_t)P->n_f * 6, s);
  if (Hfs) P->Hfs.download(Hfs, (size_t)P->n_f * 6 * P->n_shared, s);
  if (Hss) P->Hss.download(Hss, (size_t)P->n_shared * P->n_shared, s);
  if (gs) P->gs.download(gs, (size_t)P->n_shared, s);
  if (W) {
    std::vector<double> w((size_t)P->n_obs * 36);
    std::vector<int32_t> orig((size_t)P->n_obs);
    P->W.download(w.data(), w.size(), s);
    P->e_orig.download(orig.data(), orig.size(), s);
    sync(P);
    for (int64_t i = 0; i < P->n_obs; ++i) memcpy(W + (size_t)orig[i] * 36, &w[(size_t)i * 36], 36 * sizeof(double));
  }
  sync(P);
  API_END(P)
}

int rcc_ba_get_reduced_system(rcc_ba_problem* P, double* S, double* b) {
  API_BEGIN(P)
  RCC_REQUIRE(P->schur_done, RCC_NOT_READY, "reduced system not available (call schur; solve_step overwrites it)");
  const int n = P->n_red;
  std::vector<double> h((size_t)n * P->ld);
  P->S.download(h.data(), h.size(), P->stream);
  sync(P);
  for (int i = 0; i < n; ++i) {
    if (S)
      for (int j = i; j < n; ++j) {
        S[(size_t)i * n + j] = h[(size_t)i * P->ld + j];
        S[(size_t)j * n + i] = h[(size_t)i * P->ld + j];
      }
    if (b) b[i] = h[(size_t)i * P->ld + n];
  }
  API_END(P)
}

int rcc_ba_get_reduced_block(rcc_ba_problem* P, int32_t row0, int32_t n_rows, int32_t col0, int32_t n_cols, double* out) {
  API_BEGIN(P)
  RCC_REQUIRE(P->schur_done, RCC_NOT_READY, "reduced system not available (call schur; solve_step overwrites it)");
  const int n = P->n_red;
  RCC_REQUIRE(out && row0 >= 0 && n_rows > 0 && row0 + n_rows <= n && col0 >= 0 && n_cols > 0 && col0 + n_cols <= n + 1,
              RCC_BAD_ARG, "window outside the reduced system");
  // the buffer holds the upper triangle (+ rhs in column n): fetch the window and its mirror image
  std::vector<double> a((size_t)n_rows * n_cols), b;
  RCC_CUDA(cudaMemcpy2DAsync(a.data(), (size_t)n_cols * sizeof(double), P->S.p + (size_t)row0 * P->ld + col0,
                             (size_t)P->ld * sizeof(double), (size_t)n_cols * sizeof(double), n_rows,
                             cudaMemcpyDeviceToHost, P->stream));
  const int mc = std::min(n_cols, n - col0);   // mirrored part: columns < n only
  if (mc > 0) {
    b.resize((size_t)mc * n_rows);
    RCC_CUDA(cudaMemcpy2DAsync(b.data(), (size_t)n_rows * sizeof(double), P->S.p + (size_t)col0 * P->ld + row0,
                               (size_t)P->ld * sizeof(double), (size_t)n_rows * sizeof(double), mc,
                               cudaMemcpyDeviceToHost, P->stream));
  }
  sync(P);
  for (int i = 0; i < n_rows; ++i)
    for (int j = 0; j < n_cols; ++j) {
      const int r = row0 + i, c = col0 + j;
      out[(size_t)i * n_cols + j] = (c >= r) ? a[(size_t)i * n_cols + j] : b[(size_t)j * n_rows + i];
    }
  API_END(P)
}

int rcc_ba_get_step(rcc_ba_problem* P, double* d_e, double* d_f, double* d_shared) {
  API_BEGIN(P)
  RCC_REQUIRE(P->step_ready, RCC_NOT_READY, "solve_step has not been called");
  if (d_e) P->delta_e.download(d_e, (size_t)P->n_e * 6, P->stream);
  if (d_f) P->rhs.download(d_f, (size_t)P->n_f * 6, P->stream);
  if (d_shared)
    RCC_CUDA(cudaMemcpyAsync(d_shared, P->rhs.p + (size_t)6 * P->n_f, (size_t)P->n_shared * sizeof(double),
                             cudaMemcpyDeviceToHost, P->stream));
  sync(P);
  API_END(P)
}

int rcc_comm_get_unique_id(char id[RCC_COMM_ID_BYTES]) {
  if (!id) return RCC_BAD_ARG;
  static_assert(sizeof(ncclUniqueId) <= RCC_COMM_ID_BYTES, "unique id does not fit");
  ncclUniqueId u;
  if (ncclGetUniqueId(&u) != ncclSuccess) return RCC_NCCL_ERROR;
  memset(id, 0, RCC_COMM_ID_BYTES);
  memcpy(id, &u, sizeof(u));
  return RCC_OK;
}

int rcc_ba_comm_init(rcc_ba_problem* P, const char id[RCC_COMM_ID_BYTES], int32_t rank, int32_t n_ranks) {
  API_BEGIN(P)
  RCC_REQUIRE(id && n_ranks >= 1 && rank >= 0 && rank < n_ranks, RCC_BAD_ARG, "bad communicator arguments");
  if (P->comm) {
    ncclCommDestroy(P->comm);
    P->comm = nullptr;
  }
  P->rank = rank;
  P->n_ranks = n_ranks;
  P->chol_mode = -1;   // re-resolve: the distributed factorisation needs the communicator
  if (n_ranks > 1) {
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    RCC_NCCL(ncclCommInitRank(&P->comm, n_ranks, u, rank));
    if (!P->comm_stream) RCC_CUDA(cudaStreamCreateWithFlags(&P->comm_stream, cudaStreamNonBlocking));
    for (auto& e : P->ev_grp)
      if (!e) RCC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  API_END(P)
}

int rcc_ba_profile_enable(rcc_ba_problem* P, int32_t on) {
  API_BEGIN(P)
  sync(P);
  P->timer.collect();
  P->timer.on = on != 0;
  API_END(P)
}

int rcc_ba_profile_reset(rcc_ba_problem* P) {
  API_BEGIN(P)
  sync(P);
  P->timer.reset();
  API_END(P)
}

int rcc_ba_profile_get(rcc_ba_problem* P, const char* stage, double* total_ms, int64_t* launches) {
  API_BEGIN(P)
  RCC_REQUIRE(stage, RCC_BAD_ARG, "null stage name");
  sync(P);
  P->timer.collect();
  int found = -1;
  for (int i = 0; i < ST_COUNT; ++i)
    if (strcmp(stage, stage_name(i)) == 0) found = i;
  RCC_REQUIRE(found >= 0, RCC_BAD_ARG, std::string("unknown stage ") + stage);
  if (total_ms) *total_ms = P->timer.ms[found];
  if (launches) *launches = P->timer.launches[found];
  API_END(P)
}

int64_t rcc_ba_launch_count(const rcc_ba_problem* P) { return P ? P->launch_count : 0; }

int rcc_ba_flush_l2(rcc_ba_problem* P) {
  API_BEGIN(P)
  const size_t n = (size_t)256 * 1024 * 1024 / sizeof(double);  // 256 MiB > 126 MB L2
  P->flush_buf.ensure(n);
  launch_fill(P->flush_buf.p, (int64_t)n, 0.0, P->stream);
  API_END(P)
}

int rcc_ba_synchronize(rcc_ba_problem* P) {
  API_BEGIN(P)
  sync(P);
  API_END(P)
}

int rcc_dense_potrf(int32_t device, double* dA, int32_t n, int32_t ld, int32_t extra_rows, int32_t use_cusolver,
                    int32_t* info, double* ms) {
  if (!dA || n <= 0 || ld < n + extra_rows || extra_rows < 0) return RCC_BAD_ARG;
  CholDriver d;
  cusolverDnHandle_t h = nullptr;
  double* work = nullptr;
  int* dinfo = nullptr;
  cudaStream_t s = nullptr;
  cudaEvent_t a = nullptr, b = nullptr;
  int rc = RCC_OK;
  try {
    RCC_CUDA(cudaSetDevice(device));
    RCC_CUDA(cudaDeviceSynchronize());      // the caller filled dA on a stream of its own
    RCC_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    RCC_CUDA(cudaEventCreate(&a));
    RCC_CUDA(cudaEventCreate(&b));
    int lwork = 0;
    if (use_cusolver) {
      RCC_REQUIRE(extra_rows == 0, RCC_BAD_ARG, "the cuSOLVER comparator factors a square matrix");
      RCC_SOLVER(cusolverDnCreate(&h));
      RCC_SOLVER(cusolverDnSetStream(h, s));
      RCC_SOLVER(cusolverDnDpotrf_bufferSize(h, CUBLAS_FILL_MODE_LOWER, n, dA, ld, &lwork));
      RCC_CUDA(cudaMalloc(&work, (size_t)std::max(1, lwork) * sizeof(double)));
      RCC_CUDA(cudaMalloc(&dinfo, sizeof(int)));
    } else {
      d.init();
    }
    RCC_CUDA(cudaEventRecord(a, s));
    if (use_cusolver) RCC_SOLVER(cusolverDnDpotrf(h, CUBLAS_FILL_MODE_LOWER, n, dA, ld, work, lwork, dinfo));
    else chol_factor(dA, n, ld, n + extra_rows, 0, 1, nullptr, s, d);
    RCC_CUDA(cudaEventRecord(b, s));
    RCC_CUDA(cudaStreamSynchronize(s));
    float t = 0.f;
    RCC_CUDA(cudaEventElapsedTime(&t, a, b));
    if (ms) *ms = t;
    int hinfo = 0;
    RCC_CUDA(cudaMemcpy(&hinfo, use_cusolver ? dinfo : d.info, sizeof(int), cudaMemcpyDeviceToHost));
    if (info) *info = hinfo;
  } catch (const Error& e) {
    g_create_error = e.what();
    fprintf(stderr, "[rcc_dense_potrf] %s\n", e.what());
    rc = e.status;
  }
  d.destroy();
  if (h) cusolverDnDestroy(h);
  if (work) cudaFree(work);
  if (dinfo) cudaFree(dinfo);
  if (a) cudaEventDestroy(a);
  if (b) cudaEventDestroy(b);
  if (s) cudaStreamDestroy(s);
  return rc;
}

int rcc_dense_trsv(int32_t device, const double* dA, int32_t n, int32_t ld, double* dx, int32_t use_cublas, double* ms) {
  if (!dA || !dx || n <= 0 || ld < n) return RCC_BAD_ARG;
  cudaStream_t s = nullptr;
  cudaEvent_t a = nullptr, b = nullptr;
  cublasHandle_t h = nullptr;
  DBuf<double> inv;
  DBuf<int> flags;
  int rc = RCC_OK;
  try {
    RCC_CUDA(cudaSetDevice(device));
    RCC_CUDA(cudaDeviceSynchronize());
    RCC_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    RCC_CUDA(cudaEventCreate(&a));
    RCC_CUDA(cudaEventCreate(&b));
    if (use_cublas) {
      RCC_BLAS(cublasCreate(&h));
      RCC_BLAS(cublasSetStream(h, s));
    } else {
      inv.alloc(chol_trsv_workspace_doubles(n));
      flags.alloc((size_t)chol_trsv_flags(n));
    }
    RCC_CUDA(cudaEventRecord(a, s));
    if (use_cublas) RCC_BLAS(cublasDtrsv(h, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_T, CUBLAS_DIAG_NON_UNIT, n, dA, ld, dx, 1));
    else chol_trsv(dA, ld, n, dx, inv.p, flags.p, s);
    RCC_CUDA(cudaEventRecord(b, s));
    RCC_CUDA(cudaStreamSynchronize(s));
    float t = 0.f;
    RCC_CUDA(cudaEventElapsedTime(&t, a, b));
    if (ms) *ms = t;
    if (!use_cublas) {
      int e = 0;
      RCC_CUDA(cudaMemcpy(&e, flags.p + chol_trsv_flags(n) - 1, sizeof(int), cudaMemcpyDeviceToHost));
      if (e) throw Error(RCC_SOLVER_ERROR, "back-substitution: a wait for another block's part of x gave up");
    }
  } catch (const Error& e) {
    g_create_error = e.what();
    fprintf(stderr, "[rcc_dense_trsv] %s\n", e.what());
    rc = e.status;
  }
  if (h) cublasDestroy(h);
  if (a) cudaEventDestroy(a);
  if (b) cudaEventDestroy(b);
  if (s) cudaStreamDestroy(s);
  return rc;
}

int rcc_fp64_peak_tflops(int32_t device, double* tflops) {
  if (!tflops) return RCC_BAD_ARG;
  try {
    RCC_CUDA(cudaSetDevice(device));
    cudaStream_t s;
    RCC_CUDA(cudaStreamCreate(&s));
    cudaEvent_t a, b;
    RCC_CUDA(cudaEventCreate(&a));
    RCC_CUDA(cudaEventCreate(&b));
    double* sink = nullptr;   // per call and per device (a process-wide pointer would belong to one device only)
    RCC_CUDA(cudaMalloc(&sink, 8));
    launch_fp64_peak(200, sink, s);
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
      RCC_CUDA(cudaEventRecord(a, s));
      const double fmas = launch_fp64_peak(4000, sink, s);
      RCC_CUDA(cudaEventRecord(b, s));
      RCC_CUDA(cudaStreamSynchronize(s));
      float ms = 0.f;
      RCC_CUDA(cudaEventElapsedTime(&ms, a, b));
      best = std::max(best, 2.0 * fmas / (ms * 1e-3) * 1e-12);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaStreamDestroy(s);
    cudaFree(sink);
    *tflops = best;
  } catch (const Error& e) {
    g_create_error = e.what();
    return e.status;
  }
  return RCC_OK;
}

}  // extern "C"
