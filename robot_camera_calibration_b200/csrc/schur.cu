// K3 -- Schur complement of the Gauss-Newton normal equations: the eliminated
// 6-dof blocks (E) are folded into the reduced system over the kept blocks (F)
// and the shared intrinsics / distortion / rig-extrinsics border.
//
// Replaces (SURVEY.md 8a row a8) the Schur eliminator that would run inside
// Ceres for the reference's missing optimiser stage.
//
// With H_ee + D_e = L L^T per eliminated block,  Y_ef = L^-1 W_ef,
// Yb_e = L^-1 [H_es | g_e]:
//     S   = H_FF - sum_e Y_e^T Y_e          (block-sparse SYRK, upper triangle)
//     b   = g_F  - sum_e Y_e^T (L^-1 g_e)   (carried as one more column of S)
//     d_e = -L^-T ( L^-1 g_e + Y_e d_F )    (back-substitution)
// Every 6-row block of S is owned by exactly one CTA per column tile and summed
// in a fixed order: no FP64 atomics, bitwise reproducible.
#include "common.cuh"
#include "kernels.h"

namespace rcc {

// ---------------------------------------------------------------------------
// schur_prep: one warp per eliminated block
// ---------------------------------------------------------------------------
constexpr int PREP_REC = 38;   // staged 6x6 record stride (doubles): 36 + 2 keeps the 16-byte row reads of 8 lanes on distinct banks
__global__ void __launch_bounds__(128, 3) schur_prep_kernel(const SchurPrepArgs a) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= a.n_e) return;
  // every lane factors the 6x6 block redundantly (registers only)
  double L[6][6], Li[6][6], d2[6];
  const double* H = a.Hee + (size_t)e * 36;
  const bool is_const = a.e_const[e] != 0;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const double dg = H[i * 6 + i];
    d2[i] = lm_diagonal(dg, a.radius, a.min_diag, a.max_diag, a.jacobi);
  }
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      L[i][j] = 0.0;
      Li[i][j] = 0.0;
    }
  // Cholesky (lower)
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double s = H[j * 6 + j] + d2[j];
#pragma unroll
    for (int k = 0; k < j; ++k) s -= L[j][k] * L[j][k];
    if (a.pivot_fail && !is_const && !(s > 1e-300) && lane == 0) *a.pivot_fail = 1;
    s = fmax(s, 1e-300);
    const double ljj = sqrt(s);
    L[j][j] = ljj;
    const double inv = 1.0 / ljj;
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
      double v = H[i * 6 + j];
#pragma unroll
      for (int k = 0; k < j; ++k) v -= L[i][k] * L[j][k];
      L[i][j] = v * inv;
    }
  }
  // inverse of the lower-triangular factor (forward substitution per column)
#pragma unroll
  for (int c = 0; c < 6; ++c) {
#pragma unroll
    for (int i = c; i < 6; ++i) {
      double v = (i == c) ? 1.0 : 0.0;
#pragma unroll
      for (int k = c; k < i; ++k) v -= L[i][k] * Li[k][c];
      Li[i][c] = v / L[i][i];
    }
  }
  if (is_const) {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      d2[i] = 0.0;
#pragma unroll
      for (int j = 0; j < 6; ++j) Li[i][j] = 0.0;
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      a.d2e[(size_t)e * 6 + i] = d2[i];
#pragma unroll
      for (int j = 0; j < 6; ++j) a.Linv[(size_t)e * 36 + i * 6 + j] = Li[i][j];
    }
  }
  // Y = L^-1 * (sum of the member W blocks) for every pair of row e, 32 pairs per round.  The 288-byte
  // W and Y records of a round are contiguous in HBM when every pair has one member at consecutive sorted
  // positions (always in the single-camera model): they then cross the SM through shared memory so that
  // the global accesses are coalesced 16-byte pieces instead of 32 strided records per instruction.
  __shared__ __align__(16) double rec_all[4][32 * PREP_REC];
  double* rec = rec_all[threadIdx.x >> 5];
  const int p_begin = a.row_ptr[e], p_end = a.row_ptr[e + 1];
  const int row_pos0 = a.row_pos0[e];
  const bool fast = row_pos0 >= 0;   // warp-uniform; no per-pair index loads on this path
  for (int p0 = p_begin; p0 < p_end; p0 += 32) {
    const int np = min(32, p_end - p0);
    const int p = p0 + lane;
    const bool on = lane < np;
    int m0 = 0, m1 = 0;
    if (on && !fast) {
      m0 = a.pair_mptr[p];
      m1 = a.pair_mptr[p + 1];
    }
    const int pos0 = row_pos0 + (p0 - p_begin);
    double Wm[36];
    if (fast) {
      const double2* src = reinterpret_cast<const double2*>(a.W + (size_t)pos0 * 36);
      for (int k = lane; k < np * 18; k += 32) {
        const int q = k / 18;
        reinterpret_cast<double2*>(rec + q * PREP_REC)[k - q * 18] = src[k];
      }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 18; ++i) {
        const double2 v = reinterpret_cast<const double2*>(rec + lane * PREP_REC)[i];
        Wm[2 * i] = v.x;
        Wm[2 * i + 1] = v.y;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 36; ++i) Wm[i] = 0.0;
      for (int m = m0; m < m1; ++m) {
        const double2* w = reinterpret_cast<const double2*>(a.W + (size_t)a.pair_members[m] * 36);
#pragma unroll
        for (int i = 0; i < 18; ++i) {
          const double2 v = w[i];
          Wm[2 * i] += v.x;
          Wm[2 * i + 1] += v.y;
        }
      }
    }
    // y = L^-1 Wm, column-major; staged through the same record when the round is contiguous
    double* y = fast ? rec + lane * PREP_REC : a.Y + (size_t)p * 36;
    if (on) {
#pragma unroll
      for (int c = 0; c < 6; ++c)
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          double v = 0.0;
#pragma unroll
          for (int j = 0; j <= k; ++j) v += Li[k][j] * Wm[j * 6 + c];
          y[c * 6 + k] = v;  // column-major
        }
    }
    if (fast) {
      __syncwarp();
      double2* dst = reinterpret_cast<double2*>(a.Y + (size_t)p0 * 36);
      for (int k = lane; k < np * 18; k += 32) {
        const int q = k / 18;
        dst[k] = reinterpret_cast<const double2*>(rec + q * PREP_REC)[k - q * 18];
      }
      __syncwarp();
    }
  }
  // border: columns 0..n_shared-1 = H_es, column n_shared = g_e, rest zero
  const int ncol = a.n_bb * 6;
  for (int s = lane; s < ncol; s += 32) {
    double v[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      if (s < a.n_shared) v[j] = a.Hes[((size_t)e * 6 + j) * a.n_shared + s];
      else if (s == a.n_shared) v[j] = a.ge[(size_t)e * 6 + j];
      else v[j] = 0.0;
    }
    double* y = a.Yb + ((size_t)e * a.n_bb + s / 6) * 36 + (s % 6) * 6;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j <= k; ++j) acc += Li[k][j] * v[j];
      y[k] = acc;
    }
  }
}

void launch_schur_prep(const SchurPrepArgs& a, cudaStream_t s) {
  if (a.n_e == 0) return;
  schur_prep_kernel<<<ceil_div((int64_t)a.n_e * 32, 128), 128, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
// schur_syrk: CTA (f, J) owns the 6 x (6 * SY_WARPS * SY_SUB) strip of S in
// block row f and column tile J; warp w of the CTA owns the SY_SUB kept blocks of
// sub-tile J * SY_WARPS + w and keeps their 6 x 6 output blocks in its private
// slice of shared memory.  The CTA walks the pairs (e, f) of column f in
// batches (Y_ef staged by cp.async, double buffered, one barrier per batch);
// for each pair every warp holds Y_ef in 36 registers and its lanes take the
// (partner block f', column c) items of row e that fall in the warp's sub-tile:
// 48 B coalesced load of Y_ef'[:, c], 36 DFMA, 6-double read-modify-write on the
// warp's slice.  No barrier per pair, no cross-warp traffic, fixed summation
// order (ascending e) -> bitwise reproducible.
// ---------------------------------------------------------------------------
constexpr int SY_WARPS = SYRK_CTA_SUBTILES;   // one warp per sub-tile
constexpr int SY_SUB = SYRK_SUBTILE;          // kept blocks per warp sub-tile = tile_ptr granularity
constexpr int SY_IPB = 6;                     // items (columns) per partner block
constexpr int SY_BATCH = 32;                  // pairs of column f staged per round (<= 32: one lane per pair holds its range)
static_assert(SY_BATCH <= 32, "a batch must fit the lanes of a warp");

__device__ __forceinline__ void sy_cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}

// position of a warp in the (pair, step) sequence of a staged batch -- warp-uniform
struct SyCursor { int q, lo, n_items, base; };
// moves to the next 32-item step; lane q of the warp holds the partner range [lo_q, hi_q) of pair q
__device__ __forceinline__ bool sy_advance(SyCursor& c, int nb, int lo_lane, int hi_lane) {
  c.base += 32;
  while (c.base >= c.n_items) {
    if (++c.q >= nb) return false;
    c.lo = __shfl_sync(0xffffffffu, lo_lane, c.q);
    c.n_items = (__shfl_sync(0xffffffffu, hi_lane, c.q) - c.lo) * SY_IPB;
    c.base = 0;
  }
  return true;
}
// one lane's item of a step: column c of partner block Y_ef' and its slot in the warp's output slice
struct SyItem { double2 y[3]; int pf, col; };   // pf < 0: idle lane.  (raw loads only: nothing here waits on memory)
__device__ __forceinline__ void sy_load(const SchurSyrkArgs& a, const SyCursor& c, int lane, int subbase, SyItem& it) {
  const int idx = c.base + lane;
  it.pf = -1;
  it.col = 0;
  if (idx < c.n_items) {
    const int jj = idx / SY_IPB, col = idx - jj * SY_IPB;
    const int j = c.lo + jj;
    const double2* yp = reinterpret_cast<const double2*>(a.Y + (size_t)j * 36 + col * 6);
#pragma unroll
    for (int i = 0; i < 3; ++i) it.y[i] = yp[i];
    it.pf = a.pair_f[j];
    it.col = col;
  }
}

// SchurSyrkArgs stays in the parameter bank (__grid_constant__) and its fields are read where they are used.
// Without it the compiler loads a by-value struct of up to 128 bytes into registers at entry, which costs
// schur_border_kernel 24 registers.
__global__ void __launch_bounds__(SY_WARPS * 32, 6) schur_syrk_kernel(const __grid_constant__ SchurSyrkArgs a) {
  extern __shared__ __align__(16) double sm[];
  // work list: (block row f, column tile J >= tile of f), largest estimated work first
  const int f = a.cta_list[2 * blockIdx.x];
  const int J = a.cta_list[2 * blockIdx.x + 1];
  const int sub_of_f = f / SY_SUB;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double* acc = sm + warp * (SY_SUB * 36);            // [SY_SUB blocks][6 columns][6 rows]
  double* yi = sm + SY_WARPS * SY_SUB * 36;           // [2][SY_BATCH][36] staged Y_ef
  for (int k = lane; k < SY_SUB * 36; k += 32) acc[k] = 0.0;

  const int js = J * SY_WARPS + warp;                 // this warp's sub-tile
  const bool active = (js >= sub_of_f) && (js < a.n_tiles);
  const int subbase = js * SY_SUB;
  const int c0 = a.col_ptr[f], c1 = a.col_ptr[f + 1];
  const int tps = a.n_tiles + 1;

  auto stage = [&](int cb, int buf) {
    const int nb = min(SY_BATCH, c1 - cb);
    double2* dst = reinterpret_cast<double2*>(yi + buf * SY_BATCH * 36);
    for (int k = tid; k < nb * 18; k += SY_WARPS * 32) {
      const int q = k / 18, piece = k - q * 18;
      const int p = a.col_pair[cb + q];
      sy_cp_async16(dst + k, reinterpret_cast<const double2*>(a.Y + (size_t)p * 36) + piece);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  // lane q of every warp: partner range of pair q of the batch inside the warp's sub-tile
  auto meta = [&](int cb, int& lo, int& hi) {
    lo = 0;
    hi = 0;
    if (active && cb + lane < c1) {
      const int p = a.col_pair[cb + lane];
      const int* tp = a.tile_ptr + (size_t)a.pair_e[p] * tps;
      lo = (js == sub_of_f) ? p : tp[js];
      hi = tp[min(js + 1, a.n_tiles)];
    }
  };

  int lo_cur, hi_cur, lo_nxt = 0, hi_nxt = 0;
  if (c0 < c1) stage(c0, 0);
  meta(c0, lo_cur, hi_cur);
  int buf = 0;
  for (int cb = c0; cb < c1; cb += SY_BATCH, buf ^= 1) {
    const int nb = min(SY_BATCH, c1 - cb);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();   // batch `cb` staged by everyone; batch `cb - SY_BATCH` consumed by everyone
    if (cb + SY_BATCH < c1) {
      stage(cb + SY_BATCH, buf ^ 1);
      meta(cb + SY_BATCH, lo_nxt, hi_nxt);
    }
    if (active) {
      const double* ybuf = yi + buf * SY_BATCH * 36;
      // The warp walks the (pair, 32-item step) sequence of the batch; the global loads of step s+1
      // (partner column, partner index) are issued before the arithmetic of step s.
      SyCursor cur{-1, 0, 0, 0}, nxt;
      SyItem it_c, it_n;
      bool have = sy_advance(cur, nb, lo_cur, hi_cur);
      if (have) sy_load(a, cur, lane, subbase, it_c);
      int q_loaded = -1;
      double Yi[36];   // Y_ef, column-major: Yi[r * 6 + k] = Y_ef[k][r]
      while (have) {
        nxt = cur;
        const bool have_n = sy_advance(nxt, nb, lo_cur, hi_cur);
        if (have_n) sy_load(a, nxt, lane, subbase, it_n);
        if (cur.q != q_loaded) {
          const double2* src = reinterpret_cast<const double2*>(ybuf + cur.q * 36);
#pragma unroll
          for (int i = 0; i < 18; ++i) {
            const double2 v = src[i];
            Yi[2 * i] = v.x;
            Yi[2 * i + 1] = v.y;
          }
          q_loaded = cur.q;
        }
        if (it_c.pf >= 0) {
          double2* ap = reinterpret_cast<double2*>(acc + (it_c.pf - subbase) * 36 + it_c.col * 6);
          const double2 y0 = it_c.y[0], y1 = it_c.y[1], y2 = it_c.y[2];
          double v[6];
#pragma unroll
          for (int r = 0; r < 6; ++r) {
            double t = Yi[r * 6] * y0.x;
            t = fma(Yi[r * 6 + 1], y0.y, t);
            t = fma(Yi[r * 6 + 2], y1.x, t);
            t = fma(Yi[r * 6 + 3], y1.y, t);
            t = fma(Yi[r * 6 + 4], y2.x, t);
            t = fma(Yi[r * 6 + 5], y2.y, t);
            v[r] = t;
          }
          double2 a0 = ap[0], a1 = ap[1], a2 = ap[2];
          a0.x += v[0]; a0.y += v[1];
          a1.x += v[2]; a1.y += v[3];
          a2.x += v[4]; a2.y += v[5];
          ap[0] = a0; ap[1] = a1; ap[2] = a2;
        }
        __syncwarp();   // the next pair may touch the same output columns from other lanes
        cur = nxt;
        it_c = it_n;
        have = have_n;
      }
    }
    lo_cur = lo_nxt;
    hi_cur = hi_nxt;
  }
  // S strip = base - acc   (upper triangle in block granularity), rows written as contiguous runs
  if (!active) return;
  __syncwarp();
  const int nblk = min(SY_SUB, a.n_f - subbase);
  const size_t row0 = (size_t)6 * f;
  for (int r = 0; r < 6; ++r) {
    for (int cl = lane; cl < nblk * 6; cl += 32) {
      const int fl = cl / 6, c = cl - fl * 6;
      const int fp = subbase + fl;
      if (fp < f) continue;
      double base = 0.0;
      if (fp == f) base = a.Hff[(size_t)f * 36 + r * 6 + c];
      a.S[(row0 + r) * a.ld + (size_t)6 * subbase + cl] = base - acc[fl * 36 + c * 6 + r];
    }
  }
}

// border strip of block row f:  [H_fs | g_f] - sum_e Y_ef^T Yb_e.  Every pair of column f meets every
// border block, so a lane owns fixed border columns and keeps their 6-row outputs in registers:
// lane = (slot u, column); the (warp, slot) slices stride over the staged pairs and are summed in a
// fixed order at the end.  Y_ef and e are staged per batch exactly as in schur_syrk_kernel.
constexpr int SB_WARPS = 4;
constexpr int SB_MAXPASS = 4;   // up to 128 border columns (n_shared <= 125)
__global__ void __launch_bounds__(SB_WARPS * 32) schur_border_kernel(const __grid_constant__ SchurSyrkArgs a) {
  __shared__ __align__(16) double yi[2][SY_BATCH * 36];
  __shared__ int se[2][SY_BATCH];
  __shared__ double red[SB_WARPS * 32 * 6];
  const int f = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncol = a.n_bb * 6;
  const int cw = min(32, ncol);          // columns per pass
  const int U = 32 / cw;                 // pair slots per warp
  const int npass = (ncol + 31) / 32;
  const int u = lane / cw, cl = lane - u * cw;
  const bool lane_on = u < U;
  const int c0 = a.col_ptr[f], c1 = a.col_ptr[f + 1];
  double acc[SB_MAXPASS][6];
#pragma unroll
  for (int ps = 0; ps < SB_MAXPASS; ++ps)
#pragma unroll
    for (int r = 0; r < 6; ++r) acc[ps][r] = 0.0;

  auto stage = [&](int cb, int buf) {
    const int nb = min(SY_BATCH, c1 - cb);
    double2* dst = reinterpret_cast<double2*>(yi[buf]);
    for (int k = tid; k < nb * 18; k += SB_WARPS * 32) {
      const int q = k / 18, piece = k - q * 18;
      const int p = a.col_pair[cb + q];
      sy_cp_async16(dst + k, reinterpret_cast<const double2*>(a.Y + (size_t)p * 36) + piece);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (tid < nb) se[buf][tid] = a.pair_e[a.col_pair[cb + tid]];
  };
  if (c0 < c1) stage(c0, 0);
  int buf = 0;
  for (int cb = c0; cb < c1; cb += SY_BATCH, buf ^= 1) {
    const int nb = min(SY_BATCH, c1 - cb);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    if (cb + SY_BATCH < c1) stage(cb + SY_BATCH, buf ^ 1);
    if (lane_on) {
#pragma unroll 2
      for (int q = warp * U + u; q < nb; q += SB_WARPS * U) {
        const int e = se[buf][q];
        const double2* Yi = reinterpret_cast<const double2*>(yi[buf] + q * 36);
#pragma unroll
        for (int ps = 0; ps < SB_MAXPASS; ++ps) {
          const int col = ps * 32 + cl;
          if (ps < npass && col < ncol) {
            const double2* yp =
                reinterpret_cast<const double2*>(a.Yb + ((size_t)e * a.n_bb + col / 6) * 36 + (col % 6) * 6);
            const double2 y0 = yp[0], y1 = yp[1], y2 = yp[2];
#pragma unroll
            for (int r = 0; r < 6; ++r) {
              const double2 u0 = Yi[3 * r], u1 = Yi[3 * r + 1], u2 = Yi[3 * r + 2];
              double t = u0.x * y0.x;
              t = fma(u0.y, y0.y, t);
              t = fma(u1.x, y1.x, t);
              t = fma(u1.y, y1.y, t);
              t = fma(u2.x, y2.x, t);
              t = fma(u2.y, y2.y, t);
              acc[ps][r] += t;
            }
          }
        }
      }
    }
  }
  // fixed-order sum over the (warp, slot) slices
#pragma unroll
  for (int ps = 0; ps < SB_MAXPASS; ++ps) {
    if (ps >= npass) break;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 6; ++r) red[tid * 6 + r] = acc[ps][r];
    __syncthreads();
    const int col = ps * 32 + tid;
    if (tid < cw && col < ncol) {
      const int gc = 6 * a.n_f + col;
      if (gc < a.ld) {
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          double sum = 0.0;
          for (int w = 0; w < SB_WARPS; ++w)
            for (int uu = 0; uu < U; ++uu) sum += red[(w * 32 + uu * cw + tid) * 6 + r];
          double base = 0.0;
          if (col < a.n_shared) base = a.Hfs[((size_t)f * 6 + r) * a.n_shared + col];
          else if (col == a.n_shared) base = a.gf[(size_t)f * 6 + r];
          a.S[((size_t)6 * f + r) * a.ld + gc] = base - sum;
        }
      }
    }
  }
}

void launch_schur_syrk(const SchurSyrkArgs& a, cudaStream_t s) {
  if (a.n_f == 0) return;
  const size_t smem = (size_t)(SY_WARPS * SY_SUB * 36 + 2 * SY_BATCH * 36) * sizeof(double);
  static SmemOptIn optin;
  optin.ensure(schur_syrk_kernel, smem);
  if (a.n_ctas > 0) schur_syrk_kernel<<<a.n_ctas, SY_WARPS * 32, smem, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

void launch_schur_border(const SchurSyrkArgs& a, cudaStream_t s) {
  if (a.n_f == 0) return;
  RCC_REQUIRE(a.n_bb * 6 <= 32 * SB_MAXPASS, RCC_BAD_ARG, "schur_border: more than 128 border columns");
  schur_border_kernel<<<a.n_f, SB_WARPS * 32, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
// shared x shared corner:  H_ss - sum_e Yb_e^T Yb_e   (and the rhs of the border)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) schur_shared_partial_kernel(const SchurSharedArgs a) {
  const int nb = a.n_bb * 6;
  const int slice = blockIdx.x;
  const int per = (a.n_e + SHARED_SLICES - 1) / SHARED_SLICES;
  const int e0 = slice * per, e1 = min(a.n_e, e0 + per);
  for (int o = threadIdx.x; o < nb * nb; o += blockDim.x) {
    const int s1 = o / nb, s2 = o - s1 * nb;
    double acc = 0.0;
    if (s2 >= s1) {
      for (int e = e0; e < e1; ++e) {
        const double* y1 = a.Yb + ((size_t)e * a.n_bb + s1 / 6) * 36 + (s1 % 6) * 6;
        const double* y2 = a.Yb + ((size_t)e * a.n_bb + s2 / 6) * 36 + (s2 % 6) * 6;
        double v = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) v = fma(y1[k], y2[k], v);
        acc += v;
      }
    }
    a.scratch[(size_t)slice * nb * nb + o] = acc;
  }
}

__global__ void __launch_bounds__(256) schur_shared_final_kernel(const SchurSharedArgs a) {
  const int nb = a.n_bb * 6;
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= nb * nb) return;
  const int s1 = o / nb, s2 = o - s1 * nb;
  if (s1 >= a.n_shared || s2 < s1) return;
  const int gc = 6 * a.n_f + s2;
  if (gc >= a.ld) return;
  double acc = 0.0;
  for (int q = 0; q < SHARED_SLICES; ++q) acc += a.scratch[(size_t)q * nb * nb + o];
  double base = 0.0;
  if (s2 < a.n_shared) base = a.Hss[(size_t)s1 * a.n_shared + s2];
  else if (s2 == a.n_shared) base = a.gs[s1];
  a.S[((size_t)6 * a.n_f + s1) * a.ld + gc] = base - acc;
}

void launch_schur_shared(const SchurSharedArgs& a, cudaStream_t s) {
  const int nb = a.n_bb * 6;
  schur_shared_partial_kernel<<<SHARED_SLICES, 256, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
  schur_shared_final_kernel<<<ceil_div(nb * nb, 256), 256, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
// tail rows of the reduced buffer (ride along in the all-reduce)
// ---------------------------------------------------------------------------
__global__ void reduced_tail_kernel(const ReducedTailArgs a) {
  const int n = 6 * a.n_f + a.n_shared;
  double* tail = a.S + (size_t)n * a.ld;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    double hd, g;
    if (i < 6 * a.n_f) {
      const int f = i / 6, k = i - 6 * f;
      hd = a.Hff[(size_t)f * 36 + k * 6 + k];
      g = a.gf[i];
    } else {
      const int s = i - 6 * a.n_f;
      hd = a.Hss[(size_t)s * a.n_shared + s];
      g = a.gs[s];
    }
    tail[i] = hd;
    tail[n + i] = g;
  }
  if (i == 0) {
    double c2 = 0.0;
    for (int c = 0; c < a.n_cam; ++c) c2 += a.cost2_cam[c];
    tail[2 * n + 0] = c2;
    for (int k = 1; k < 8; ++k) tail[2 * n + k] = 0.0;
  }
}

void launch_reduced_tail(const ReducedTailArgs& a, cudaStream_t s) {
  const int n = 6 * a.n_f + a.n_shared;
  reduced_tail_kernel<<<ceil_div(n, 256), 256, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
// LM damping of the kept blocks + constant-parameter mask + rhs extraction
// ---------------------------------------------------------------------------
__global__ void damp_kernel(const MaskArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const double* tail = a.S + (size_t)a.n * a.ld;
  const double d2 = lm_diagonal(tail[i], a.radius, a.min_diag, a.max_diag, a.jacobi);
  a.S[(size_t)i * a.ld + i] += d2;
  a.d2f[i] = d2;
  a.rhs[i] = -a.S[(size_t)i * a.ld + a.n];
  a.gF[i] = tail[a.n + i];
}

__global__ void mask_kernel(const MaskArgs a) {
  const int c = a.const_idx[blockIdx.x];
  for (int k = threadIdx.x; k < a.n; k += blockDim.x) {
    if (k < c) a.S[(size_t)k * a.ld + c] = 0.0;       // column part of the upper triangle
    else if (k > c) a.S[(size_t)c * a.ld + k] = 0.0;  // row part
  }
  if (threadIdx.x == 0) {
    a.S[(size_t)c * a.ld + c] = 1.0;
    a.S[(size_t)c * a.ld + a.n] = 0.0;   // rhs column of the bordered factorisation
    a.rhs[c] = 0.0;
    a.d2f[c] = 0.0;
    a.gF[c] = 0.0;
  }
}

void launch_mask_damp(const MaskArgs& a, cudaStream_t s) {
  damp_kernel<<<ceil_div(a.n, 256), 256, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
  if (a.n_const > 0) {
    mask_kernel<<<a.n_const, 256, 0, s>>>(a);
    RCC_CUDA(cudaGetLastError());
  }
}

// ---------------------------------------------------------------------------
// back-substitution: one warp per eliminated block
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128) backsub_kernel(const BacksubArgs a) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= a.n_e) return;
  double v[6] = {0, 0, 0, 0, 0, 0};
  // 32 pairs per round: their Y records (contiguous in HBM) cross the SM through shared memory as
  // coalesced 16-byte pieces; each lane then multiplies its own record with its kept block's step
  __shared__ __align__(16) double rec_all[4][32 * PREP_REC];
  double* rec = rec_all[threadIdx.x >> 5];
  const int p_end = a.row_ptr[e + 1];
  for (int p0 = a.row_ptr[e]; p0 < p_end; p0 += 32) {
    const int np = min(32, p_end - p0);
    const double2* src = reinterpret_cast<const double2*>(a.Y + (size_t)p0 * 36);
    for (int k = lane; k < np * 18; k += 32) {
      const int q = k / 18;
      reinterpret_cast<double2*>(rec + q * PREP_REC)[k - q * 18] = src[k];
    }
    __syncwarp();
    if (lane < np) {
      const double* y = rec + lane * PREP_REC;
      const double* d = a.delta_F + (size_t)a.pair_f[p0 + lane] * 6;
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        const double dc = d[c];
#pragma unroll
        for (int k = 0; k < 6; ++k) v[k] = fma(y[c * 6 + k], dc, v[k]);
      }
    }
    __syncwarp();
  }
  // border: shared columns times d_shared, plus the g_e column (coefficient 1)
  const double* ds = a.delta_F + (size_t)6 * a.n_f;
  for (int s = lane; s <= a.n_shared; s += 32) {
    const double* y = a.Yb + ((size_t)e * a.n_bb + s / 6) * 36 + (s % 6) * 6;
    const double dc = (s < a.n_shared) ? ds[s] : 1.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) v[k] = fma(y[k], dc, v[k]);
  }
#pragma unroll
  for (int k = 0; k < 6; ++k)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
  if (lane == 0) {
    const double* Li = a.Linv + (size_t)e * 36;
    double mcc = 0.0, dn = 0.0, xn = 0.0;
    const bool owned = a.e_count[e] > 0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      double d = 0.0;
#pragma unroll
      for (int k = i; k < 6; ++k) d += Li[k * 6 + i] * v[k];  // L^-T v
      d = -d;
      a.delta_e[(size_t)e * 6 + i] = d;
      const double x = a.x_e[(size_t)e * 6 + i];
      mcc += -0.5 * a.ge[(size_t)e * 6 + i] * d + 0.5 * a.d2e[(size_t)e * 6 + i] * d * d;
      dn += d * d;
      if (owned) xn += x * x;
    }
    a.partials[(size_t)e * 4 + 0] = mcc;
    a.partials[(size_t)e * 4 + 1] = dn;
    a.partials[(size_t)e * 4 + 2] = xn;
    a.partials[(size_t)e * 4 + 3] = 0.0;
  }
}

void launch_backsub(const BacksubArgs& a, cudaStream_t s) {
  if (a.n_e == 0) return;
  backsub_kernel<<<ceil_div((int64_t)a.n_e * 32, 128), 128, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
// covariance of the eliminated blocks: one warp per eliminated block e, the matrix analogue of backsub_kernel.
// The inverse of [[H_EE, B], [B^T, C]] has the diagonal blocks H_ee^-1 + H_ee^-1 B_e S^-1 B_e^T H_ee^-1, i.e.
//     Cov(e) = L^-T (I + G) L^-1,   G = Y_e S^-1 Y_e^T = sum_{k,l} Y_k S^-1[k, l] Y_l^T
// over the partners k, l of row e.  With U_l = sum_{k<l} Y_k S^-1[k, l] + 1/2 Y_l S^-1[l, l] and T = sum_l U_l Y_l^T,
// G = T + T^T: only the upper triangle of S^-1 is read, each unordered pair once.  Lane j of the warp owns partner
// l = 32 lt + j of partner tile lt and keeps U_l in registers; the partner tiles kt <= lt stream their Y records
// through the warp's shared slice, and every lane multiplies the broadcast Y_k with its own 6 x 6 block of S^-1.
// Each warp owns its e: no atomics, and every sum runs in a fixed order (bitwise reproducible).
// ---------------------------------------------------------------------------
constexpr int COV_WARPS = 4;
constexpr int COV_TILE = 32;   // partners per tile = lanes

// partner k of row e: its record (column-major 6 x 6, Y_k[a][b] at b * 6 + a) and first reduced index
struct CovRow {
  int p0, m;
  __device__ const double* rec(const CovArgs& a, int e, int k) const {
    return k < m ? a.Y + (size_t)(p0 + k) * 36 : a.Yb + ((size_t)e * a.n_bb + (k - m)) * 36;
  }
  __device__ int gidx(const CovArgs& a, int k) const {
    return k < m ? 6 * a.pair_f[p0 + k] : 6 * a.n_f + 6 * (k - m);
  }
};

// stage the records of partners [k0, k0 + nk) of row e into rec and their first reduced indices into gi; border
// records keep only their shared columns (not g_e, not the pad)
__device__ __forceinline__ void cov_stage(const CovArgs& a, const CovRow& row, int e, int k0, int nk, int lane,
                                          double* rec, int* gi) {
  for (int idx = lane; idx < nk * 18; idx += 32) {
    const int q = idx / 18, piece = idx - q * 18;
    const int k = k0 + q;
    double2 v = reinterpret_cast<const double2*>(row.rec(a, e, k))[piece];
    if (k >= row.m && 6 * (k - row.m) + piece / 3 >= a.n_shared) v = make_double2(0.0, 0.0);
    reinterpret_cast<double2*>(rec + q * 36)[piece] = v;
  }
  if (lane < nk) gi[lane] = row.gidx(a, k0 + lane);
}

__global__ void __launch_bounds__(COV_WARPS * 32) cov_eliminated_kernel(const __grid_constant__ CovArgs a) {
  __shared__ __align__(16) double rec_all[COV_WARPS][COV_TILE * 36];
  __shared__ int gi_all[COV_WARPS][COV_TILE];
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (e >= a.n_e) return;
  double* rec = rec_all[warp];
  int* gi = gi_all[warp];
  CovRow row{a.row_ptr[e], a.row_ptr[e + 1] - a.row_ptr[e]};
  const int K = row.m + a.n_bb;
  const int n_tiles = (K + COV_TILE - 1) / COV_TILE;
  const int n = a.n, ld = a.ld;
  double T[36];
#pragma unroll
  for (int i = 0; i < 36; ++i) T[i] = 0.0;

  for (int lt = 0; lt < n_tiles; ++lt) {
    const int l = lt * COV_TILE + lane;
    const bool l_on = l < K;
    const int gl = l_on ? row.gidx(a, l) : 0;
    double U[36];   // U[a * 6 + c]
#pragma unroll
    for (int i = 0; i < 36; ++i) U[i] = 0.0;
    for (int kt = 0; kt <= lt; ++kt) {
      const int nk = min(COV_TILE, K - kt * COV_TILE);
      __syncwarp();
      cov_stage(a, row, e, kt * COV_TILE, nk, lane, rec, gi);
      __syncwarp();
      if (!l_on) continue;
      const int kend = (kt == lt) ? lane + 1 : nk;   // k <= l
      for (int kk = 0; kk < kend; ++kk) {
        const int gk = gi[kk];
        const bool diag = kt == lt && kk == lane;
        double Sb[36];   // S^-1[gk + b][gl + c] at b * 6 + c
        if (!diag && gk + 6 <= n && gl + 6 <= n) {
          // k < l: the block lies strictly in the upper triangle (kept blocks and border blocks ascend with k)
#pragma unroll
          for (int b = 0; b < 6; ++b) {
            const double2* sp = reinterpret_cast<const double2*>(a.Sinv + (size_t)(gk + b) * ld + gl);
#pragma unroll
            for (int i = 0; i < 3; ++i) {
              const double2 v = sp[i];
              Sb[b * 6 + 2 * i] = v.x;
              Sb[b * 6 + 2 * i + 1] = v.y;
            }
          }
        } else {
          // the diagonal block (half of it, mirrored from the upper triangle) or a block that reaches past the
          // last shared parameter (those rows / columns are zero)
#pragma unroll
          for (int b = 0; b < 6; ++b)
#pragma unroll
            for (int c = 0; c < 6; ++c) {
              int r = gk + b, cc = gl + c;
              if (diag && b > c) {
                r = gk + c;
                cc = gl + b;
              }
              const double v = (r < n && cc < n) ? a.Sinv[(size_t)r * ld + cc] : 0.0;
              Sb[b * 6 + c] = diag ? 0.5 * v : v;
            }
        }
        const double* y = rec + kk * 36;
#pragma unroll
        for (int b = 0; b < 6; ++b)
#pragma unroll
          for (int r = 0; r < 6; ++r) {
            const double ykb = y[b * 6 + r];
#pragma unroll
            for (int c = 0; c < 6; ++c) U[r * 6 + c] = fma(ykb, Sb[b * 6 + c], U[r * 6 + c]);
          }
      }
    }
    // T += U_l Y_l^T; the last staged tile is lt itself, so Y_l is this lane's record
    if (l_on) {
      const double* yl = rec + lane * 36;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int s = 0; s < 6; ++s) {
          double t = T[r * 6 + s];
#pragma unroll
          for (int c = 0; c < 6; ++c) t = fma(U[r * 6 + c], yl[c * 6 + s], t);
          T[r * 6 + s] = t;
        }
    }
  }
#pragma unroll
  for (int i = 0; i < 36; ++i)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) T[i] += __shfl_xor_sync(0xffffffffu, T[i], o);
  if (lane != 0) return;
  // M = I + T + T^T (exactly symmetric);  Cov = L^-T M L^-1, upper triangle computed, lower mirrored
  const double* Li = a.Linv + (size_t)e * 36;   // row-major lower triangular
  double X[36];                                 // X = M L^-1
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      double v = 0.0;
#pragma unroll
      for (int k = j; k < 6; ++k) v = fma(T[r * 6 + k] + T[k * 6 + r] + (r == k ? 1.0 : 0.0), Li[k * 6 + j], v);
      X[r * 6 + j] = v;
    }
  double* out = a.cov_e + (size_t)e * 36;
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = i; j < 6; ++j) {
      double v = 0.0;
#pragma unroll
      for (int r = i; r < 6; ++r) v = fma(Li[r * 6 + i], X[r * 6 + j], v);
      out[i * 6 + j] = v;
      out[j * 6 + i] = v;
    }
}

void launch_cov_eliminated(const CovArgs& a, cudaStream_t s) {
  if (a.n_e == 0) return;
  cov_eliminated_kernel<<<ceil_div((int64_t)a.n_e * 32, COV_WARPS * 32), COV_WARPS * 32, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// one thread per output element: the kept diagonal blocks, then the shared block
__global__ void cov_kept_kernel(const __grid_constant__ CovArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nf = (int64_t)a.n_f * 36;
  int g0, r, c;
  double* out;
  if (i < nf) {
    const int f = (int)(i / 36), j = (int)(i - (int64_t)f * 36);
    g0 = 6 * f;
    r = j / 6;
    c = j - 6 * r;
    out = a.cov_f + i;
  } else if (i < nf + (int64_t)a.n_shared * a.n_shared) {
    const int j = (int)(i - nf);
    g0 = 6 * a.n_f;
    r = j / a.n_shared;
    c = j - r * a.n_shared;
    out = a.cov_s + j;
  } else {
    return;
  }
  const int lo = min(r, c), hi = max(r, c);
  *out = a.Sinv[(size_t)(g0 + lo) * a.ld + g0 + hi];
}

void launch_cov_kept(const CovArgs& a, cudaStream_t s) {
  const int64_t total = (int64_t)a.n_f * 36 + (int64_t)a.n_shared * a.n_shared;
  cov_kept_kernel<<<ceil_div(total, 256), 256, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
// cross-covariance blocks (kernels.h CovPairDesc): one warp per work item (pair, chunk of side a, tile of side b).
// Lane j owns item l = l0 + j of side b and accumulates U_l = sum_k C_ak S^-1[k, l] over the chunk, whose records
// stream through the warp's shared slice as in cov_eliminated_kernel; then X = sum_l U_l C_bl^T over the tile is
// summed across the lanes and stored as the item's partial.  cov_pairs_combine_kernel adds a pair's partials in item
// order and applies P_a, P_b and the diagonal term.  Every sum has a fixed order that depends on the pair alone.
// ---------------------------------------------------------------------------

// Sb[b * 6 + c] = S^-1[gk + b][gl + c] for b < wk, c < wl (zero elsewhere and past n), read from the upper triangle
__device__ __forceinline__ void cov_load_block(const double* __restrict__ S, int n, int ld, int gk, int wk, int gl,
                                               int wl, double* Sb) {
  const bool whole = wk == 6 && wl == 6 && gk + 6 <= n && gl + 6 <= n && ((gk | gl) & 1) == 0;
  if (whole && gk + 5 <= gl) {
#pragma unroll
    for (int b = 0; b < 6; ++b) {
      const double2* sp = reinterpret_cast<const double2*>(S + (size_t)(gk + b) * ld + gl);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const double2 v = sp[i];
        Sb[b * 6 + 2 * i] = v.x;
        Sb[b * 6 + 2 * i + 1] = v.y;
      }
    }
  } else if (whole && gl + 5 <= gk) {
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const double2* sp = reinterpret_cast<const double2*>(S + (size_t)(gl + c) * ld + gk);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const double2 v = sp[i];
        Sb[2 * i * 6 + c] = v.x;
        Sb[(2 * i + 1) * 6 + c] = v.y;
      }
    }
  } else {
    // a window that straddles the diagonal, is narrower than 6, or reaches past the last shared parameter
#pragma unroll
    for (int b = 0; b < 6; ++b)
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        const int r = gk + b, cc = gl + c, lo = min(r, cc), hi = max(r, cc);
        Sb[b * 6 + c] = (b < wk && c < wl && hi < n) ? S[(size_t)lo * ld + hi] : 0.0;
      }
  }
}

__global__ void __launch_bounds__(COV_WARPS * 32) cov_pairs_kernel(const __grid_constant__ CovPairsArgs a) {
  __shared__ __align__(16) double rec_all[COV_WARPS][COV_TILE * 36];
  __shared__ int gi_all[COV_WARPS][COV_TILE];
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (w >= a.n_items) return;
  double* rec = rec_all[warp];
  int* gi = gi_all[warp];
  const CovArgs& m = a.m;
  const CovPairItem it = a.items[w];
  const CovPairDesc pd = a.pairs[it.pair];
  CovRow ra{0, 0}, rb{0, 0};
  int Ka = 1, Kb = 1;
  if (pd.e_a >= 0) {
    ra = CovRow{m.row_ptr[pd.e_a], m.row_ptr[pd.e_a + 1] - m.row_ptr[pd.e_a]};
    Ka = ra.m + m.n_bb;
  }
  if (pd.e_b >= 0) {
    rb = CovRow{m.row_ptr[pd.e_b], m.row_ptr[pd.e_b + 1] - m.row_ptr[pd.e_b]};
    Kb = rb.m + m.n_bb;
  }
  const int na = min(COV_PAIR_CHUNK, Ka - it.k0);
  const int l = it.l0 + lane;
  const bool l_on = l < Kb;
  const int gl = pd.e_b >= 0 ? (l_on ? rb.gidx(m, l) : 0) : pd.g_b;
  const int wl = pd.e_b >= 0 ? 6 : pd.w_b, wk = pd.e_a >= 0 ? 6 : pd.w_a;
  double U[36];   // U[r * 6 + c]: row r of side a, column c of item l
#pragma unroll
  for (int i = 0; i < 36; ++i) U[i] = 0.0;
  for (int kt = 0; kt < na; kt += COV_TILE) {
    const int nk = min(COV_TILE, na - kt);
    __syncwarp();
    if (pd.e_a >= 0) {
      cov_stage(m, ra, pd.e_a, it.k0 + kt, nk, lane, rec, gi);
    } else {
      for (int i = lane; i < 36; i += 32) rec[i] = (i % 7 == 0) ? 1.0 : 0.0;   // the identity record
      if (lane == 0) gi[0] = pd.g_a;
    }
    __syncwarp();
    if (!l_on) continue;
    for (int kk = 0; kk < nk; ++kk) {
      double Sb[36];
      cov_load_block(m.Sinv, m.n, m.ld, gi[kk], wk, gl, wl, Sb);
      const double* y = rec + kk * 36;
#pragma unroll
      for (int b = 0; b < 6; ++b)
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          const double ykb = y[b * 6 + r];
#pragma unroll
          for (int c = 0; c < 6; ++c) U[r * 6 + c] = fma(ykb, Sb[b * 6 + c], U[r * 6 + c]);
        }
    }
  }
  // X = U_l C_bl^T (C_bl = I on a kept or shared side); the border records lose their g_e and pad columns
  if (l_on && pd.e_b >= 0) {
    const double* yl = rb.rec(m, pd.e_b, l);
    const int ncol = l < rb.m ? 6 : min(6, m.n_shared - 6 * (l - rb.m));
    double X[36];
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int s = 0; s < 6; ++s) {
        double t = 0.0;
#pragma unroll
        for (int c = 0; c < 6; ++c) t = fma(U[r * 6 + c], c < ncol ? yl[c * 6 + s] : 0.0, t);
        X[r * 6 + s] = t;
      }
#pragma unroll
    for (int i = 0; i < 36; ++i) U[i] = X[i];
  } else if (!l_on) {
#pragma unroll
    for (int i = 0; i < 36; ++i) U[i] = 0.0;
  }
#pragma unroll
  for (int i = 0; i < 36; ++i)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) U[i] += __shfl_xor_sync(0xffffffffu, U[i], o);
  if (lane == 0) {
    double* out = a.partial + (size_t)w * 36;
#pragma unroll
    for (int i = 0; i < 36; ++i) out[i] = U[i];
  }
}

// one 64-thread block per pair: X = the pair's partials summed in item order, M = X (or I + (X + X^T) / 2 for
// (e, e), exactly symmetric), Cov = +-L_a^-T M L_b^-1 with the L^-1 of the eliminated sides only
__global__ void __launch_bounds__(64) cov_pairs_combine_kernel(const __grid_constant__ CovPairsArgs a) {
  __shared__ double M[36], Z[36], O[36];
  const int t = threadIdx.x;
  const int p = a.pair_begin + blockIdx.x;
  const CovPairDesc pd = a.pairs[p];
  const bool same = pd.e_a >= 0 && pd.e_a == pd.e_b;
  if (t < 36) {
    const double* src = a.partial + (size_t)pd.item0 * 36 + t;
    double v = 0.0;
    for (int i = 0; i < pd.n_items; ++i) v += src[(size_t)i * 36];
    M[t] = v;
    O[t] = 0.0;
  }
  __syncthreads();
  const int r = t / 6, c = t - 6 * (t / 6);
  double sym = 0.0;
  if (same && t < 36) sym = 0.5 * (M[r * 6 + c] + M[c * 6 + r]) + (r == c ? 1.0 : 0.0);
  __syncthreads();
  if (same && t < 36) M[t] = sym;
  __syncthreads();
  // Z = M L_b^-1 (Linv row-major lower triangular)
  if (t < 36) {
    double v = M[t];
    if (pd.e_b >= 0) {
      const double* Lb = a.m.Linv + (size_t)pd.e_b * 36;
      v = 0.0;
      for (int j = c; j < 6; ++j) v = fma(M[r * 6 + j], Lb[j * 6 + c], v);
    }
    Z[t] = v;
  }
  __syncthreads();
  // Cov = L_a^-T Z, negated when exactly one side is eliminated; (e, e): the upper triangle, mirrored
  if (t < 36 && !(same && r > c)) {
    double v = Z[t];
    if (pd.e_a >= 0) {
      const double* La = a.m.Linv + (size_t)pd.e_a * 36;
      v = 0.0;
      for (int i = r; i < 6; ++i) v = fma(La[i * 6 + r], Z[i * 6 + c], v);
    }
    if ((pd.e_a >= 0) != (pd.e_b >= 0)) v = -v;
    if (r < pd.rows && c < pd.cols) {
      O[pd.transpose ? c * pd.rows + r : r * pd.cols + c] = v;
      if (same) O[c * pd.cols + r] = v;
    }
  }
  __syncthreads();
  if (t < 36) a.out[(size_t)p * 36 + t] = O[t];
}

void launch_cov_pairs(const CovPairsArgs& a, cudaStream_t s) {
  cov_pairs_kernel<<<ceil_div((int64_t)a.n_items * 32, COV_WARPS * 32), COV_WARPS * 32, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
  cov_pairs_combine_kernel<<<a.n_pairs, 64, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
// small reductions (single CTA, fixed order)
// ---------------------------------------------------------------------------
__device__ void cta_sum3(double s0, double s1, double s2, double* out3) {
  __shared__ double red[3][256];
  red[0][threadIdx.x] = s0;
  red[1][threadIdx.x] = s1;
  red[2][threadIdx.x] = s2;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      red[0][threadIdx.x] += red[0][threadIdx.x + o];
      red[1][threadIdx.x] += red[1][threadIdx.x + o];
      red[2][threadIdx.x] += red[2][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out3[0] = red[0][0];
    out3[1] = red[1][0];
    out3[2] = red[2][0];
  }
}

__global__ void __launch_bounds__(256) f_stats_kernel(const double* gF, const double* d2f, const double* dF,
                                                      const double* x_f, const double* x_s, int n_f, int n_shared,
                                                      double* out3) {
  const int n = 6 * n_f + n_shared;
  double mcc = 0.0, dn = 0.0, xn = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) {
    const double d = dF[i];
    const double x = (i < 6 * n_f) ? x_f[i] : x_s[i - 6 * n_f];
    mcc += -0.5 * gF[i] * d + 0.5 * d2f[i] * d * d;
    dn += d * d;
    xn += x * x;
  }
  cta_sum3(mcc, dn, xn, out3);
}

void launch_f_stats(const double* gF, const double* d2f, const double* delta_F, const double* x_f, const double* x_s,
                    int32_t n_f, int32_t n_shared, double* out3, cudaStream_t s) {
  f_stats_kernel<<<1, 256, 0, s>>>(gF, d2f, delta_F, x_f, x_s, n_f, n_shared, out3);
  RCC_CUDA(cudaGetLastError());
}

__global__ void __launch_bounds__(256) e_stats_kernel(const double* partials, int n_e, double* out3) {
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (int e = threadIdx.x; e < n_e; e += 256) {
    s0 += partials[(size_t)e * 4 + 0];
    s1 += partials[(size_t)e * 4 + 1];
    s2 += partials[(size_t)e * 4 + 2];
  }
  cta_sum3(s0, s1, s2, out3);
}

void launch_e_stats(const double* partials, int32_t n_e, double* out3, cudaStream_t s) {
  e_stats_kernel<<<1, 256, 0, s>>>(partials, n_e, out3);
  RCC_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------
__global__ void apply_kernel(const double* __restrict__ x, const double* __restrict__ d, double* __restrict__ out,
                             int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = x[i] + d[i];
}
void launch_apply(const double* x, const double* d, double* out, int64_t n, cudaStream_t s) {
  if (n == 0) return;
  apply_kernel<<<ceil_div(n, 256), 256, 0, s>>>(x, d, out, n);
  RCC_CUDA(cudaGetLastError());
}

// ---- column bands (overlapped reduction): row i < c0 keeps [c0, c1), row i in [c0, c1) keeps [i, c1)
static __host__ __device__ inline size_t band_row_offset(int64_t i, int64_t c0, int64_t c1) {
  const int64_t w = c1 - c0;
  if (i <= c0) return (size_t)(i * w);
  const int64_t t = i - c0;                     // rows c0 .. i-1 of the triangle: sum_{k=0}^{t-1} (w - k)
  return (size_t)(c0 * w + t * w - t * (t - 1) / 2);
}
size_t packed_band_doubles(int32_t n_rows, int32_t c0, int32_t c1) {
  return band_row_offset(std::min<int64_t>(n_rows, c1), c0, c1);
}
__global__ void __launch_bounds__(256) pack_band_kernel(double* __restrict__ S, int ld, int c0, int c1,
                                                        double* __restrict__ packed, bool to_packed) {
  const int i = blockIdx.x;
  const int start = max(i, c0);
  double* a = S + (size_t)i * ld + start;
  double* b = packed + band_row_offset(i, c0, c1);
  const int len = c1 - start;
  if (to_packed) for (int k = threadIdx.x; k < len; k += 256) b[k] = a[k];
  else for (int k = threadIdx.x; k < len; k += 256) a[k] = b[k];
}
void launch_pack_band(double* S, int32_t ld, int32_t n_rows, int32_t c0, int32_t c1, double* packed, bool to_packed,
                      cudaStream_t s) {
  const int rows = std::min(n_rows, c1);
  if (rows <= 0 || c1 <= c0) return;
  pack_band_kernel<<<rows, 256, 0, s>>>(S, ld, c0, c1, packed, to_packed);
  RCC_CUDA(cudaGetLastError());
}

__global__ void symmetrize_kernel(double* S, int n, int ld) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;  // column
  const int i = blockIdx.y;                             // row
  if (j < n && j > i) S[(size_t)j * ld + i] = S[(size_t)i * ld + j];
}
void launch_symmetrize(double* S, int32_t n, int32_t ld, cudaStream_t s) {
  dim3 grid(ceil_div(n, 256), n);
  symmetrize_kernel<<<grid, 256, 0, s>>>(S, n, ld);
  RCC_CUDA(cudaGetLastError());
}

// one corner (x, y) of a caller's pixel block, widened to FP64: one 16-, 8- or 4-byte load
__device__ __forceinline__ double2 load_corner(const double* p) { return *reinterpret_cast<const double2*>(p); }
__device__ __forceinline__ double2 load_corner(const int32_t* p) {
  const int2 v = *reinterpret_cast<const int2*>(p);
  return make_double2((double)v.x, (double)v.y);
}
__device__ __forceinline__ double2 load_corner(const int16_t* p) {
  const short2 v = *reinterpret_cast<const short2*>(p);
  return make_double2((double)v.x, (double)v.y);
}

// one thread per corner: 16-byte records on both sides; the F-sorted side is a scatter of whole 64-byte blocks
template <typename T>
__global__ void load_pixels_kernel(const T* __restrict__ src, const int32_t* __restrict__ orig,
                                   double* __restrict__ e_pix, const int32_t* __restrict__ f_inv,
                                   double* __restrict__ f_pix, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 4) return;
  const int64_t g = i >> 2;
  const int q = (int)(i & 3);
  double2 v;
  if (src) {
    const int64_t sg = orig ? (int64_t)orig[g] : g;
    v = load_corner(src + sg * 8 + q * 2);
    reinterpret_cast<double2*>(e_pix + g * 8)[q] = v;
  } else {
    v = reinterpret_cast<const double2*>(e_pix + g * 8)[q];
  }
  reinterpret_cast<double2*>(f_pix + (int64_t)f_inv[g] * 8)[q] = v;
}
template <typename T>
void launch_load_pixels(const T* src, const int32_t* orig, double* e_pix, const int32_t* f_inv, double* f_pix,
                        int64_t n, cudaStream_t s) {
  if (n == 0) return;
  load_pixels_kernel<T><<<ceil_div(n * 4, 256), 256, 0, s>>>(src, orig, e_pix, f_inv, f_pix, n);
  RCC_CUDA(cudaGetLastError());
}
template void launch_load_pixels(const double*, const int32_t*, double*, const int32_t*, double*, int64_t, cudaStream_t);
template void launch_load_pixels(const int32_t*, const int32_t*, double*, const int32_t*, double*, int64_t, cudaStream_t);
template void launch_load_pixels(const int16_t*, const int32_t*, double*, const int32_t*, double*, int64_t, cudaStream_t);

__global__ void fill_kernel(double* p, int64_t n, double v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}
void launch_fill(double* p, int64_t n, double v, cudaStream_t s) {
  fill_kernel<<<NUM_SMS_B200 * 8, 256, 0, s>>>(p, n, v);
  RCC_CUDA(cudaGetLastError());
}

// FP64 FMA microbenchmark: 8 independent chains per thread
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
  }
  const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 12345.678) out[0] = s;
}
double launch_fp64_peak(int iters, double* sink, cudaStream_t s) {
  const int grid = NUM_SMS_B200 * 8;
  fp64_peak_kernel<<<grid, 256, 0, s>>>(sink, iters);   // sink: 8 bytes on the current device, never written
  RCC_CUDA(cudaGetLastError());
  return (double)grid * 256.0 * (double)iters * 64.0;  // FMAs
}

}  // namespace rcc
