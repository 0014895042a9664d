// Gaussian priors on parameter blocks (ceres::NormalPrior): the residual block r_i = A_i (x_i - mu_i) on block x_i,
// linear in the stored parameters (a Rodrigues vector is differenced as a plain 3-vector).
//
// One thread per prior.  Its block is its own: the priors of one kind have distinct indices, view and marker priors
// land in different arrays, and intr / dist / ext occupy disjoint diagonal blocks of a camera's H_ss.  So every
// thread adds into H and g with plain loads and stores.  The cost leaves each CTA as one partial, summed in a fixed
// order (warp shuffles, then the warps in order), and the caller's reduction adds the partials in index order: the
// results are bitwise reproducible, with no atomics.
#include "common.cuh"
#include "kernels.h"

namespace rcc {

constexpr int PRIOR_THREADS = 128;

int prior_grid(int n) { return n > 0 ? ceil_div(n, PRIOR_THREADS) : 0; }

// AtA = A^T A of every prior (6 x 6 row-major, zero padded like A).  Both triangles are computed with the same
// products in the same order, so AtA is exactly symmetric.
__global__ void __launch_bounds__(PRIOR_THREADS) prior_gram_kernel(int n, const double* __restrict__ A,
                                                                   double* __restrict__ AtA) {
  const int i = blockIdx.x * PRIOR_THREADS + threadIdx.x;
  if (i >= n) return;
  const double* a = A + (size_t)i * 36;
  double* g = AtA + (size_t)i * 36;
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      double s = 0.0;
#pragma unroll
      for (int m = 0; m < 6; ++m) s = fma(a[m * 6 + r], a[m * 6 + c], s);
      g[r * 6 + c] = s;
    }
}

template <bool LIN>
__global__ void __launch_bounds__(PRIOR_THREADS) prior_kernel(const PriorArgs a) {
  __shared__ double red[PRIOR_THREADS / 32];
  const int i = blockIdx.x * PRIOR_THREADS + threadIdx.x;
  double c2 = 0.0;
  if (i < a.off[PRIOR_KINDS]) {
    int kind = 0;
    while (i >= a.off[kind + 1]) ++kind;
    const int k = prior_block_size(kind);
    const int idx = a.index[i];
    const double* x;
    double* H = nullptr;
    double* g = nullptr;
    int ldh = 6;
    if (kind == RCC_BLOCK_VIEW || kind == RCC_BLOCK_MARKER) {
      x = (kind == RCC_BLOCK_VIEW ? a.views : a.markers) + (size_t)idx * 6;
      if (LIN) {
        const bool elim = (kind == RCC_BLOCK_VIEW) == (a.elim_view != 0);
        H = (elim ? a.Hee : a.Hff) + (size_t)idx * 36;
        g = (elim ? a.ge : a.gf) + (size_t)idx * 6;
      }
    } else {
      const int o = idx * a.sp + (kind == RCC_BLOCK_INTR ? 0 : kind == RCC_BLOCK_DIST ? 4 : 9);
      x = a.shared + o;
      if (LIN) {
        H = a.Hss + (size_t)o * a.n_shared + o;
        g = a.gs + o;
        ldh = a.n_shared;
      }
    }
    const double* mu = a.mean + (size_t)i * 6;
    const double* A = a.A + (size_t)i * 36;
    double d[6], r[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) d[j] = j < k ? x[j] - mu[j] : 0.0;
#pragma unroll
    for (int m = 0; m < 6; ++m) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < 6; ++j) s = fma(A[m * 6 + j], d[j], s);
      r[m] = s;
      c2 = fma(s, s, c2);
    }
    if (LIN) {
      // g += A^T r = A^T A (x - mu);  H += A^T A (the k x k block; A is zero padded beyond k).  Every load comes
      // before the first store: the pointers may alias as far as the compiler knows, so an interleaved
      // read-modify-write would wait out one memory round trip per element.
      const double* G = a.AtA + (size_t)i * 36;
      double hv[36], gv[6];
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        gv[j] = j < k ? g[j] : 0.0;
#pragma unroll
        for (int l = 0; l < 6; ++l) hv[j * 6 + l] = (j < k && l < k) ? H[(size_t)j * ldh + l] + G[j * 6 + l] : 0.0;
      }
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        double s = 0.0;
#pragma unroll
        for (int m = 0; m < 6; ++m) s = fma(A[m * 6 + j], r[m], s);
        gv[j] += s;
      }
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        if (j >= k) break;
        g[j] = gv[j];
#pragma unroll
        for (int l = 0; l < 6; ++l)
          if (l < k) H[(size_t)j * ldh + l] = hv[j * 6 + l];
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c2 += __shfl_xor_sync(0xffffffffu, c2, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c2;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < PRIOR_THREADS / 32; ++w) s += red[w];
    a.cost2[blockIdx.x] = s;
  }
}

void launch_prior_gram(int n, const double* A, double* AtA, cudaStream_t s) {
  prior_gram_kernel<<<prior_grid(n), PRIOR_THREADS, 0, s>>>(n, A, AtA);
  RCC_CUDA(cudaGetLastError());
}

void launch_prior(bool linearize, const PriorArgs& a, cudaStream_t s) {
  const int grid = prior_grid(a.off[PRIOR_KINDS]);
  if (linearize) prior_kernel<true><<<grid, PRIOR_THREADS, 0, s>>>(a);
  else prior_kernel<false><<<grid, PRIOR_THREADS, 0, s>>>(a);
  RCC_CUDA(cudaGetLastError());
}

}  // namespace rcc
