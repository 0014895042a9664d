// K1 -- materialised cost-functor evaluation (residuals + per-parameter-block
// Jacobians in the Ceres CostFunction::Evaluate layout: materialise_kernel), and
// K6's cost-only evaluation used for the LM gain ratio (evaluate_kernel).  The
// kernel templates are in evaluate.cuh.
//
// K1 is HBM-write-bound: 1 408 B out per 72 B in per observation block.
#include "evaluate.cuh"

namespace rcc {

int eval_grid(int64_t n) {
  const int64_t groups = (n + 7) / 8;
  return (int)std::max<int64_t>(1, std::min<int64_t>((groups + EVAL_THREADS / 32 - 1) / (EVAL_THREADS / 32),
                                                     (int64_t)NUM_SMS_B200 * EVAL_CTAS_PER_SM));
}

int eval_partials(bool want_jac, const EvalArgs& a) { return want_jac ? a.n_chunks : eval_grid(a.n); }

void launch_evaluate(bool rig, bool want_jac, int lens, const EvalArgs& a, cudaStream_t s) {
  if (a.n == 0) return;
  if (a.corners) launch_evaluate_target(rig, want_jac, lens, a, s);
  else launch_evaluate_any<false>(rig, want_jac, lens, a, s);
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
