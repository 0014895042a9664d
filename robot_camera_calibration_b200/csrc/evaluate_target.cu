// K1 and K6 with the corners of a corner layout (rcc_ba_set_corner_layout): materialise_target_kernel and
// evaluate_target_kernel, the bodies of evaluate.cuh with the TARGET corner source, in their own translation unit so
// that they build in parallel with the others.
#include "evaluate.cuh"

namespace rcc {

void launch_evaluate_target(bool rig, bool want_jac, int lens, const EvalArgs& a, cudaStream_t s) {
  launch_evaluate_any<true>(rig, want_jac, lens, a, s);
}

__global__ void sort_slots_kernel(const int32_t* __restrict__ slot, const int32_t* __restrict__ orig,
                                  const int32_t* __restrict__ f_inv, int32_t* __restrict__ e_slot,
                                  int32_t* __restrict__ f_slot, int64_t n) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  const int32_t v = slot[orig[g]];
  e_slot[g] = v;
  f_slot[f_inv[g]] = v;
}

void launch_sort_slots(const int32_t* slot, const int32_t* orig, const int32_t* f_inv, int32_t* e_slot, int32_t* f_slot,
                       int64_t n, cudaStream_t s) {
  if (n == 0) return;
  sort_slots_kernel<<<ceil_div(n, 256), 256, 0, s>>>(slot, orig, f_inv, e_slot, f_slot, n);
  RCC_CUDA(cudaGetLastError());
}

}  // namespace rcc
