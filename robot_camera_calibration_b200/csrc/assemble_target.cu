// K2 with the corners of a corner layout (rcc_ba_set_corner_layout), radial-tangential lens: assemble_target_kernel,
// the body of assemble.cuh with the TARGET corner source (chunk.cuh), compiled in its own translation unit so that its
// 16 instantiations build in parallel with the others.
#include "assemble.cuh"

namespace rcc {

void launch_assemble_target(bool rig, bool epass, bool own_is_view, const AssembleArgs& a, cudaStream_t s) {
  if (a.loss != 0) launch_assemble_l<true, LENS_RADTAN, true>(rig, epass, own_is_view, a, s);
  else launch_assemble_l<false, LENS_RADTAN, true>(rig, epass, own_is_view, a, s);
}

}  // namespace rcc
