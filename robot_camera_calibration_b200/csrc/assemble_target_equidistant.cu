// K2 with the corners of a corner layout, equidistant lens (see assemble_target.cu).
#include "assemble.cuh"

namespace rcc {

void launch_assemble_target_equidistant(bool rig, bool epass, bool own_is_view, const AssembleArgs& a, cudaStream_t s) {
  if (a.loss != 0) launch_assemble_l<true, LENS_EQUIDISTANT, true>(rig, epass, own_is_view, a, s);
  else launch_assemble_l<false, LENS_EQUIDISTANT, true>(rig, epass, own_is_view, a, s);
}

}  // namespace rcc
