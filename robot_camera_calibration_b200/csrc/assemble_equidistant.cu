// K2 for the equidistant lens: the same kernel template as assemble.cu (assemble.cuh), compiled in its own
// translation unit so that its 16 instantiations build in parallel with the radial-tangential ones.
#include "assemble.cuh"

namespace rcc {

void launch_assemble_equidistant(bool rig, bool epass, bool own_is_view, const AssembleArgs& a, cudaStream_t s) {
  if (a.loss != 0) launch_assemble_l<true, LENS_EQUIDISTANT>(rig, epass, own_is_view, a, s);
  else launch_assemble_l<false, LENS_EQUIDISTANT>(rig, epass, own_is_view, a, s);
}

}  // namespace rcc
