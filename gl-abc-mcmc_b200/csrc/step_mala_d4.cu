// K3 instantiations for theta_dim = 4
#include "step_mala_fast.cuh"

namespace glabc {
template cudaError_t launch_mala_dim<4>(const MalaConsts&, const DistConsts&, const RunParams&, bool, bool, int, cudaStream_t);
}  // namespace glabc
