// K3 instantiations for theta_dim = 3
#include "step_mala_fast.cuh"

namespace glabc {
template cudaError_t launch_mala_dim<3>(const MalaConsts&, const DistConsts&, const RunParams&, bool, bool, int, cudaStream_t);
}  // namespace glabc
