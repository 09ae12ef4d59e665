// Dispatcher of K3 (GLMALA) over theta_dim; kernels are instantiated per dimension in
// step_mala_d{1..4}.cu so they compile in parallel.
#include "step_mala.cuh"

namespace glabc {

extern template cudaError_t launch_mala_dim<1>(const MalaConsts&, const DistConsts&, const RunParams&, bool, bool, int, cudaStream_t);
extern template cudaError_t launch_mala_dim<2>(const MalaConsts&, const DistConsts&, const RunParams&, bool, bool, int, cudaStream_t);
extern template cudaError_t launch_mala_dim<3>(const MalaConsts&, const DistConsts&, const RunParams&, bool, bool, int, cudaStream_t);
extern template cudaError_t launch_mala_dim<4>(const MalaConsts&, const DistConsts&, const RunParams&, bool, bool, int, cudaStream_t);

cudaError_t launch_mala(const MalaConsts& K, const DistConsts& prior, int dim, const RunParams& R, bool strict, bool replay, int block,
                        cudaStream_t st)
{
    return with_dim(dim, [&](auto d) { return launch_mala_dim<d>(K, prior, R, strict, replay, block, st); });
}

}  // namespace glabc
