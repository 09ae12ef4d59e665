// Dispatcher of K1 over theta_dim; the kernels are instantiated one dimension per translation unit
// (step_global_d{1..4}.cu) so they compile in parallel.
#include "step_global.cuh"

namespace glabc {

extern template cudaError_t launch_global_mcmc_dim<1>(const ModelConsts&, const GaussConsts&, const GaussConsts&, const RunParams&, bool, bool, int, int, cudaStream_t);
extern template cudaError_t launch_global_mcmc_dim<2>(const ModelConsts&, const GaussConsts&, const GaussConsts&, const RunParams&, bool, bool, int, int, cudaStream_t);
extern template cudaError_t launch_global_mcmc_dim<3>(const ModelConsts&, const GaussConsts&, const GaussConsts&, const RunParams&, bool, bool, int, int, cudaStream_t);
extern template cudaError_t launch_global_mcmc_dim<4>(const ModelConsts&, const GaussConsts&, const GaussConsts&, const RunParams&, bool, bool, int, int, cudaStream_t);

cudaError_t launch_global_mcmc(const ModelConsts& model, const GaussConsts& lp, const GaussConsts& gp, int dim,
                               const RunParams& R, bool strict, bool replay, int layout, int block, cudaStream_t st)
{
    return with_dim(dim, [&](auto d) { return launch_global_mcmc_dim<d>(model, lp, gp, R, strict, replay, layout, block, st); });
}

}  // namespace glabc
