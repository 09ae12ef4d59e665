// Dispatcher of K2 (iSIR / GLMCMC) over theta_dim; kernels are instantiated per dimension in
// step_isir_d{1..4}.cu so they compile in parallel.
#include "step_isir.cuh"

namespace glabc {

extern template cudaError_t launch_isir_dim<1>(const ModelConsts&, const GaussConsts&, const GaussConsts&, const RunParams&, bool, bool, int, int, cudaStream_t);
extern template cudaError_t launch_isir_dim<2>(const ModelConsts&, const GaussConsts&, const GaussConsts&, const RunParams&, bool, bool, int, int, cudaStream_t);
extern template cudaError_t launch_isir_dim<3>(const ModelConsts&, const GaussConsts&, const GaussConsts&, const RunParams&, bool, bool, int, int, cudaStream_t);
extern template cudaError_t launch_isir_dim<4>(const ModelConsts&, const GaussConsts&, const GaussConsts&, const RunParams&, bool, bool, int, int, cudaStream_t);

cudaError_t launch_isir(const ModelConsts& model, const GaussConsts& lp, const GaussConsts& ip, int dim, const RunParams& R,
                        bool strict, bool replay, int layout, int block, cudaStream_t st)
{
    return with_dim(dim, [&](auto d) { return launch_isir_dim<d>(model, lp, ip, R, strict, replay, layout, block, st); });
}

}  // namespace glabc
