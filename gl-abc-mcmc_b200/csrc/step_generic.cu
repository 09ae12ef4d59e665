// Launchers of the general-proposal GlobalMCMC / GLMCMC kernels (the model's DiagGaussian prior or a bound general one)
// and of the device-side distribution evaluation (step_generic.cuh).
#include "step_generic.cuh"

namespace glabc {

cudaError_t launch_global_generic(const GenericConsts& K, const DistConsts& prior, int dim, const RunParams& R, int layout, int block,
                                  bool replay, cudaStream_t st)
{
    if (replay && generic_prior(prior)) return cudaErrorInvalidValue;
    if (block > 128) block = 128;
    return with_dim(dim, [&](auto d) {
        const unsigned grid = static_cast<unsigned>((R.n_chains + block - 1) / block);
        if (replay) k_global_generic<d, true, false><<<grid, block, 0, st>>>(K, R, layout, prior);
        else if (generic_prior(prior)) k_global_generic<d, false, true><<<grid, block, 0, st>>>(K, R, layout, prior);
        else k_global_generic<d, false, false><<<grid, block, 0, st>>>(K, R, layout, prior);
        return cudaGetLastError();
    });
}

cudaError_t launch_isir_generic(const IsirGenericConsts& K, const DistConsts& prior, int dim, const RunParams& R, int layout, int block,
                                bool replay, cudaStream_t st)
{
    if (replay && generic_prior(prior)) return cudaErrorInvalidValue;
    if (block > 128) block = 128;
    return with_dim(dim, [&](auto d) {
        const unsigned grid = static_cast<unsigned>((R.n_chains + block - 1) / block);
        if (replay) k_isir_generic<d, true, false><<<grid, block, 0, st>>>(K, R, layout, prior);
        else if (generic_prior(prior)) k_isir_generic<d, false, true><<<grid, block, 0, st>>>(K, R, layout, prior);
        else k_isir_generic<d, false, false><<<grid, block, 0, st>>>(K, R, layout, prior);
        return cudaGetLastError();
    });
}

cudaError_t launch_dist_eval(const DistConsts& q, int dim, const RoundKeys& rk, int64_t n, const float* z_in, float* z_out, float* logp,
                             cudaStream_t st)
{
    if (n <= 0) return cudaSuccess;
    const unsigned grid = static_cast<unsigned>((n + 255) / 256);
    return with_dim(dim, [&](auto d) {
        k_dist_eval<d><<<grid, 256, 0, st>>>(q, rk, n, z_in, z_out, logp);
        return cudaGetLastError();
    });
}

}  // namespace glabc
