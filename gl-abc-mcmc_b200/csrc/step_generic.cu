// Launchers of the general-proposal GlobalMCMC / GLMCMC kernels (the model's DiagGaussian prior or a bound general one)
// and of the device-side distribution evaluation (step_generic.cuh).
#include "step_generic.cuh"

namespace glabc {

template <int D, int FAMILY>
static void global_generic_family(const GenericConsts& K, const DistConsts& prior, const RunParams& R, int layout, unsigned grid,
                                  int block, bool replay, cudaStream_t st)
{
    if (replay) k_global_generic<D, FAMILY, true, false><<<grid, block, 0, st>>>(K, R, layout, prior);
    else if (generic_prior(prior)) k_global_generic<D, FAMILY, false, true><<<grid, block, 0, st>>>(K, R, layout, prior);
    else k_global_generic<D, FAMILY, false, false><<<grid, block, 0, st>>>(K, R, layout, prior);
}

template <int D>
static cudaError_t generic_dim(const GenericConsts& K, const DistConsts& prior, const RunParams& R, int layout, int block, bool replay,
                               cudaStream_t st)
{
    const unsigned grid = static_cast<unsigned>((R.n_chains + block - 1) / block);
    if (K.model.family == GLABC_MODEL_ABS_NORMAL) global_generic_family<D, GLABC_MODEL_ABS_NORMAL>(K, prior, R, layout, grid, block, replay, st);
    else global_generic_family<D, GLABC_MODEL_ID_NORMAL>(K, prior, R, layout, grid, block, replay, st);
    return cudaGetLastError();
}

cudaError_t launch_global_generic(const GenericConsts& K, const DistConsts& prior, int dim, const RunParams& R, int layout, int block,
                                  bool replay, cudaStream_t st)
{
    if (replay && generic_prior(prior)) return cudaErrorInvalidValue;
    if (block > 128) block = 128;
    switch (dim) {
    case 1: return generic_dim<1>(K, prior, R, layout, block, replay, st);
    case 2: return generic_dim<2>(K, prior, R, layout, block, replay, st);
    case 3: return generic_dim<3>(K, prior, R, layout, block, replay, st);
    case 4: return generic_dim<4>(K, prior, R, layout, block, replay, st);
    default: return cudaErrorInvalidValue;
    }
}

template <int D, int FAMILY>
static void isir_generic_family(const IsirGenericConsts& K, const DistConsts& prior, const RunParams& R, int layout, unsigned grid,
                                int block, bool replay, cudaStream_t st)
{
    if (replay) k_isir_generic<D, FAMILY, true, false><<<grid, block, 0, st>>>(K, R, layout, prior);
    else if (generic_prior(prior)) k_isir_generic<D, FAMILY, false, true><<<grid, block, 0, st>>>(K, R, layout, prior);
    else k_isir_generic<D, FAMILY, false, false><<<grid, block, 0, st>>>(K, R, layout, prior);
}

template <int D>
static cudaError_t isir_generic_dim(const IsirGenericConsts& K, const DistConsts& prior, const RunParams& R, int layout, int block,
                                    bool replay, cudaStream_t st)
{
    const unsigned grid = static_cast<unsigned>((R.n_chains + block - 1) / block);
    if (K.model.family == GLABC_MODEL_ABS_NORMAL) isir_generic_family<D, GLABC_MODEL_ABS_NORMAL>(K, prior, R, layout, grid, block, replay, st);
    else isir_generic_family<D, GLABC_MODEL_ID_NORMAL>(K, prior, R, layout, grid, block, replay, st);
    return cudaGetLastError();
}

cudaError_t launch_isir_generic(const IsirGenericConsts& K, const DistConsts& prior, int dim, const RunParams& R, int layout, int block,
                                bool replay, cudaStream_t st)
{
    if (replay && generic_prior(prior)) return cudaErrorInvalidValue;
    if (block > 128) block = 128;
    switch (dim) {
    case 1: return isir_generic_dim<1>(K, prior, R, layout, block, replay, st);
    case 2: return isir_generic_dim<2>(K, prior, R, layout, block, replay, st);
    case 3: return isir_generic_dim<3>(K, prior, R, layout, block, replay, st);
    case 4: return isir_generic_dim<4>(K, prior, R, layout, block, replay, st);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_dist_eval(const DistConsts& q, int dim, const RoundKeys& rk, int64_t n, const float* z_in, float* z_out, float* logp,
                             cudaStream_t st)
{
    if (n <= 0) return cudaSuccess;
    const unsigned grid = static_cast<unsigned>((n + 255) / 256);
    switch (dim) {
    case 1: k_dist_eval<1><<<grid, 256, 0, st>>>(q, rk, n, z_in, z_out, logp); break;
    case 2: k_dist_eval<2><<<grid, 256, 0, st>>>(q, rk, n, z_in, z_out, logp); break;
    case 3: k_dist_eval<3><<<grid, 256, 0, st>>>(q, rk, n, z_in, z_out, logp); break;
    case 4: k_dist_eval<4><<<grid, 256, 0, st>>>(q, rk, n, z_in, z_out, logp); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

}  // namespace glabc
