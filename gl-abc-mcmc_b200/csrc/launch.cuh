// Host-callable launchers of the sampler kernels (one translation unit per sampler).
#pragma once
#include <cuda_runtime.h>

#include <type_traits>

#include "sampler_common.cuh"

namespace glabc {

// The theta dimensions the kernels are instantiated for: f(std::integral_constant<int, D>{}) for D in 1..4.
template <class F>
cudaError_t with_dim(int dim, F&& f)
{
    switch (dim) {
    case 1: return f(std::integral_constant<int, 1>{});
    case 2: return f(std::integral_constant<int, 2>{});
    case 3: return f(std::integral_constant<int, 3>{});
    case 4: return f(std::integral_constant<int, 4>{});
    }
    return cudaErrorInvalidValue;
}

// The link of the fused model family as a compile-time constant, for the tuned kernels that read it at compile time.
template <class F>
cudaError_t with_family(int family, F&& f)
{
    switch (family) {
    case GLABC_MODEL_ABS_NORMAL: return f(std::integral_constant<int, GLABC_MODEL_ABS_NORMAL>{});
    case GLABC_MODEL_ID_NORMAL: return f(std::integral_constant<int, GLABC_MODEL_ID_NORMAL>{});
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_global_mcmc(const ModelConsts& model, const GaussConsts& lp, const GaussConsts& gp, int dim,
                               const RunParams& R, bool strict, bool replay, int layout, int block, cudaStream_t st);

cudaError_t launch_isir(const ModelConsts& model, const GaussConsts& lp, const GaussConsts& ip, int dim, const RunParams& R,
                        bool strict, bool replay, int layout, int block, cudaStream_t st);

struct MalaConsts;
template <int MAXD>
struct DistConstsT;
using DistConsts = DistConstsT<4>;   // dist_device.cuh; the built-in kernels take distributions of dim <= 4
// `prior`: a Uniform / Gamma / GaussianMixture prior of the model (FAST, native RNG) or GLABC_DIST_DIAG_GAUSSIAN for K.model's
cudaError_t launch_mala(const MalaConsts& K, const DistConsts& prior, int dim, const RunParams& R, bool strict, bool replay, int block,
                        cudaStream_t st);

cudaError_t launch_esjd(const float* trace, int layout, int64_t rows, int64_t chains, int dim, float* out,
                        cudaStream_t st);

cudaError_t launch_summarize(const float* stats, int64_t chains, int dim, double* out, cudaStream_t st);

cudaError_t launch_resample(const float* w, int64_t n, int64_t N, float u0, int64_t* idx, unsigned long long* count, double* scratch,
                            cudaStream_t st);

cudaError_t launch_philox_kat(const uint32_t* ctr, const uint32_t* key, int64_t n, uint32_t* out, cudaStream_t st);

}  // namespace glabc
