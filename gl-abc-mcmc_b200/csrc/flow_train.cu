// Host launchers of the flow's training step (flow_train.cuh).
#include <cmath>

#include "flow_train.cuh"

namespace glabc {

cudaError_t launch_flow_bwd(const FlowDev& W, const float* z_final, int64_t n, float* partial, int n_slices, cudaStream_t st)
{
    if (n <= 0 || n_slices <= 0) return cudaSuccess;
    if (W.w2p_lo == nullptr) return cudaErrorInvalidValue;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(k_flow_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, kTrSmemBytes);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    k_flow_bwd<<<static_cast<unsigned>(n_slices), kTrThreads, kTrSmemBytes, st>>>(W, z_final, n, partial);
    return cudaGetLastError();
}

cudaError_t launch_flow_grad_reduce(const float* partial, int n_slices, int64_t total, int64_t n, float* grad, cudaStream_t st)
{
    k_flow_grad_reduce<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(partial, n_slices, total, 1.0f / static_cast<float>(n), grad);
    return cudaGetLastError();
}

cudaError_t launch_flow_loss(const float* lq, int64_t n, float* loss, cudaStream_t st)
{
    k_flow_loss<<<1, 1024, 0, st>>>(lq, n, loss);
    return cudaGetLastError();
}

cudaError_t launch_flow_adam(float* p, float* m, float* v, const float* g, int64_t total, const float* loss, float lr, float beta1, float beta2,
                             float eps, float wd, int64_t t, cudaStream_t st)
{
    const float bc1 = static_cast<float>(1.0 - std::pow(static_cast<double>(beta1), static_cast<double>(t)));
    const float bc2_sqrt = static_cast<float>(std::sqrt(1.0 - std::pow(static_cast<double>(beta2), static_cast<double>(t))));
    k_flow_adam<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(p, m, v, g, total, loss, lr, beta1, beta2, eps, wd, bc1, bc2_sqrt);
    return cudaGetLastError();
}

int flow_train_chunk_samples() { return kTrTiles * kFlowTile; }
int64_t flow_param_count(int n_blocks) { return FlowParamLayout(n_blocks).total; }

}  // namespace glabc
