// Host launchers of K4 (RealNVP flow on tcgen05 tensor cores: flow.cuh, flow_pipe.cuh).
#include "flow.cuh"
#include "flow_pipe.cuh"

namespace glabc {

cudaError_t launch_flow_pack(const float* w2, float* w2p, float* w2p_lo, int n_blocks, cudaStream_t st)
{
    const int64_t total = static_cast<int64_t>(n_blocks) * kFlowHidden * kFlowHidden;
    if (total <= 0) return cudaSuccess;
    k_flow_pack<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(w2, w2p, w2p_lo, total);
    return cudaGetLastError();
}

cudaError_t launch_flow_pack_aux(const float* w1, const float* b1, const float* b2, const float* w3, const float* b3, uint8_t* aux,
                                 int n_blocks, cudaStream_t st)
{
    if (n_blocks <= 0) return cudaSuccess;
    k_flow_pack_aux<<<n_blocks, 256, 0, st>>>(w1, b1, b2, w3, b3, aux);
    return cudaGetLastError();
}

cudaError_t launch_flow(const FlowDev& W, bool sample, bool precise, const float* in, int64_t n, float* out_theta, float* out_lq,
                        int sm_count, cudaStream_t st)
{
    if (n <= 0) return cudaSuccess;
    if (W.aux == nullptr || (precise && W.w2p_lo == nullptr)) return cudaErrorInvalidValue;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(k_flow_pipe<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPipeSmemBytes);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_flow_pipe<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPipeSmemBytes);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_flow_pipe_precise<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPipePSmemBytes);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_flow_pipe_precise<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPipePSmemBytes);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    // tiles per chunk: at most what the shared-memory state holds, sized so that the chunks divide evenly over the SMs, rounded
    // up to an even count (the pipelines' measured throughput was taken with this geometry)
    const int64_t tiles = (n + kFlowTile - 1) / kFlowTile;
    const int64_t waves = (tiles + int64_t(sm_count) * kFlowTilesPerCta - 1) / (int64_t(sm_count) * kFlowTilesPerCta);
    int64_t tpc = (tiles + sm_count * waves - 1) / (sm_count * waves);   // every SM gets `waves` chunks of (almost) equal size
    tpc = (tpc + 1) / 2 * 2;
    if (tpc < 2) tpc = 2;
    if (tpc > kFlowTilesPerCta) tpc = kFlowTilesPerCta;
    if (tpc < kPipeMinTiles) tpc = kPipeMinTiles;   // the pipelines' smallest chunk (flow_pipe.cuh)
    const int64_t chunks = (tiles + tpc - 1) / tpc;
    const unsigned grid = static_cast<unsigned>(chunks < sm_count ? chunks : sm_count);  // persistent: one CTA per SM
    if (precise) {
        if (sample) k_flow_pipe_precise<true><<<grid, 18 * 32, kPipePSmemBytes, st>>>(W, in, n, out_theta, out_lq, static_cast<int>(tpc));
        else k_flow_pipe_precise<false><<<grid, 18 * 32, kPipePSmemBytes, st>>>(W, in, n, out_theta, out_lq, static_cast<int>(tpc));
    } else {
        if (sample) k_flow_pipe<true><<<grid, kPipeThreads, kPipeSmemBytes, st>>>(W, in, n, out_theta, out_lq, static_cast<int>(tpc));
        else k_flow_pipe<false><<<grid, kPipeThreads, kPipeSmemBytes, st>>>(W, in, n, out_theta, out_lq, static_cast<int>(tpc));
    }
    return cudaGetLastError();
}

}  // namespace glabc

#ifdef GLABC_FLOW_TRACE
extern "C" __attribute__((visibility("default"))) int glabc_debug_pipe_trace(long long* out)
{
    return static_cast<int>(cudaMemcpyFromSymbol(out, glabc::g_pipe_trace, sizeof(glabc::g_pipe_trace)));
}
#endif
