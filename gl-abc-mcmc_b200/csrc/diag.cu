// Diagnostics: esjd() over device traces (ESJD.py:17-24) and the Philox known-answer kernel.
#include "launch.cuh"

namespace glabc {

template <int D>
__device__ __forceinline__ float esjd_from_gram(const float (&g)[D * (D + 1) / 2], float n)
{
    // det(G / n)^(1/D), G symmetric upper-triangular row-major
    if constexpr (D == 1) {
        return g[0] / n;
    } else if constexpr (D == 2) {
        const float a = g[0] / n, b = g[1] / n, c = g[2] / n;
        return sqrtf(a * c - b * b);
    } else {
        const float a = g[0] / n, b = g[1] / n, c = g[2] / n, d = g[3] / n, e = g[4] / n, f = g[5] / n;
        const float det = a * (d * f - e * e) - b * (b * f - e * c) + c * (b * e - d * c);
        return cbrtf(det);
    }
}

// time-major [rows][chains][D]: one thread per chain, coalesced across chains
template <int D>
__global__ void k_esjd_time_major(const float* __restrict__ trace, int64_t rows, int64_t chains, float* __restrict__ out)
{
    const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= chains) return;
    float g[D * (D + 1) / 2] = {};
    float prev[D];
#pragma unroll
    for (int k = 0; k < D; ++k) prev[k] = trace[c * D + k];
    for (int64_t t = 1; t < rows; ++t) {
        float dl[D];
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float v = trace[(t * chains + c) * D + k];
            dl[k] = v - prev[k];
            prev[k] = v;
        }
        int q = 0;
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = i; j < D; ++j, ++q) g[q] = fmaf(dl[i], dl[j], g[q]);
    }
    out[c] = esjd_from_gram<D>(g, static_cast<float>(rows - 1));
}

// chain-major [chains][rows][D]: one warp per chain, lanes stride the rows
template <int D>
__global__ void k_esjd_chain_major(const float* __restrict__ trace, int64_t rows, int64_t chains, float* __restrict__ out)
{
    const int64_t c = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (c >= chains) return;
    const float* base = trace + c * rows * D;
    float g[D * (D + 1) / 2] = {};
    for (int64_t t = 1 + lane; t < rows; t += 32) {
        float dl[D];
#pragma unroll
        for (int k = 0; k < D; ++k) dl[k] = base[t * D + k] - base[(t - 1) * D + k];
        int q = 0;
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = i; j < D; ++j, ++q) g[q] = fmaf(dl[i], dl[j], g[q]);
    }
#pragma unroll
    for (int q = 0; q < D * (D + 1) / 2; ++q)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) g[q] += __shfl_xor_sync(0xffffffffu, g[q], o);
    if (lane == 0) out[c] = esjd_from_gram<D>(g, static_cast<float>(rows - 1));
}

template <int D>
static cudaError_t esjd_dim(const float* trace, int layout, int64_t rows, int64_t chains, float* out, cudaStream_t st)
{
    if (layout == GLABC_TRACE_TIME_MAJOR) {
        const int block = 128;
        k_esjd_time_major<D><<<static_cast<unsigned>((chains + block - 1) / block), block, 0, st>>>(trace, rows, chains, out);
    } else {
        const int block = 128;  // 4 chains per block
        k_esjd_chain_major<D><<<static_cast<unsigned>((chains * 32 + block - 1) / block), block, 0, st>>>(trace, rows, chains, out);
    }
    return cudaGetLastError();
}

cudaError_t launch_esjd(const float* trace, int layout, int64_t rows, int64_t chains, int dim, float* out, cudaStream_t st)
{
    return with_dim(dim, [&](auto d) {
        if constexpr (d == 4) return cudaErrorInvalidValue;   // esjd_from_gram: D <= 3
        else return esjd_dim<d>(trace, layout, rows, chains, out, st);
    });
}

// Summary of a shard's per-chain statistics in ONE launch (sharding.summarize): out[6 + 2d] float64 +=
// {chains, steps, global steps, accepted local, accepted global, sum of per-chain ESJD (ESJD.py:21-24 from the Gram
// accumulators), sum theta[d], sum theta^2[d]} — the additive vector the ranks all-reduce.
template <int D>
__global__ void __launch_bounds__(256) k_summarize(const float* __restrict__ stats, int64_t chains, double* __restrict__ out)
{
    constexpr int NS = 4 + 2 * D + D * (D + 1) / 2, NO = 6 + 2 * D;
    double acc[NO];
#pragma unroll
    for (int k = 0; k < NO; ++k) acc[k] = 0.0;
    for (int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < chains; c += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const float* st = stats + c * NS;
        const double n = fmax(static_cast<double>(st[GLABC_STAT_STEPS]), 1.0);
        acc[0] += 1.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[1 + k] += static_cast<double>(st[k]);
        // det(G / n)^(1/D), G the symmetric Gram matrix (upper triangle, row-major), by elimination in float64
        double g[D][D];
        int q = 0;
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = i; j < D; ++j, ++q) g[i][j] = g[j][i] = static_cast<double>(st[GLABC_STAT_SUM + 2 * D + q]) / n;
        double det = 1.0;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            const double piv = g[i][i];
            det *= piv;
            if (piv != 0.0) {
#pragma unroll
                for (int r = i + 1; r < D; ++r) {
                    const double f = g[r][i] / piv;
#pragma unroll
                    for (int cc = i + 1; cc < D; ++cc) g[r][cc] -= f * g[i][cc];
                }
            }
        }
        acc[5] += det > 0.0 ? pow(det, 1.0 / D) : 0.0;
#pragma unroll
        for (int k = 0; k < 2 * D; ++k) acc[6 + k] += static_cast<double>(st[GLABC_STAT_SUM + k]);
    }
    __shared__ double red[8][NO];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NO; ++k) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            int lo = __double2loint(v), hi = __double2hiint(v);
            lo = __shfl_xor_sync(0xffffffffu, lo, o);
            hi = __shfl_xor_sync(0xffffffffu, hi, o);
            v += __hiloint2double(hi, lo);
        }
        if (lane == 0) red[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < NO) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        atomicAdd(out + threadIdx.x, v);
    }
}

cudaError_t launch_summarize(const float* stats, int64_t chains, int dim, double* out, cudaStream_t st)
{
    if (chains <= 0) return cudaSuccess;
    int64_t blocks = (chains + 255) / 256;
    if (blocks > 296) blocks = 296;
    const unsigned g = static_cast<unsigned>(blocks);
    return with_dim(dim, [&](auto d) {
        k_summarize<d><<<g, 256, 0, st>>>(stats, chains, out);
        return cudaGetLastError();
    });
}

__global__ void k_philox_kat(const uint32_t* __restrict__ ctr, const uint32_t* __restrict__ key, int64_t n,
                             uint32_t* __restrict__ out)
{
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const RoundKeys rk = expand_key(make_uint2(key[2 * i], key[2 * i + 1]));
    const uint4 r = philox4x32_10(make_uint4(ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3]), rk);
    out[4 * i] = r.x;
    out[4 * i + 1] = r.y;
    out[4 * i + 2] = r.z;
    out[4 * i + 3] = r.w;
}

cudaError_t launch_philox_kat(const uint32_t* ctr, const uint32_t* key, int64_t n, uint32_t* out, cudaStream_t st)
{
    if (n <= 0) return cudaSuccess;
    k_philox_kat<<<static_cast<unsigned>((n + 127) / 128), 128, 0, st>>>(ctr, key, n, out);
    return cudaGetLastError();
}

}  // namespace glabc
