// Host launchers of the KernelDensity kernels (kde.cuh), dispatched over the feature dimension.
#include "kde.cuh"
#include "launch.cuh"

namespace glabc {

cudaError_t launch_kde_fit(const float* X, const float* w, const int32_t* n, const int32_t* active, int64_t sets, int64_t cap,
                           int dim, int rule, float* weights_out, float* lw_out, float* bw_out, cudaStream_t st)
{
    if (sets <= 0) return cudaSuccess;
    const unsigned grid = static_cast<unsigned>(sets);
    return with_dim(dim, [&](auto d) {
        k_kde_fit<d><<<grid, 256, 0, st>>>(X, w, n, active, cap, rule, weights_out, lw_out, bw_out);
        return cudaGetLastError();
    });
}

// Queries per thread for (sets, m): more queries per thread amortise the shared-memory broadcast of a point pair
// (5 -> 4.5 -> 4.25 issue slots per pair), as long as the query tiles alone still give every SM a few CTAs.
// Without the point split (STRICT, or no scratch: the AGLMCMC-internal launches) the query tiles alone must fill the machine.
static int kde_queries_per_thread(int64_t sets, int64_t m, bool strict, bool can_split)
{
    const int64_t ctas1 = sets * ((m + kKdeThreads - 1) / kKdeThreads);
    const int64_t need = can_split && !strict ? 148 : 8 * 148;
    if (!strict && ctas1 >= need * 4) return 4;
    return ctas1 >= need * 2 ? 2 : 1;
}

// A small query batch against a big point set (the stand-alone estimator: 1e5 x 1e5) gives too few CTAs to hide the
// MUFU / shared-memory latency; the point tiles are then dealt to `ksplit` CTAs per query tile (FAST arithmetic only:
// with the fixed shift the partial sums simply add).  Target: ~12 CTAs of 4 warps per SM.
int kde_logprob_split(int64_t sets, int64_t m, int64_t cap)
{
    const int q = kde_queries_per_thread(sets, m, false, true);
    const int64_t ctas = sets * ((m + kKdeThreads * q - 1) / (kKdeThreads * q));
    const int64_t tiles = (cap + kKdeTile - 1) / kKdeTile;
    if (ctas <= 0 || ctas >= 12 * 148 || tiles < 4) return 1;
    int64_t k = (12 * 148 + ctas - 1) / ctas;
    if (k > tiles / 2) k = tiles / 2;
    if (k > 64) k = 64;
    return k < 1 ? 1 : static_cast<int>(k);
}

template <int D>
static cudaError_t logprob_dim(const KdeSets& S, const float* lw, const float* x, int64_t m, float* out, bool strict, cudaStream_t st,
                               int ksplit, float* partial)
{
    const int q = kde_queries_per_thread(S.sets, m, strict, partial != nullptr && ksplit >= 1);
    if (strict || partial == nullptr || ksplit < 1) ksplit = 1;
    const int64_t per_cta = static_cast<int64_t>(kKdeThreads) * q;
    const int64_t qtiles = (m + per_cta - 1) / per_cta;
    const int64_t grid = S.sets * qtiles * ksplit;
    if (grid <= 0) return cudaSuccess;
    if (grid > 0x7fffffffll) return cudaErrorInvalidValue;
    const unsigned g = static_cast<unsigned>(grid);
    if (strict) {
        if (q == 2) k_kde_logprob<D, 2, true><<<g, kKdeThreads, 0, st>>>(S, lw, x, m, qtiles, out);
        else k_kde_logprob<D, 1, true><<<g, kKdeThreads, 0, st>>>(S, lw, x, m, qtiles, out);
    } else {
        if (q == 4) k_kde_logprob<D, 4, false><<<g, kKdeThreads, 0, st>>>(S, lw, x, m, qtiles, out, ksplit, partial);
        else if (q == 2) k_kde_logprob<D, 2, false><<<g, kKdeThreads, 0, st>>>(S, lw, x, m, qtiles, out, ksplit, partial);
        else k_kde_logprob<D, 1, false><<<g, kKdeThreads, 0, st>>>(S, lw, x, m, qtiles, out, ksplit, partial);
        if (ksplit > 1) {
            const int64_t tot = S.sets * m;
            k_kde_logprob_finish<D><<<static_cast<unsigned>((tot + 255) / 256), 256, 0, st>>>(S, lw, x, m, ksplit, partial, out);
        }
    }
    return cudaGetLastError();
}

cudaError_t launch_kde_logprob(const KdeSets& S, const float* lw, int dim, const float* x, int64_t m, float* out, bool strict,
                               cudaStream_t st, int ksplit, float* partial)
{
    return with_dim(dim, [&](auto d) { return logprob_dim<d>(S, lw, x, m, out, strict, st, ksplit, partial); });
}

cudaError_t launch_kde_cdf(const float* weights, const int32_t* n, const int32_t* active, int64_t sets, int64_t cap, double* cdf,
                           cudaStream_t st)
{
    if (sets <= 0) return cudaSuccess;
    k_kde_cdf<<<static_cast<unsigned>(sets), 256, 0, st>>>(weights, n, active, cap, cdf);
    return cudaGetLastError();
}

cudaError_t launch_kde_sample(const KdeSets& S, int dim, const double* cdf, int64_t m, const RoundKeys& rk, uint64_t chain_id_base,
                              const int32_t* round_dev, const int32_t* idx_tape, const float* noise_tape, int64_t tape_set_stride,
                              int64_t tape_set_stride_noise, int64_t tape_q_stride, int64_t tape_round_stride_idx,
                              int64_t tape_round_stride_noise, int max_round, float* out, cudaStream_t st)
{
    const int64_t total = S.sets * m;
    if (total <= 0) return cudaSuccess;
    const int64_t grid = (total + 255) / 256;
    if (grid > 0x7fffffffll) return cudaErrorInvalidValue;
    const unsigned g = static_cast<unsigned>(grid);
    return with_dim(dim, [&](auto d) {
        k_kde_sample<d><<<g, 256, 0, st>>>(S, cdf, m, rk, chain_id_base, round_dev, idx_tape, noise_tape, tape_set_stride,
                                           tape_set_stride_noise, tape_q_stride, tape_round_stride_idx, tape_round_stride_noise, max_round, out);
        return cudaGetLastError();
    });
}

}  // namespace glabc
