// Orchestration of K6 (AGLMCMC): step / adapt rounds on one stream, dispatched over theta_dim.
#include "step_aglmcmc.cuh"

namespace glabc {

template <int D>
static cudaError_t run_aglmcmc(const AgConsts& K, const DistConsts& prior, const AgWorkspace& W, const AgTapes& T, const RunParams& R,
                               int init, int kde_rule, bool strict, bool replay, int layout, int block, cudaStream_t st)
{
    const bool gprior = generic_prior(prior);
    if (gprior && (strict || replay)) return cudaErrorInvalidValue;
    const int64_t C = W.C, B = W.B;
    const unsigned g_chain = static_cast<unsigned>((C + 255) / 256);
    const int64_t cb = (C * B + 255) / 256;
    if (cb > 0x7fffffffll) return cudaErrorInvalidValue;
    const unsigned g_cb = static_cast<unsigned>(cb);
    const unsigned g_step = static_cast<unsigned>((C + block - 1) / block);
    cudaError_t e;
    if (init) {
        k_ag_reset<<<g_chain, 256, 0, st>>>(W, R.first_step);
        if (replay) k_ag_block<D, true, true><<<g_cb, 256, 0, st>>>(K, R, W, T, prior);
        else k_ag_block<D, true, false><<<g_cb, 256, 0, st>>>(K, R, W, T, prior);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    if (R.write_row0 && layout != GLABC_TRACE_NONE) k_ag_row0<D><<<g_chain, 256, 0, st>>>(R, C, layout);
    const int64_t n_steps = static_cast<int64_t>(R.last_step) - R.first_step + 1;
    const int64_t rounds = (n_steps > 0 ? n_steps : 0) / K.S + 2;
    KdeSets S{W.kde_X, W.kde_wn, W.kde_bw, W.kde_n, W.pending, C, B};
    for (int64_t r = 0; r < rounds; ++r) {
        if (gprior) {
            k_ag_step<D, false, false, false, true><<<g_step, block, 0, st>>>(K, R, W, layout, prior);
        } else if (strict) {
            if (replay) k_ag_step<D, true, true, false, false><<<g_step, block, 0, st>>>(K, R, W, layout, prior);
            else k_ag_step<D, true, false, false, false><<<g_step, block, 0, st>>>(K, R, W, layout, prior);
        } else {
            if (replay) k_ag_step<D, false, true, false, false><<<g_step, block, 0, st>>>(K, R, W, layout, prior);
            else k_ag_step<D, false, false, false, false><<<g_step, block, 0, st>>>(K, R, W, layout, prior);
        }
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if (r == rounds - 1) break;
        // ---- adaptation of the chains that paused (AGLMCMC.py:170-249); every kernel skips the others ----
        k_ag_adapt<D><<<static_cast<unsigned>(C), 256, 0, st>>>(K, W, prior);
        if ((e = launch_kde_fit(W.kde_X, W.kde_w, W.kde_n, W.pending, C, B, D, kde_rule, W.kde_wn, W.kde_lw, W.kde_bw, st)) != cudaSuccess)
            return e;
        if (!replay && (e = launch_kde_cdf(W.kde_wn, W.kde_n, W.pending, C, B, W.cdf, st)) != cudaSuccess) return e;
        const uint64_t base = (static_cast<uint64_t>(R.chain_hi0) << 32) | R.chain_lo0;
        if (replay) {
            e = launch_kde_sample(S, D, W.cdf, 4 * B, R.rk, base, W.n_adapt, T.ad_idx, T.ad_noise, 1, 1, C, 4 * B * C, 4 * B * D * C,
                                  T.tape_rounds - 1, W.smp, st);
            if (e != cudaSuccess) return e;
            k_ag_filter<D><<<static_cast<unsigned>(C), 256, 0, st>>>(K, W, prior);
        } else {
            k_ag_sample_filter<D><<<static_cast<unsigned>(C), 256, 0, st>>>(K, W, S, R.rk, base, prior);
        }
        if ((e = launch_kde_logprob(S, W.kde_lw, D, W.blk_theta, B, W.blk_lq, strict, st)) != cudaSuccess) return e;
        if (replay) k_ag_block<D, false, true><<<g_cb, 256, 0, st>>>(K, R, W, T, prior);
        else k_ag_block<D, false, false><<<g_cb, 256, 0, st>>>(K, R, W, T, prior);
        k_ag_commit<D><<<g_chain, 256, 0, st>>>(W, T);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t launch_block_isir(const AgConsts& K, const DistConsts& prior, const AgWorkspace& W, const RunParams& R, int dim, bool strict,
                              int layout, int block, cudaStream_t st)
{
    return with_dim(dim, [&](auto d) {
        const bool gprior = generic_prior(prior);
        if (gprior && strict) return cudaErrorInvalidValue;
        const unsigned g_step = static_cast<unsigned>((W.C + block - 1) / block);
        if (R.write_row0 && layout != GLABC_TRACE_NONE) k_ag_row0<d><<<static_cast<unsigned>((W.C + 255) / 256), 256, 0, st>>>(R, W.C, layout);
        if (gprior) k_ag_step<d, false, false, true, true><<<g_step, block, 0, st>>>(K, R, W, layout, prior);
        else if (strict) k_ag_step<d, true, false, true, false><<<g_step, block, 0, st>>>(K, R, W, layout, prior);
        else k_ag_step<d, false, false, true, false><<<g_step, block, 0, st>>>(K, R, W, layout, prior);
        return cudaGetLastError();
    });
}

cudaError_t launch_block_weights(const AgConsts& K, const DistConsts& prior, const AgWorkspace& W, const RunParams& R, int dim,
                                 uint32_t round, cudaStream_t st)
{
    const int64_t cb = (W.C * W.B + 255) / 256;
    if (cb > 0x7fffffffll) return cudaErrorInvalidValue;
    const unsigned g = static_cast<unsigned>(cb);
    return with_dim(dim, [&](auto d) {
        k_blk_weights<d><<<g, 256, 0, st>>>(K, R, W, round, prior);
        return cudaGetLastError();
    });
}

cudaError_t launch_aglmcmc(const AgConsts& K, const DistConsts& prior, const AgWorkspace& W, const AgTapes& T, const RunParams& R,
                           int dim, int init, int kde_rule, bool strict, bool replay, int layout, int block, cudaStream_t st)
{
    return with_dim(dim, [&](auto d) { return run_aglmcmc<d>(K, prior, W, T, R, init, kde_rule, strict, replay, layout, block, st); });
}

}  // namespace glabc
