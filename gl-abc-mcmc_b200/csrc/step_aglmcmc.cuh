// K6 — AGLMCMC (reference AGLMCMC.py:44-288, SURVEY.md A.5): iSIR against a per-chain block of
// B = batch_size * step_size pre-generated importance candidates; after step_size global moves the chain
// adapts — eps-hat quantile update, weighted KernelDensity refit on the block, new block from the KDE.
//
//   k_ag_step     one thread = one chain, runs until the chain has done its iterations or reaches an
//                 adaptation (chains pause individually: with gf < 1 they adapt at different iterations).
//                 The proposal log-density of the current state is cached (the reference re-evaluates
//                 KDE.log_prob(theta_old), a 1 x n pass, every global move — it only changes when the state
//                 or the KDE does); a stale cache is refreshed warp-cooperatively (32 lanes split the n points).
//   k_ag_adapt    one CTA per pausing chain: bitonic sort of the block's discrepancies -> torch.quantile,
//                 training weights, order-preserving compaction of the positive ones
//   kde.cuh       fit / cdf / sample / log_prob batched over the pausing chains
//   k_ag_filter   first B prior-valid KDE samples (order-preserving), k_ag_block simulator + weights,
//   k_ag_commit   per-chain counters
// All per-chain buffers are chain-major ([C][B]...): a chain's block is contiguous for the CTA-per-chain
// kernels, and the step kernel touches one 32-byte sector per array per global move.
#pragma once
#include "kde.cuh"
#include "launch.cuh"
#include "sampler_common.cuh"
#include "step_generic.cuh"

namespace glabc {

struct AgWorkspace {
    float *blk_theta, *blk_x, *blk_w, *blk_lq, *blk_dis;  // [C][B][D], [C][B][D], [C][B] x3
    float *kde_X, *kde_w, *kde_wn, *kde_lw, *kde_bw;      // [C][B][D], [C][B] x3, [C][D]
    float* smp;                                           // [C][4B][D] KDE samples
    double* cdf;                                          // [C][B]
    int32_t *kde_n, *kk, *n_adapt, *pending, *lq_valid;   // [C]
    uint32_t* next_step;                                  // [C] loop index of the next iteration to perform
    float *hat_eps, *lq_cur;                              // [C]
    int64_t C;
    int32_t B;
};

struct AgConsts {
    ModelConsts model;
    GaussConsts lp, ip;
    int32_t S;            // step_size
    float alpha, hat_eps_T;
    float log_prior_floor;  // float32(log(1e-10)), AGLMCMC.py:223-224
    int32_t ip_generic;     // Initial_ISIR_prop is a Uniform / Gamma / GaussianMixture (`ipg`; FAST arithmetic, native RNG), else `ip`
    DistConsts ipg;
};

struct AgTapes {
    const float *init_p, *init_s, *ad_noise, *ad_sim;
    const int32_t* ad_idx;
    float *ad_rec, *ad_blk, *init_w;
    int32_t tape_rounds, dump_rounds;
};

// log N(dis; 0, eps) the way Mixture.py:47-53 evaluates it for a float32 eps
__device__ __forceinline__ float log_kernel_dis_eps(float c_kern, float dis, float ls, float scale)
{
    const float r = __fdiv_rn(__fsub_rn(dis, 0.0f), scale);
    return __fsub_rn(c_kern, __fadd_rn(ls, __fmul_rn(0.5f, __fmul_rn(r, r))));
}

template <int D>
__device__ __forceinline__ float model_discrepancy(const ModelConsts& m, const float (&y)[D])
{
    float t[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        const float dy = __fsub_rn(y[i], m.y_obs[i]);
        t[i] = __fmul_rn(dy, dy);
    }
    return __fsqrt_rn(torch_sum_strict<D>(t));
}

// ---------------------------------------------------------------------------------------------
// block construction: INIT draws theta0 / log q0 from Initial_ISIR_prop (AGLMCMC.py:84-91); both variants
// simulate, take the discrepancy and form the weights (:94-112 / :232-249).  One thread per (chain, b).
// ---------------------------------------------------------------------------------------------
template <int D, bool INIT, bool REPLAY>
__global__ void __launch_bounds__(256) k_ag_block(const __grid_constant__ AgConsts K, const __grid_constant__ RunParams R,
                                                  AgWorkspace W, AgTapes T, const __grid_constant__ DistConsts prior)
{
    const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (g >= W.C * W.B) return;
    const int64_t c = g / W.B;
    const int b = static_cast<int>(g - c * W.B);
    if (!INIT && W.pending[c] == 0) return;
    const int64_t C = W.C;
    const int round = INIT ? 0 : W.n_adapt[c];
    const uint64_t gid = (static_cast<uint64_t>(R.chain_hi0) << 32 | R.chain_lo0) + static_cast<uint64_t>(c);
    const Stream st{static_cast<uint32_t>(gid), static_cast<uint32_t>(gid >> 32)};
    float th[D], eps_s[D], lq;
    if constexpr (INIT) {
        float eps_p[D];
        if constexpr (REPLAY) {
#pragma unroll
            for (int k = 0; k < D; ++k) {
                eps_p[k] = T.init_p[static_cast<int64_t>(b * D + k) * C + c];
                eps_s[k] = T.init_s[static_cast<int64_t>(b * D + k) * C + c];
            }
        } else {
            constexpr int G = (2 * D + 3) / 4;
            float z[G * 4];
#pragma unroll
            for (int q = 0; q < G; ++q) {
                const uint4 w = st.block(R.rk, 0u, kSlotInit + static_cast<uint32_t>(b * G + q));
                box_muller(w.x, w.y, z[4 * q], z[4 * q + 1]);
                box_muller(w.z, w.w, z[4 * q + 2], z[4 * q + 3]);
            }
#pragma unroll
            for (int k = 0; k < D; ++k) {
                eps_p[k] = z[k];
                eps_s[k] = z[D + k];
            }
        }
        if (!REPLAY && K.ip_generic) {   // candidate b's draw and its simulator normals from one word stream (as k_isir_generic's)
            WordStream ws(R.rk, st, 0u, kSlotGeneric + 64u * static_cast<uint32_t>(b));
            lq = dist_forward<D>(K.ipg, ws, th);
#pragma unroll
            for (int k = 0; k < D; ++k) eps_s[k] = ws.normal();
        } else {
            lq = gauss_forward<D, true>(K.ip, eps_p, th);
        }
#pragma unroll
        for (int k = 0; k < D; ++k) W.blk_theta[(c * W.B + b) * D + k] = th[k];
        W.blk_lq[c * W.B + b] = lq;
    } else {
#pragma unroll
        for (int k = 0; k < D; ++k) th[k] = W.blk_theta[(c * W.B + b) * D + k];
        lq = W.blk_lq[c * W.B + b];
        if constexpr (REPLAY) {
            const int rr = min(round, T.tape_rounds - 1);
#pragma unroll
            for (int k = 0; k < D; ++k)
                eps_s[k] = T.ad_sim[(static_cast<int64_t>(rr) * W.B * D + static_cast<int64_t>(b) * D + k) * C + c];
        } else {
            const uint4 w = st.block(R.rk, static_cast<uint32_t>(round), kSlotAdSim + static_cast<uint32_t>(b));
            float z[4];
            box_muller(w.x, w.y, z[0], z[1]);
            box_muller(w.z, w.w, z[2], z[3]);
#pragma unroll
            for (int k = 0; k < D; ++k) eps_s[k] = z[k];
        }
    }
    float x[D];
    model_simulate<D, true>(K.model, th, eps_s, x);
    const float dis = model_discrepancy<D>(K.model, x);
    const float like = log_kernel_dis_eps(K.model.c_kern, dis, K.model.eps_log_scale, K.model.eps_scale);
    float w = expf(__fsub_rn(__fadd_rn(prior_log_prob_rt<D>(K.model, prior, th), like), lq));
    if (INIT && w != w) w = 0.0f;  // AGLMCMC.py:110-112; the regenerated blocks keep NaN weights (:248-249)
#pragma unroll
    for (int k = 0; k < D; ++k) W.blk_x[(c * W.B + b) * D + k] = x[k];
    W.blk_dis[c * W.B + b] = dis;
    W.blk_w[c * W.B + b] = w;
    if (INIT) {
        if (T.init_w != nullptr) T.init_w[static_cast<int64_t>(b) * C + c] = w;
    } else if (T.ad_blk != nullptr && round < T.dump_rounds) {
        float* o = T.ad_blk + ((static_cast<int64_t>(round) * W.B + b) * (D + 3)) * C + c;
#pragma unroll
        for (int k = 0; k < D; ++k) o[static_cast<int64_t>(k) * C] = th[k];
        o[static_cast<int64_t>(D) * C] = lq;
        o[static_cast<int64_t>(D + 1) * C] = w;
        o[static_cast<int64_t>(D + 2) * C] = dis;
    }
}

static __global__ void __launch_bounds__(256) k_ag_reset(AgWorkspace W, uint32_t first_step)
{
    const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= W.C) return;
    W.kk[c] = 0;
    W.n_adapt[c] = 0;
    W.pending[c] = 0;
    W.lq_valid[c] = 0;
    W.kde_n[c] = 0;
    W.next_step[c] = first_step;
    W.hat_eps[c] = 1000000.0f;  // AGLMCMC.py:119
    W.lq_cur[c] = 0.0f;
}

template <int D>
__global__ void __launch_bounds__(256) k_ag_commit(AgWorkspace W, AgTapes T)
{
    const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= W.C || W.pending[c] == 0) return;
    const int round = W.n_adapt[c];
    if (T.ad_rec != nullptr && round < T.dump_rounds) {
        float* o = T.ad_rec + static_cast<int64_t>(round) * GLABC_AG_REC_SLOTS * W.C + c;
        o[0] = W.hat_eps[c];
        o[W.C] = static_cast<float>(W.kde_n[c]);
#pragma unroll
        for (int k = 0; k < D; ++k) o[static_cast<int64_t>(2 + k) * W.C] = W.kde_bw[c * D + k];
    }
    W.n_adapt[c] = round + 1;  // num_train, AGLMCMC.py:217
    W.pending[c] = 0;
    W.kk[c] = 0;               // :171
    W.lq_valid[c] = 0;         // the proposal changed
}

// ---------------------------------------------------------------------------------------------
// adaptation, AGLMCMC.py:174-211: one CTA per pausing chain
// ---------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256) k_ag_adapt(const __grid_constant__ AgConsts K, AgWorkspace W, const __grid_constant__ DistConsts prior)
{
    __shared__ float sorted[GLABC_AG_MAX_BLOCK];
    __shared__ int cnt[256];
    __shared__ double red[8];
    __shared__ float s_eps;
    const int64_t c = blockIdx.x;
    if (W.pending[c] == 0) return;
    const int B = W.B, tid = threadIdx.x;
    const float* dis = W.blk_dis + c * B;
    float hat_eps = W.hat_eps[c];

    if (hat_eps > K.hat_eps_T) {  // :174
        int np2 = 1;
        while (np2 < B) np2 <<= 1;
        int my_a = 0, my_v = 0;
        for (int j = tid; j < np2; j += 256) {
            float v = INFINITY;
            if (j < B) {
                const float dj = dis[j];
                if (dj < hat_eps) ++my_a;  // :178
                if (dj == dj) {            // :181 (NaNs dropped)
                    v = dj;
                    ++my_v;
                }
            }
            sorted[j] = v;
        }
        const double na = block_sum_f64(static_cast<double>(my_a), red);
        const double nvd = block_sum_f64(static_cast<double>(my_v), red);
        __syncthreads();
        for (int k = 2; k <= np2; k <<= 1)  // bitonic sort, ascending
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < np2; i += 256) {
                    const int l = i ^ j;
                    if (l > i) {
                        const float a = sorted[i], b = sorted[l];
                        const bool up = (i & k) == 0;
                        if ((a > b) == up) {
                            sorted[i] = b;
                            sorted[l] = a;
                        }
                    }
                }
                __syncthreads();
            }
        if (tid == 0) {
            const int nv = static_cast<int>(nvd);
            if (nv > 0) {  // :183-193
                float q = __fdiv_rn(__fmul_rn(K.alpha, static_cast<float>(static_cast<int>(na))), static_cast<float>(nv));
                q = fminf(fmaxf(q, 0.0f), 1.0f);
                // torch.quantile, 'linear': rank = q * (n - 1), lerp between the neighbours
                const float rank = __fmul_rn(q, static_cast<float>(nv - 1));
                const float lo = floorf(rank), fr = __fsub_rn(rank, lo);
                const float a = sorted[static_cast<int>(lo)], b = sorted[static_cast<int>(ceilf(rank))];
                hat_eps = fr < 0.5f ? __fadd_rn(a, __fmul_rn(fr, __fsub_rn(b, a)))
                                    : __fsub_rn(b, __fmul_rn(__fsub_rn(b, a), __fsub_rn(1.0f, fr)));
            }
            if (!(hat_eps > K.hat_eps_T)) hat_eps = K.hat_eps_T;  // torch.max, :196
            s_eps = hat_eps;
        }
        __syncthreads();
        hat_eps = s_eps;
    }
    if (tid == 0) W.hat_eps[c] = hat_eps;

    // training weights exp(prior + log K_epshat(dis) - log q0), :199-201; keep the positive ones in order, :206-208
    const float ls = logf(hat_eps), scale = expf(ls);
    const int per = (B + 255) / 256;
    const int lo = tid * per, hi = min(B, lo + per);
    int mine = 0;
    for (int j = lo; j < hi; ++j) {
        float th[D];
#pragma unroll
        for (int k = 0; k < D; ++k) th[k] = W.blk_theta[(c * B + j) * D + k];
        const float like = log_kernel_dis_eps(K.model.c_kern, dis[j], ls, scale);
        const float tw = expf(__fsub_rn(__fadd_rn(prior_log_prob_rt<D>(K.model, prior, th), like), W.blk_lq[c * B + j]));
        sorted[j] = tw;  // the sort buffer is free again
        mine += tw > 0.0f;
    }
    cnt[tid] = mine;
    __syncthreads();
    int base = 0, total = 0;
    for (int i = 0; i < 256; ++i) {
        if (i < tid) base += cnt[i];
        total += cnt[i];
    }
    double acc = 0.0;
    for (int j = lo; j < hi; ++j) {
        const float tw = sorted[j];
        if (tw > 0.0f) {
#pragma unroll
            for (int k = 0; k < D; ++k) W.kde_X[(c * B + base) * D + k] = W.blk_theta[(c * B + j) * D + k];
            W.kde_w[c * B + base] = tw;
            ++base;
            acc += static_cast<double>(tw);
        }
    }
    const float sw = static_cast<float>(block_sum_f64(acc, red));
    __syncthreads();
    for (int j = tid; j < total; j += 256) W.kde_w[c * B + j] = __fdiv_rn(W.kde_w[c * B + j], sw);  // :211
    if (tid == 0) W.kde_n[c] = total;
}

// Theta_prop0 = the first B of the 4B KDE samples whose prior log-density exceeds log(1e-10), AGLMCMC.py:220-226 (a draw
// outside the support of a Uniform / Gamma prior has log prior -inf and never enters the block)
template <int D>
__global__ void __launch_bounds__(256) k_ag_filter(const __grid_constant__ AgConsts K, AgWorkspace W, const __grid_constant__ DistConsts prior)
{
    __shared__ int cnt[256];
    const int64_t c = blockIdx.x;
    if (W.pending[c] == 0) return;
    const int B = W.B, M = 4 * W.B, tid = threadIdx.x;
    const float* smp = W.smp + c * M * D;
    const int per = (M + 255) / 256;
    const int lo = tid * per, hi = min(M, lo + per);
    int mine = 0;
    for (int j = lo; j < hi; ++j) {
        float th[D];
#pragma unroll
        for (int k = 0; k < D; ++k) th[k] = smp[static_cast<int64_t>(j) * D + k];
        mine += prior_log_prob_rt<D>(K.model, prior, th) > K.log_prior_floor;
    }
    cnt[tid] = mine;
    __syncthreads();
    int base = 0;
    for (int i = 0; i < tid; ++i) base += cnt[i];
    for (int j = lo; j < hi && base < B; ++j) {
        float th[D];
#pragma unroll
        for (int k = 0; k < D; ++k) th[k] = smp[static_cast<int64_t>(j) * D + k];
        if (prior_log_prob_rt<D>(K.model, prior, th) > K.log_prior_floor) {
#pragma unroll
            for (int k = 0; k < D; ++k) W.blk_theta[(c * B + base) * D + k] = th[k];
            ++base;
        }
    }
}

// Native RNG: KDE.sample(4B) + the prior filter fused (AGLMCMC.py:219-226).  Draw q is a pure function of (chain, round, q),
// so the CTA generates draws in order, 256 at a time, and stops as soon as B valid ones are placed — with a prior that almost
// never rejects that is B draws instead of 4B, and the [C][4B][D] sample buffer is never touched.  Same block as
// k_kde_sample + k_ag_filter produce (tested through the native-mode oracle comparison).
template <int D>
__global__ void __launch_bounds__(256) k_ag_sample_filter(const __grid_constant__ AgConsts K, AgWorkspace W, KdeSets S, RoundKeys rk,
                                                          uint64_t chain_id_base, const __grid_constant__ DistConsts prior)
{
    __shared__ int wsum[8];
    const int64_t c = blockIdx.x;
    if (W.pending[c] == 0) return;
    const int B = W.B, M = 4 * W.B, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = W.kde_n[c], round = W.n_adapt[c];
    int have = 0;
    for (int start = 0; start < M && have < B; start += 256) {
        const int j = start + tid;
        float th[D];
        bool valid = false;
        if (j < M) {
            kde_draw_native<D>(S, W.cdf, c, n, round, j, rk, chain_id_base, th);
            valid = prior_log_prob_rt<D>(K.model, prior, th) > K.log_prior_floor;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, valid);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int before = __popc(bal & ((1u << lane) - 1u)), total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            before += w < warp ? wsum[w] : 0;
            total += wsum[w];
        }
        const int pos = have + before;
        if (valid && pos < B) {
#pragma unroll
            for (int k = 0; k < D; ++k) W.blk_theta[(c * B + pos) * D + k] = th[k];
        }
        have += total;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// the chain step, AGLMCMC.py:124-168 (global) / :251-271 (local)
// ---------------------------------------------------------------------------------------------
// EXT = the importance proposal lives outside this kernel (GLMCMC-NFs: the shared RealNVP flow): the cached
// proposal log-density of a state that changed is not recomputed here — the chain pauses (pending bit 1) and the
// host refreshes it in one batched tensor-core log_prob launch (flow.cuh) before relaunching.
// GPRIOR: the model's prior is `prior` (FAST arithmetic, native RNG; step_generic.cuh prior_log_prob).
template <int D, bool STRICT, bool REPLAY, bool EXT, bool GPRIOR>
__global__ void __launch_bounds__(128) k_ag_step(const __grid_constant__ AgConsts K, const __grid_constant__ RunParams R,
                                                 AgWorkspace W, int layout, const __grid_constant__ DistConsts prior)
{
    static_assert(!GPRIOR || (!STRICT && !REPLAY), "a general prior runs FAST arithmetic with the native RNG");
    const int lane = threadIdx.x & 31;
    const int64_t chain = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool in_range = chain < W.C;
    const int64_t c = in_range ? chain : W.C - 1;
    const int64_t C = W.C;
    const int B = W.B, NK = R.n_candidates;
    constexpr int kGroups = (2 * D + 3) / 4;
    constexpr int kSlots = 2 + 2 * D;

    float theta[D], y[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        theta[k] = R.theta[c * D + k];
        y[k] = R.y[c * D + k];
    }
    int kk = W.kk[c];
    const int n_adapt = EXT ? 1 : W.n_adapt[c];
    uint32_t i = W.next_step[c];
    float lq_cur = W.lq_cur[c];
    bool lq_valid = W.lq_valid[c] != 0;
    const int kn = EXT ? 0 : W.kde_n[c];
    bool pend_lq = false;
    bool running = in_range && i <= R.last_step && R.last_step >= R.first_step && kk < K.S;
    ChainStats<D> stats;
    uint32_t done = 0;
    const Stream stream = chain_stream(R, static_cast<int32_t>(c));

    while (__any_sync(0xffffffffu, running)) {
        bool is_global = false;
        float u_a = 0.0f, eps_p[D], eps_s[D];
        double u64 = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) eps_p[k] = eps_s[k] = 0.0f;
        const int64_t srow = static_cast<int64_t>(i) - R.first_step;
        if (running) {
            if constexpr (REPLAY) {
                const float* tp = R.tape32 + (srow * kSlots) * C + c;
                is_global = __ldg(tp) < R.gf;  // AGLMCMC.py:125-126
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    eps_p[k] = __ldg(tp + static_cast<int64_t>(1 + k) * C);
                    eps_s[k] = __ldg(tp + static_cast<int64_t>(1 + D + k) * C);
                }
                u_a = __ldg(tp + static_cast<int64_t>(1 + 2 * D) * C);
                u64 = R.tape64[srow * C + c];
            } else {
                const uint4 w0 = stream.block(R.rk, i, kSlotStep);
                is_global = (step_block_ub(w0) < R.gf_thr_hi) || R.gf_all_global;
                float z[kGroups * 4];
                box_muller(w0.x, w0.y, z[0], z[1]);
                box_muller(w0.z, w0.w, z[2], z[3]);
#pragma unroll
                for (int g = 1; g < kGroups; ++g) {
                    const uint4 w = stream.block(R.rk, i, kSlotNormal + g - 1);
                    box_muller(w.x, w.y, z[4 * g], z[4 * g + 1]);
                    box_muller(w.z, w.w, z[4 * g + 2], z[4 * g + 3]);
                }
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    eps_p[k] = z[k];
                    eps_s[k] = z[D + k];
                }
                u_a = __uint2float_rn(step_block_ua(w0)) * 0x1p-24f;
                // a global move does not use the block's normals: their bits make the 53-bit resampling uniform
                const uint64_t m53 = (static_cast<uint64_t>(w0.x >> 8) << 29) | (static_cast<uint64_t>(w0.z >> 8) << 5) |
                                     static_cast<uint64_t>(w0.y >> 27);
                u64 = static_cast<double>(m53) * 0x1p-53;
            }
        }
        if constexpr (EXT) {
            if (running && is_global && !lq_valid) {  // pause before the move: its draws are counter-based, so it replays
                running = false;
                pend_lq = true;
            }
        }
        // ---- refresh stale KDE log-densities of current states, one chain at a time, 32 lanes per chain ----
        unsigned need = EXT ? 0u : __ballot_sync(0xffffffffu, running && is_global && n_adapt > 0 && !lq_valid);
        while (need) {
            const int src = __ffs(need) - 1;
            need &= need - 1;
            const int64_t cs = chain - lane + src;
            float xs[D];
#pragma unroll
            for (int k = 0; k < D; ++k) xs[k] = __shfl_sync(0xffffffffu, theta[k], src);
            const int ns = __shfl_sync(0xffffffffu, kn, src);
            const KdeConst<D> kc = kde_const<D>(W.kde_bw + cs * D);
            const float part = kde_log_prob_scan<D>(kc, xs, W.kde_X + cs * B * D, W.kde_lw + cs * B, ns, lane, 32);
            const float lq = warp_logsumexp(part);
            if (lane == src) {
                lq_cur = lq;
                lq_valid = true;
            }
        }
        if (running) {
            float prev[D];
#pragma unroll
            for (int k = 0; k < D; ++k) prev[k] = theta[k];
            bool moved = false;
            int ind = -1;
            float d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
            const float prior_old = prior_log_prob<D, STRICT, GPRIOR>(K.model, prior, theta);
            const float kern_old = model_log_kernel<D, STRICT>(K.model, y);
            if (is_global) {
                // :137-149: weight of the current state under the current importance proposal
                const float lq_old = n_adapt == 0 ? (K.ip_generic ? dist_log_prob<D>(K.ipg, theta) : gauss_log_prob<D, STRICT>(K.ip, theta)) : lq_cur;
                const float lw = STRICT ? __fsub_rn(__fadd_rn(prior_old, kern_old), lq_old) : (prior_old + kern_old) - lq_old;
                float w_old;
                if constexpr (STRICT) {
                    w_old = expf(lw);
                } else {
                    asm("ex2.approx.f32 %0, %1;" : "=f"(w_old) : "f"(lw * 1.4426950408889634f));
                }
                const float* bw = W.blk_w + c * B + kk * NK;
                const int n = NK + 1;
                float Ssum;
                double run = 0.0;
                if constexpr (STRICT) {
                    // torch.sum over the K+1 weights in ATen's order (SURVEY.md B-3), element 0 = current state
                    if (n >= 16) {
                        float acc = 0.0f;
                        for (int j = 16; j < n; ++j) acc = __fadd_rn(acc, bw[j - 1]);
                        acc = __fadd_rn(acc, w_old);
                        for (int j = 1; j < 16; ++j) acc = __fadd_rn(acc, bw[j - 1]);
                        Ssum = acc;
                    } else {
                        float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
                        const int body = n & ~3;
                        for (int j = 0; j < n; ++j) {
                            const float v = j == 0 ? w_old : bw[j - 1];
                            const int slot = j < body ? (j & 3) : 0;
                            p0 = __fadd_rn(p0, slot == 0 ? v : 0.0f);
                            p1 = __fadd_rn(p1, slot == 1 ? v : 0.0f);
                            p2 = __fadd_rn(p2, slot == 2 ? v : 0.0f);
                            p3 = __fadd_rn(p3, slot == 3 ? v : 0.0f);
                        }
                        Ssum = __fadd_rn(__fadd_rn(__fadd_rn(p0, p1), p2), p3);
                    }
                    for (int j = 0; j < n; ++j) {  // weight_sampling, AGLMCMC.py:12-27: float64 running sum of float32 quotients
                        run += static_cast<double>(__fdiv_rn(j == 0 ? w_old : bw[j - 1], Ssum));
                        if (ind < 0 && u64 < run) ind = j;
                    }
                } else {
                    Ssum = w_old;
                    for (int j = 0; j < NK; ++j) Ssum += bw[j];
                    const double thr = u64 * static_cast<double>(Ssum);
                    for (int j = 0; j < n; ++j) {
                        run += static_cast<double>(j == 0 ? w_old : bw[j - 1]);
                        if (ind < 0 && thr < run) ind = j;
                    }
                }
                if (ind > 0) {  // :161-163
                    const int64_t o = c * B + kk * NK + ind - 1;
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        theta[k] = W.blk_theta[o * D + k];
                        y[k] = W.blk_x[o * D + k];
                    }
                    lq_cur = W.blk_lq[o];  // KDE.log_prob(theta0[o]) under the same KDE
                    lq_valid = n_adapt > 0;
                }
#pragma unroll
                for (int k = 0; k < D; ++k) moved |= theta[k] != prev[k];
                d1 = lq_old;
                d2 = w_old;
                d3 = Ssum;
                ++kk;  // :166
            } else {
                // local random-walk MH, :251-271
                float z[D], th_l[D], y_l[D];
                (void)gauss_forward<D, STRICT>(K.lp, eps_p, z);
#pragma unroll
                for (int k = 0; k < D; ++k) th_l[k] = STRICT ? __fadd_rn(z[k], theta[k]) : z[k] + theta[k];
                model_simulate<D, STRICT>(K.model, th_l, eps_s, y_l);
                const float prior_l = prior_log_prob<D, STRICT, GPRIOR>(K.model, prior, th_l);
                const float kern_l = model_log_kernel<D, STRICT>(K.model, y_l);
                const float log_acc = STRICT ? __fsub_rn(__fsub_rn(__fadd_rn(prior_l, kern_l), prior_old), kern_old)
                                             : (prior_l + kern_l) - (prior_old + kern_old);
                const float log_w = STRICT ? logf(u_a) : log_approx(u_a);
                if (log_w < log_acc) {
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        theta[k] = th_l[k];
                        y[k] = y_l[k];
                    }
                    moved = true;
                    lq_valid = false;
                }
                d1 = prior_l;
                d2 = kern_l;
                d3 = log_acc;
            }
            stats.update(is_global, moved, theta, prev);
            ++done;
            if (layout != GLABC_TRACE_NONE) {
                const int64_t row = static_cast<int64_t>(i) - R.trace_row_base;
                float* dst = layout == GLABC_TRACE_CHAIN_MAJOR ? R.trace + ((R.trace_chain_off + c) * R.trace_rows + row) * D
                                                               : R.trace + (row * R.trace_chains + R.trace_chain_off + c) * D;
                store_row<D>(dst, theta);
            }
            if constexpr (REPLAY) {
                if (R.debug != nullptr) {
                    float* g = R.debug + srow * GLABC_DEBUG_SLOTS * C + c;
                    g[0] = static_cast<float>(static_cast<int>(is_global) | (static_cast<int>(moved) << 1) |
                                              ((is_global ? ind + 1 : 0) << 8));
                    g[C] = d1;
                    g[2 * C] = d2;
                    g[3 * C] = d3;
                }
            }
            ++i;
            running = i <= R.last_step && kk < K.S;
        }
    }

    if (in_range) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            R.theta[c * D + k] = theta[k];
            R.y[c * D + k] = y[k];
        }
        W.kk[c] = kk;
        W.next_step[c] = i;
        W.lq_cur[c] = lq_cur;
        W.lq_valid[c] = lq_valid ? 1 : 0;
        W.pending[c] = (kk >= K.S ? 1 : 0) | (pend_lq ? 2 : 0);  // :169: adapt before the next iteration
        if (R.stats != nullptr && done > 0) stats.store(R.stats + c * GLABC_NSTATS(D), done);
    }
}

// row 0 of the trace = the initial theta (the reference leaves zeros there, SURVEY.md B-10)
template <int D>
__global__ void __launch_bounds__(256) k_ag_row0(RunParams R, int64_t C, int layout)
{
    const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const int64_t row = static_cast<int64_t>(R.first_step) - 1 - R.trace_row_base;
    float v[D];
#pragma unroll
    for (int k = 0; k < D; ++k) v[k] = R.theta[c * D + k];
    float* dst = layout == GLABC_TRACE_CHAIN_MAJOR ? R.trace + ((R.trace_chain_off + c) * R.trace_rows + row) * D
                                                   : R.trace + (row * R.trace_chains + R.trace_chain_off + c) * D;
    store_row<D>(dst, v);
}

// GLMCMC-NFs block refresh (GLMCMC_NFs.py:73-85,129-140): theta0 / log q0 come from the flow; simulate, log-kernel,
// weights exp(prior + log K - log q0) with NaN -> 0.  One thread per (chain, b); `round` keys the simulator normals.
template <int D>
__global__ void __launch_bounds__(256) k_blk_weights(const __grid_constant__ AgConsts K, const __grid_constant__ RunParams R,
                                                     AgWorkspace W, uint32_t round, const __grid_constant__ DistConsts prior)
{
    const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (g >= W.C * W.B) return;
    const int64_t c = g / W.B;
    const int b = static_cast<int>(g - c * W.B);
    const uint64_t gid = (static_cast<uint64_t>(R.chain_hi0) << 32 | R.chain_lo0) + static_cast<uint64_t>(c);
    const Stream st{static_cast<uint32_t>(gid), static_cast<uint32_t>(gid >> 32)};
    float th[D], eps_s[D], x[D];
#pragma unroll
    for (int k = 0; k < D; ++k) th[k] = W.blk_theta[(c * W.B + b) * D + k];
    const uint4 w = st.block(R.rk, round, kSlotAdSim + static_cast<uint32_t>(b));
    float z[4];
    box_muller(w.x, w.y, z[0], z[1]);
    box_muller(w.z, w.w, z[2], z[3]);
#pragma unroll
    for (int k = 0; k < D; ++k) eps_s[k] = z[k];
    model_simulate<D, true>(K.model, th, eps_s, x);
    const float like = model_log_kernel<D, true>(K.model, x);
    float wgt = expf(__fsub_rn(__fadd_rn(prior_log_prob_rt<D>(K.model, prior, th), like), W.blk_lq[c * W.B + b]));
    if (wgt != wgt) wgt = 0.0f;  // GLMCMC_NFs.py:84-85 (rows with NaN proposals get weight 0 as well, :83)
#pragma unroll
    for (int k = 0; k < D; ++k) W.blk_x[(c * W.B + b) * D + k] = x[k];
    W.blk_w[c * W.B + b] = wgt;
}

// `prior`: a Uniform / Gamma / GaussianMixture prior of the model (FAST, native RNG only) or GLABC_DIST_DIAG_GAUSSIAN for K.model's
cudaError_t launch_block_isir(const AgConsts& K, const DistConsts& prior, const AgWorkspace& W, const RunParams& R, int dim, bool strict,
                              int layout, int block, cudaStream_t st);
cudaError_t launch_block_weights(const AgConsts& K, const DistConsts& prior, const AgWorkspace& W, const RunParams& R, int dim,
                                 uint32_t round, cudaStream_t st);

cudaError_t launch_aglmcmc(const AgConsts& K, const DistConsts& prior, const AgWorkspace& W, const AgTapes& T, const RunParams& R,
                           int dim, int init, int kde_rule, bool strict, bool replay, int layout, int block, cudaStream_t st);

}  // namespace glabc
