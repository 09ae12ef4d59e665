// The GlobalMCMC step (GlobalMCMC.py:37-68) for ANY of the reference's proposal distributions (dist_device.cuh) in the
// Local_Proposal / Global_Proposal slots.  K1 (step_global.cuh) is the tuned kernel for the all-Gaussian case; this is
// the general one: one thread = one chain, native Philox RNG, float32 (the reference evaluates Gamma / GaussianMixture
// in float64 — agreement is to float32 rounding, checked against the reference's recorded log-densities).
#pragma once
#include "launch.cuh"
#include "sampler_common.cuh"
#include "dist_device.cuh"

namespace glabc {

constexpr int kGenMaxDim = 4;

using DistConsts = DistConstsT<kGenMaxDim>;

struct GenericConsts {
    ModelConsts model;
    DistConsts lp, gp;
};

constexpr uint32_t kSlotGeneric = 0x50000000u;  // word stream of the generic proposals: blocks kSlotGeneric + 0, 1, ...

// sequential 32-bit words / uniforms / normals of one (chain, step): successive Philox blocks of a dedicated slot range
struct WordStream {
    const RoundKeys& rk;
    Stream st;
    uint32_t step, slot;
    uint4 cur;
    int used;
    float spare;
    bool has_spare;
    __device__ __forceinline__ WordStream(const RoundKeys& k, const Stream& s, uint32_t stp, uint32_t slot0)
        : rk(k), st(s), step(stp), slot(slot0), cur(make_uint4(0, 0, 0, 0)), used(4), spare(0.0f), has_spare(false) {}
    __device__ __forceinline__ uint32_t next()
    {
        if (used == 4) {
            cur = st.block(rk, step, slot++);
            used = 0;
        }
        const uint32_t w = used == 0 ? cur.x : used == 1 ? cur.y : used == 2 ? cur.z : cur.w;
        ++used;
        return w;
    }
    __device__ __forceinline__ float uniform() { return u24(next()); }                       // [0, 1) on the 2^-24 grid
    __device__ __forceinline__ float uniform_open() { return fmaf(__uint2float_rn(next() >> 8), 0x1p-24f, 0x1p-25f); }  // (0, 1)
    __device__ __forceinline__ float normal()
    {
        if (has_spare) {
            has_spare = false;
            return spare;
        }
        const uint32_t w0 = next(), w1 = next();
        float n0, n1;
        box_muller(w0, w1, n0, n1);
        spare = n1;
        has_spare = true;
        return n0;
    }
};

// The model's prior.  A DiagGaussian prior lives in ModelConsts (model_prior, the tuned arithmetic of both modes); a
// Uniform / Gamma / GaussianMixture one bound with glabc_model_prior_set arrives as a DistConsts and is evaluated by
// dist_log_prob (FAST only): GPRIOR kernels are instantiated for that case.  The kernels that run once per adaptation
// choose at run time (generic_prior): `prior.kind` is GLABC_DIST_DIAG_GAUSSIAN when the model's own prior applies.
template <int D, bool STRICT, bool GPRIOR>
__device__ __forceinline__ float prior_log_prob(const ModelConsts& m, const DistConsts& prior, const float (&theta)[D])
{
    if constexpr (GPRIOR) return dist_log_prob<D>(prior, theta);
    else return model_prior<D, STRICT>(m, theta);
}

__host__ __device__ __forceinline__ bool generic_prior(const DistConsts& prior) { return prior.kind != GLABC_DIST_DIAG_GAUSSIAN; }

template <int D>
__device__ __forceinline__ float prior_log_prob_rt(const ModelConsts& m, const DistConsts& prior, const float (&theta)[D])
{
    return generic_prior(prior) ? dist_log_prob<D>(prior, theta) : model_prior<D, true>(m, theta);
}

// GlobalMCMC.py:37-68 with arbitrary proposal kinds.
// REPLAY (parity mode): the reference's own draws drive the step — tape32 [steps][2 + D][C] = U_b, eps_sim[D], U_a and
// tape64 [steps][D][C] = the proposal's draw in float64 (theta' of a global move, the increment z of a local one; Gamma and
// GaussianMixture draw in float64, distribution.py:118,238-240).  The state is carried in float64 with the reference's dtype
// promotion: theta becomes a float64 tensor after the first accepted float64 candidate, and `z + theta` is then a float64
// add (GlobalMCMC.py:56) — so the float32 trace rows (Theta_Re[i] = Theta_old, :52,67) match bit for bit.  Densities are
// evaluated in float32 from the rounded state (the reference's are float64 after promotion: agreement to 1e-6).
// GPRIOR: the model's prior is `prior` (native RNG only).  Outside its support the log prior is -inf, so the first
// candidate with a finite prior is accepted (log_acc = +inf) and one with -inf never is.
template <int D, bool REPLAY, bool GPRIOR>
__global__ void __launch_bounds__(128) k_global_generic(const __grid_constant__ GenericConsts K, const __grid_constant__ RunParams R,
                                                        int layout, const __grid_constant__ DistConsts prior)
{
    static_assert(!(REPLAY && GPRIOR), "replay runs the model's DiagGaussian prior");
    const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= R.n_chains) return;
    float theta[D], y[D];
    double th64[D];
    bool wide = false;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        theta[k] = R.theta[c * D + k];
        y[k] = R.y[c * D + k];
        th64[k] = static_cast<double>(theta[k]);
    }
    auto put = [&](uint32_t row_abs) {
        if (layout == GLABC_TRACE_NONE) return;
        const int64_t row = static_cast<int64_t>(row_abs) - R.trace_row_base;
        float* dst = layout == GLABC_TRACE_CHAIN_MAJOR ? R.trace + ((R.trace_chain_off + c) * R.trace_rows + row) * D
                                                       : R.trace + (row * R.trace_chains + R.trace_chain_off + c) * D;
        store_row<D>(dst, theta);
    };
    if (R.write_row0) put(R.first_step - 1u);
    ChainStats<D> stats;
    const Stream stream = chain_stream(R, static_cast<int32_t>(c));
    float prior_old = prior_log_prob<D, false, GPRIOR>(K.model, prior, theta), kern_old = model_log_kernel<D, false>(K.model, y);
    const bool lp64 = K.lp.kind == GLABC_DIST_GAMMA || K.lp.kind == GLABC_DIST_GAUSSIAN_MIXTURE;
    const bool gp64 = K.gp.kind == GLABC_DIST_GAMMA || K.gp.kind == GLABC_DIST_GAUSSIAN_MIXTURE;

    for (uint32_t i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
        bool is_global, p_wide = false;
        float log_w, th_p[D], y_p[D], eps_s[D], corr = 0.0f;
        double th_p64[D];
        if constexpr (REPLAY) {
            const int64_t srow = static_cast<int64_t>(i - R.first_step), C = R.n_chains;
            const float* tp = R.tape32 + srow * (2 + D) * C + c;
            is_global = __ldg(tp) < R.gf;                                            // GlobalMCMC.py:39
            log_w = logf(__ldg(tp + static_cast<int64_t>(1 + D) * C));                // :47,62
            double draw[D];
#pragma unroll
            for (int k = 0; k < D; ++k) {
                eps_s[k] = __ldg(tp + static_cast<int64_t>(1 + k) * C);
                draw[k] = R.tape64[(srow * D + k) * C + c];
            }
            if (is_global) {
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    th_p64[k] = draw[k];
                    th_p[k] = static_cast<float>(draw[k]);
                }
                corr = dist_log_prob<D>(K.gp, theta) - dist_log_prob<D>(K.gp, th_p);   // :45-46 (forward's log_p == log_prob(theta'))
                p_wide = gp64;
            } else {
                p_wide = wide || lp64;                                                // dtype of z + Theta_old, :56
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    th_p64[k] = p_wide ? draw[k] + th64[k]
                                       : static_cast<double>(__fadd_rn(static_cast<float>(draw[k]), static_cast<float>(th64[k])));
                    th_p[k] = static_cast<float>(th_p64[k]);
                }
            }
        } else {
            const uint4 w0 = stream.block(R.rk, i, kSlotStep);
            is_global = (step_block_ub(w0) < R.gf_thr_hi) || R.gf_all_global;  // GlobalMCMC.py:39
            log_w = log_approx(__uint2float_rn(step_block_ua(w0)) * 0x1p-24f);  // :47,62
            WordStream ws(R.rk, stream, i, kSlotGeneric);
            if (is_global) {
                const float lq_p = dist_forward<D>(K.gp, ws, th_p);       // :40
                corr = dist_log_prob<D>(K.gp, theta) - lq_p;              // :45-46
            } else {
                float z[D];
                (void)dist_forward<D>(K.lp, ws, z);                       // Local_Proposal.sample(1), :56
#pragma unroll
                for (int k = 0; k < D; ++k) th_p[k] = z[k] + theta[k];
            }
#pragma unroll
            for (int k = 0; k < D; ++k) eps_s[k] = ws.normal();
        }
        model_simulate<D, false>(K.model, th_p, eps_s, y_p);           // :41,57
        const float prior_p = prior_log_prob<D, false, GPRIOR>(K.model, prior, th_p), kern_p = model_log_kernel<D, false>(K.model, y_p);
        const float log_acc = (prior_p + kern_p) + corr - (prior_old + kern_old);   // :44-46 / :60-61
        const bool accept = log_w < log_acc;                                        // :49,64 (NaN rejects)
        float prev[D];
#pragma unroll
        for (int k = 0; k < D; ++k) prev[k] = theta[k];
        if (accept) {
#pragma unroll
            for (int k = 0; k < D; ++k) {
                theta[k] = th_p[k];
                y[k] = y_p[k];
                if constexpr (REPLAY) th64[k] = th_p64[k];
            }
            prior_old = prior_p;
            kern_old = kern_p;
            if constexpr (REPLAY) wide = p_wide;
        }
        stats.update(is_global, accept, theta, prev);
        put(i);
        if constexpr (REPLAY) {
            if (R.debug != nullptr) {
                float* g = R.debug + static_cast<int64_t>(i - R.first_step) * GLABC_DEBUG_SLOTS * R.n_chains + c;
                g[0] = static_cast<float>(static_cast<int>(is_global) | (static_cast<int>(accept) << 1));
                g[R.n_chains] = prior_p;
                g[2 * static_cast<int64_t>(R.n_chains)] = kern_p;
                g[3 * static_cast<int64_t>(R.n_chains)] = log_acc;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        R.theta[c * D + k] = theta[k];
        R.y[c * D + k] = y[k];
    }
    if (R.stats != nullptr) stats.store(R.stats + c * GLABC_NSTATS(D), R.last_step + 1u - R.first_step);
}

// torch.sum over n (< 32) contiguous values in ATen's order (SumKernel row_sum: four interleaved partials for n < 16, the
// 16-lane vector path — tail first — for n >= 16; SURVEY.md B-3), in the values' own type
template <typename T>
__device__ __forceinline__ T torch_sum_rt(const T* v, int n)
{
    if (n >= 16) {
        T acc = T(0);
        for (int i = 16; i < n; ++i) acc = acc + v[i];
        for (int i = 0; i < 16; ++i) acc = acc + v[i];
        return acc;
    }
    T p0 = T(0), p1 = T(0), p2 = T(0), p3 = T(0);
    const int rows = n >> 2;
    for (int r = 0; r < rows; ++r) {
        p0 = p0 + v[4 * r];
        p1 = p1 + v[4 * r + 1];
        p2 = p2 + v[4 * r + 2];
        p3 = p3 + v[4 * r + 3];
    }
    for (int i = 4 * rows; i < n; ++i) p0 = p0 + v[i];
    return ((p0 + p1) + p2) + p3;
}

struct IsirGenericConsts {
    ModelConsts model;
    DistConsts lp, ip;
};

// GLMCMC.py:58-104 (weight_sampling :7-22) with arbitrary proposal kinds in the Local / Importance slots.
// dtype rules of the reference, reproduced because they change decisions: a Gamma / GaussianMixture draw is float64
// (distribution.py:118,238-240), so after such a candidate is taken — or after a local move with a float64 increment — the
// state is a float64 tensor, and the log-weights of a global move are float64 as soon as the current state's or the
// candidates' are (torch.cat promotes): their exp does not underflow near -104 as the float32 one does (B-1).
// REPLAY: tape32 [steps][2 + K D][C] = U_b, eps_sim[K][D] (a local move: eps_sim[D] first), U_a (last slot);
// tape64 [steps][1 + K D][C] = the numpy resampling uniform, then the proposal's own draws (theta_j; local: increment z).
// GPRIOR: the model's prior is `prior` (native RNG only), as in k_global_generic; a candidate outside its support has
// log-weight -inf, i.e. weight 0, and is never selected.
template <int D, bool REPLAY, bool GPRIOR>
__global__ void __launch_bounds__(128) k_isir_generic(const __grid_constant__ IsirGenericConsts K, const __grid_constant__ RunParams R,
                                                      int layout, const __grid_constant__ DistConsts prior)
{
    static_assert(!(REPLAY && GPRIOR), "replay runs the model's DiagGaussian prior");
    const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= R.n_chains) return;
    const int64_t C = R.n_chains;
    const int NK = R.n_candidates;
    float theta[D], y[D];
    double th64[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        theta[k] = R.theta[c * D + k];
        y[k] = R.y[c * D + k];
        th64[k] = static_cast<double>(theta[k]);
    }
    float* aux = R.aux + c * GLABC_AUX_SLOTS;
    double lw_old = static_cast<double>(aux[GLABC_AUX_LOGW]);
    bool local = aux[GLABC_AUX_LOCAL] != 0.0f, wide = aux[GLABC_AUX_WIDE] != 0.0f, lw_wide = aux[GLABC_AUX_LW_WIDE] != 0.0f;
    auto put = [&](uint32_t row_abs) {
        if (layout == GLABC_TRACE_NONE) return;
        const int64_t row = static_cast<int64_t>(row_abs) - R.trace_row_base;
        float* dst = layout == GLABC_TRACE_CHAIN_MAJOR ? R.trace + ((R.trace_chain_off + c) * R.trace_rows + row) * D
                                                       : R.trace + (row * R.trace_chains + R.trace_chain_off + c) * D;
        store_row<D>(dst, theta);
    };
    if (R.write_row0) put(R.first_step - 1u);
    ChainStats<D> stats;
    const Stream stream = chain_stream(R, static_cast<int32_t>(c));
    const bool lp64 = K.lp.kind == GLABC_DIST_GAMMA || K.lp.kind == GLABC_DIST_GAUSSIAN_MIXTURE;
    const bool ip64 = K.ip.kind == GLABC_DIST_GAMMA || K.ip.kind == GLABC_DIST_GAUSSIAN_MIXTURE;
    const int tslots = 2 + NK * D;   // U_b, eps_sim[K][D], U_a

    for (uint32_t i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
        const int64_t srow = static_cast<int64_t>(i - R.first_step);
        const float* tp = nullptr;
        const double* tq = nullptr;
        bool is_global;
        uint4 w0 = make_uint4(0, 0, 0, 0);
        if constexpr (REPLAY) {
            tp = R.tape32 + srow * tslots * C + c;
            tq = R.tape64 + srow * (1 + NK * D) * C + c;
            is_global = __ldg(tp) < R.gf;                                   // GLMCMC.py:59
        } else {
            w0 = stream.block(R.rk, i, kSlotStep);
            is_global = (step_block_ub(w0) < R.gf_thr_hi) || R.gf_all_global;
        }
        WordStream ws(R.rk, stream, i, kSlotGeneric);
        float prev[D];
#pragma unroll
        for (int k = 0; k < D; ++k) prev[k] = theta[k];
        bool changed = false;
        float d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
        int ind = -1;
        bool w64 = false;
        float lw[GLABC_MAX_K + 1];

        if (is_global) {
            if (local) {                                                     // :60-64
                lw_old = static_cast<double>((prior_log_prob<D, false, GPRIOR>(K.model, prior, theta) + model_log_kernel<D, false>(K.model, y)) -
                                             dist_log_prob<D>(K.ip, theta));
                lw_wide = wide;
            }
            local = false;
            float th_c[GLABC_MAX_K][D], x_c[GLABC_MAX_K][D];
            double th_c64[GLABC_MAX_K][D];
            for (int j = 0; j < NK; ++j) {                                   // :66-74
                float tj[D], xj[D], es[D], lq;
                if constexpr (REPLAY) {
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        th_c64[j][k] = tq[static_cast<int64_t>(1 + j * D + k) * C];
                        tj[k] = static_cast<float>(th_c64[j][k]);
                        es[k] = __ldg(tp + static_cast<int64_t>(1 + j * D + k) * C);
                    }
                    lq = dist_log_prob<D>(K.ip, tj);                         // forward()'s log_p of its own draw
                } else {
                    lq = dist_forward<D>(K.ip, ws, tj);
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        es[k] = ws.normal();
                        th_c64[j][k] = static_cast<double>(tj[k]);
                    }
                }
                model_simulate<D, false>(K.model, tj, es, xj);
                lw[j + 1] = (prior_log_prob<D, false, GPRIOR>(K.model, prior, tj) + model_log_kernel<D, false>(K.model, xj)) - lq;
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    th_c[j][k] = tj[k];
                    x_c[j][k] = xj[k];
                }
            }
            double u64;
            if constexpr (REPLAY) {
                u64 = tq[0];
            } else {
                const uint4 wu = stream.block(R.rk, i, kSlotU64);
                u64 = static_cast<double>((static_cast<uint64_t>(wu.x) << 21) | (wu.y >> 11)) * 0x1p-53;
            }
            w64 = lw_wide || ip64;                                           // dtype of torch.cat((log_weight_old, log_weight0)), :75
            lw[0] = static_cast<float>(lw_old);
            double S, w0n;
            if (w64) {                                                       // float64 weights: no underflow near -104
                double w[GLABC_MAX_K + 1];
                w[0] = exp(lw_old);
                for (int j = 1; j <= NK; ++j) w[j] = exp(static_cast<double>(lw[j]));
                for (int j = 0; j <= NK; ++j)
                    if (w[j] != w[j]) w[j] = 0.0;                            // :80-81
                S = torch_sum_rt<double>(w, NK + 1);
                double run = 0.0;
                for (int j = 0; j <= NK; ++j) {                              // weight_sampling, :7-22
                    const double q = w[j] / S;
                    run += q;
                    if (ind < 0 && u64 < run) ind = j;
                }
                w0n = w[0] / S;
            } else {                                                         // float32 weights, un-shifted (B-1)
                float w[GLABC_MAX_K + 1];
                for (int j = 0; j <= NK; ++j) {
                    w[j] = expf(lw[j]);
                    if (w[j] != w[j]) w[j] = 0.0f;
                }
                const float Sf = torch_sum_rt<float>(w, NK + 1);
                double run = 0.0;
                for (int j = 0; j <= NK; ++j) {
                    const float q = __fdiv_rn(w[j], Sf);
                    run += static_cast<double>(q);
                    if (ind < 0 && u64 < run) ind = j;
                }
                S = static_cast<double>(Sf);
                w0n = static_cast<double>(__fdiv_rn(w[0], Sf));
            }
            d1 = static_cast<float>(lw_old);
            d2 = static_cast<float>(S);
            d3 = static_cast<float>(w0n);
            if (ind > 0) {                                                   // :84-88
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    theta[k] = th_c[ind - 1][k];
                    y[k] = x_c[ind - 1][k];
                    th64[k] = th_c64[ind - 1][k];
                }
                lw_old = static_cast<double>(lw[ind]);
                wide = wide || ip64;
                lw_wide = w64;
            }
        } else {
            // ---- local random walk, :90-104 (the prior-sentinel redraw of :92-93 cannot fire for the fused Gaussian prior) ----
            float th_p[D], y_p[D], es[D], u_a;
            double th_p64[D];
            const bool p_wide = wide || lp64;                                // dtype of Local_Proposal.sample(1) + Theta_old, :91
            if constexpr (REPLAY) {
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    const double z = tq[static_cast<int64_t>(1 + k) * C];
                    th_p64[k] = p_wide ? z + th64[k] : static_cast<double>(__fadd_rn(static_cast<float>(z), static_cast<float>(th64[k])));
                    th_p[k] = static_cast<float>(th_p64[k]);
                    es[k] = __ldg(tp + static_cast<int64_t>(1 + k) * C);
                }
                u_a = __ldg(tp + static_cast<int64_t>(1 + NK * D) * C);
            } else {
                float z[D];
                (void)dist_forward<D>(K.lp, ws, z);
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    th_p[k] = z[k] + theta[k];
                    th_p64[k] = static_cast<double>(th_p[k]);
                    es[k] = ws.normal();
                }
                u_a = __uint2float_rn(step_block_ua(w0)) * 0x1p-24f;
            }
            model_simulate<D, false>(K.model, th_p, es, y_p);
            const float pr_p = prior_log_prob<D, false, GPRIOR>(K.model, prior, th_p), k_p = model_log_kernel<D, false>(K.model, y_p);
            const float log_acc = (pr_p + k_p) - (prior_log_prob<D, false, GPRIOR>(K.model, prior, theta) +
                                                  model_log_kernel<D, false>(K.model, y));   // :96-97
            d1 = pr_p;
            d2 = k_p;
            d3 = log_acc;
            if (logf(u_a) < log_acc) {                                       // :98-103
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    theta[k] = th_p[k];
                    y[k] = y_p[k];
                    th64[k] = th_p64[k];
                }
                wide = p_wide;
                local = true;
            }
        }
#pragma unroll
        for (int k = 0; k < D; ++k) changed |= theta[k] != prev[k];
        stats.update(is_global, changed, theta, prev);
        put(i);
        if constexpr (REPLAY) {
            if (R.debug != nullptr) {
                float* g = R.debug + srow * GLABC_DEBUG_SLOTS * C + c;
                g[0] = static_cast<float>(static_cast<int>(is_global) | (static_cast<int>(changed) << 1) | ((is_global ? ind + 1 : 0) << 8) |
                                          (static_cast<int>(is_global && w64) << 16));
                g[C] = d1;
                g[2 * C] = d2;
                g[3 * C] = d3;
                if (is_global)
                    for (int j = 0; j < NK; ++j) g[static_cast<int64_t>(4 + j) * C] = lw[j + 1];
            }
        }
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        R.theta[c * D + k] = theta[k];
        R.y[c * D + k] = y[k];
    }
    aux[GLABC_AUX_LOGW] = static_cast<float>(lw_old);
    aux[GLABC_AUX_LOCAL] = local ? 1.0f : 0.0f;
    aux[GLABC_AUX_WIDE] = wide ? 1.0f : 0.0f;
    aux[GLABC_AUX_LW_WIDE] = lw_wide ? 1.0f : 0.0f;
    if (R.stats != nullptr) stats.store(R.stats + c * GLABC_NSTATS(D), R.last_step + 1u - R.first_step);
}

// device-side forward() / log_prob() of a bound distribution (glabc_dist_sample / glabc_dist_log_prob)
template <int D>
__global__ void __launch_bounds__(256) k_dist_eval(const __grid_constant__ DistConsts q, RoundKeys rk, int64_t n, const float* __restrict__ z_in,
                                                   float* __restrict__ z_out, float* __restrict__ logp)
{
    const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (g >= n) return;
    float z[D];
    float lp;
    if (z_in != nullptr) {
#pragma unroll
        for (int k = 0; k < D; ++k) z[k] = z_in[g * D + k];
        lp = dist_log_prob<D>(q, z);
    } else {
        const Stream st{static_cast<uint32_t>(g), static_cast<uint32_t>(g >> 32)};
        WordStream ws(rk, st, 0u, kSlotGeneric);
        lp = dist_forward<D>(q, ws, z);
#pragma unroll
        for (int k = 0; k < D; ++k) z_out[g * D + k] = z[k];
    }
    if (logp != nullptr) logp[g] = lp;
}

// `prior`: the model's prior when generic_prior(prior) (native RNG only), else the DiagGaussian of K.model applies
cudaError_t launch_global_generic(const GenericConsts& K, const DistConsts& prior, int dim, const RunParams& R, int layout, int block,
                                  bool replay, cudaStream_t st);
cudaError_t launch_isir_generic(const IsirGenericConsts& K, const DistConsts& prior, int dim, const RunParams& R, int layout, int block,
                                bool replay, cudaStream_t st);
cudaError_t launch_dist_eval(const DistConsts& q, int dim, const RoundKeys& rk, int64_t n, const float* z_in, float* z_out, float* logp,
                             cudaStream_t st);

}  // namespace glabc
