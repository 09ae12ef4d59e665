// K3, throughput path (FAST arithmetic, native Philox, no tape dump): GLMALA.py:150-200 with
//   * one THREAD per chain for everything that is cheap and per-chain — the branch coin, the iSIR global move
//     (GLMALA.py:151-180; the K candidates are independent, so a thread has K-way instruction-level parallelism) and the
//     tail of the MALA move (proposal, five log-densities, accept; GLMALA.py:186-199);
//   * the WARP for the one expensive piece, numberical_gradient_logABC (GLMALA.py:46-95): the chains of a warp that drew a
//     local move this step (a ballot) are served one after the other, the d * num_grad Philox / Box-Muller / simulate /
//     discrepancy items of a gradient dealt over the 32 lanes (D = 2: lanes 0-15 dimension 0, lanes 16-31 dimension 1, so
//     a gradient folds four float32 sums over 16 lanes), and only the owner keeps the folded sums.
// The warp-per-chain kernel of step_mala.cuh (STRICT / replay / tape dump — the parity path) spends 32 lanes on every
// per-chain scalar; here a warp-step costs about 700 (global moves, 32 chains at once) + 6.4 x 600 (gradients, gf = 0.8)
// + 200 (tails) warp-instructions for 32 chain-steps instead of 32 x 533.
//
// Same Philox stream layout as step_mala.cuh (and the oracle's native mode): a chain's draws do not depend on which of
// the two kernels ran it.  State is float32 here (the reference's float64 promotion only matters for the un-shifted
// float32 exp of the iSIR weights, which is handled as in step_mala.cuh: max-shifted once the state is `wide`).
#pragma once
#include "step_mala.cuh"

#ifndef GLABC_MALA_UNROLL
#define GLABC_MALA_UNROLL 1
#endif
#ifndef GLABC_MALA_KUNROLL
#define GLABC_MALA_KUNROLL 5
#endif
// one warp per CTA: at 32,768 chains 64-thread CTAs are 512 CTAs = 3.46 per SM (a 4 : 3 imbalance over the SMs); 32-thread
// CTAs measured 5 % faster there and 2 % faster at 262,144 chains (profiles/micro/k3_block.sh)
#ifndef GLABC_MALA_BLOCK
#define GLABC_MALA_BLOCK 32
#endif
#define GLABC_PRAGMA(x) _Pragma(#x)
#define GLABC_UNROLL(n) GLABC_PRAGMA(unroll n)

namespace glabc {

// dealing of a gradient's (dimension k, Philox block g) items over the lanes
template <int D> struct GradDeal { static constexpr int kLanesPerDim = 32; };  // k one after the other
template <> struct GradDeal<2> { static constexpr int kLanesPerDim = 16; };    // both dimensions at once
template <> struct GradDeal<4> { static constexpr int kLanesPerDim = 8; };     // four at once

template <int D, int FAMILY>
__device__ __forceinline__ float sim_discrepancy_fast(const ModelConsts& m, const float (&base)[D], const float (&eps)[D])
{
    // base[i] = mean(theta_i) + noise_loc_i - y_obs_i, hoisted out of the draw loop
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < D; ++i) {
        const float dy = fmaf(m.noise_scale[i], eps[i], base[i]);
        s = fmaf(dy, dy, s);
    }
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(s));
    return r;
}

// One chain's gradient sums, computed by the whole warp.  tgt = theta (float32) of the chain owned by lane `src`;
// on return lane `src` holds, for every k, (sum x+, sum x+^2, sum x-, sum x-^2) with x = discrepancy - noise-free
// discrepancy, and the noise-free discrepancies c+-.
template <int D, int FAMILY>
__device__ __forceinline__ void warp_gradient_sums(const MalaConsts& K, const RoundKeys& rk, const Stream& src_stream, uint32_t step,
                                                   uint32_t slot0, const float (&th)[D], int lane, bool mine,
                                                   float (&sums)[D][4], float (&cpm)[D][2])
{
    constexpr int kDpb = D == 3 ? 1 : 4 / D;  // draws per Philox block
    constexpr int LPD = GradDeal<D>::kLanesPerDim;
    constexpr int KPAR = 32 / LPD;            // dimensions in flight
    const int num = K.num_grad;
    const int nblk = (num + kDpb - 1) / kDpb;
    const int sub = lane & (LPD - 1);
#pragma unroll 1
    for (int k0 = 0; k0 < D; k0 += KPAR) {
        const int k = k0 + (KPAR > 1 ? lane / LPD : 0);
        float bp[D], bm[D];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            const float tp = i == k ? th[i] + 0.1f : th[i];  // GLMALA.py:63-67
            const float tm = i == k ? th[i] - 0.1f : th[i];
            const float off = K.model.noise_loc[i] - K.model.y_obs[i];
            bp[i] = (FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(tp) : tp) + off;
            bm[i] = (FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(tm) : tm) + off;
        }
        const float zero[D] = {};
        const float cp = sim_discrepancy_fast<D, FAMILY>(K.model, bp, zero), cm = sim_discrepancy_fast<D, FAMILY>(K.model, bm, zero);
        float f1p = 0.0f, f2p = 0.0f, f1m = 0.0f, f2m = 0.0f;
        const uint32_t slot_k = slot0 + static_cast<uint32_t>(k * nblk);
        auto block_of_draws = [&](int g, int n_live) {
            const uint4 w = src_stream.block(rk, step, slot_k + static_cast<uint32_t>(g));
            float z[4];
            box_muller(w.x, w.y, z[0], z[1]);
            box_muller(w.z, w.w, z[2], z[3]);
#pragma unroll
            for (int t = 0; t < kDpb; ++t) {
                float eps[D];
#pragma unroll
                for (int q = 0; q < D; ++q) eps[q] = z[t * D + q];
                float xp = sim_discrepancy_fast<D, FAMILY>(K.model, bp, eps) - cp;  // :78-79
                float xm = sim_discrepancy_fast<D, FAMILY>(K.model, bm, eps) - cm;  // :80-83 (the same draws)
                if (t >= n_live) xp = xm = 0.0f;     // compile-time false in the full-block loop
                f1p += xp;
                f2p = fmaf(xp, xp, f2p);
                f1m += xm;
                f2m = fmaf(xm, xm, f2m);
            }
        };
        // NOT unrolled: measured at 262,144 chains, unroll 1 / 2 / 4 = 5.0e9 / 4.5e9 / 3.5e9 chain-steps/s — the loop body must
        // stay resident in the instruction cache while the warps of an SM sit in different phases of the step
        const int nfull = num / kDpb;                 // blocks whose kDpb draws all count; at most one partial block follows
GLABC_UNROLL(GLABC_MALA_UNROLL)
        for (int g = sub; g < nfull; g += LPD) block_of_draws(g, kDpb);
        if (nfull < nblk && (nfull & (LPD - 1)) == sub) block_of_draws(nfull, num - nfull * kDpb);
#pragma unroll
        for (int off = LPD / 2; off > 0; off >>= 1) {
            f1p += __shfl_xor_sync(0xffffffffu, f1p, off);
            f2p += __shfl_xor_sync(0xffffffffu, f2p, off);
            f1m += __shfl_xor_sync(0xffffffffu, f1m, off);
            f2m += __shfl_xor_sync(0xffffffffu, f2m, off);
        }
        // hand the sums of dimension k0 + q to the owner: lane q * LPD holds them after the fold
#pragma unroll
        for (int q = 0; q < KPAR; ++q) {
            const int from = q * LPD;
            const float a = __shfl_sync(0xffffffffu, f1p, from), b = __shfl_sync(0xffffffffu, f2p, from);
            const float c = __shfl_sync(0xffffffffu, f1m, from), d = __shfl_sync(0xffffffffu, f2m, from);
            const float e = __shfl_sync(0xffffffffu, cp, from), f = __shfl_sync(0xffffffffu, cm, from);
#pragma unroll
            for (int kk = 0; kk < D; ++kk) {
                if (mine && kk == k0 + q) {
                    sums[kk][0] = a; sums[kk][1] = b; sums[kk][2] = c; sums[kk][3] = d;
                    cpm[kk][0] = e; cpm[kk][1] = f;
                }
            }
        }
    }
}

// numberical_gradient_logABC from the folded sums (GLMALA.py:84-95), per chain.  GPRIOR: the prior's finite difference
// straddling the edge of its support is non-finite, and so is the drift: the proposal is rejected (NaN / -inf log_acc).
template <int D, bool GPRIOR>
__device__ __forceinline__ void gradient_from_sums(const MalaConsts& K, const DistConsts& prior, const float (&th)[D],
                                                   const float (&sums)[D][4], const float (&cpm)[D][2], float (&grad)[D])
{
    const float rn = 1.0f / static_cast<float>(K.num_grad), rn1 = 1.0f / static_cast<float>(K.num_grad - 1);
    const float e2 = static_cast<float>(K.eps2);
#pragma unroll
    for (int k = 0; k < D; ++k) {
        float ta[D], tb[D];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            ta[i] = i == k ? __fadd_rn(th[i], 0.00001f) : th[i];  // :84-85
            tb[i] = i == k ? __fsub_rn(th[i], 0.00001f) : th[i];
        }
        // the float32 finite-difference prior gradient in the reference's exact operation order: its rounding IS its value (B-8)
        const float gprior = __fdiv_rn(__fsub_rn(prior_log_prob<D, true, GPRIOR>(K.model, prior, ta), prior_log_prob<D, true, GPRIOR>(K.model, prior, tb)),
                                       static_cast<float>(2 * 0.00001));
        const float f1p = sums[k][0], f2p = sums[k][1], f1m = sums[k][2], f2m = sums[k][3];
        const float mup = fmaf(f1p, rn, cpm[k][0]), mum = fmaf(f1m, rn, cpm[k][1]);
        const float vp = fmaf(fmaf(-f1p * rn, f1p, f2p), rn1, e2), vm = fmaf(fmaf(-f1m * rn, f1m, f2m), rn1, e2);
        // lpp - lpm = -0.5 * (log(vp / vm) + mup^2 / vp - mum^2 / vm)
        const float ivp = __fdividef(1.0f, vp), ivm = __fdividef(1.0f, vm);
        const float dl = 0.69314718055994531f * lg2_approx(vp * ivm) + (mup * mup * ivp - mum * mum * ivm);
        grad[k] = fmaf(dl, -2.5f, gprior);  // -0.5 / (2 * 0.1)
    }
}

// GIP: the Importance_Proposal is one of the non-Gaussian classes (K.ipg, step_generic.cuh): candidate j of a step is
// dist_forward over the word stream of Philox slots kSlotGeneric + 64 j .., its simulator normals follow in the same stream.
// GPRIOR: the model's prior is `prior` (step_generic.cuh prior_log_prob) in the iSIR weights, the MALA target and the
// finite-difference prior gradient.
template <int D, int FAMILY, int LAYOUT, bool GIP, bool GPRIOR>
__global__ void __launch_bounds__(GLABC_MALA_BLOCK) k_mala_fast(const __grid_constant__ MalaConsts K, const __grid_constant__ RunParams R,
                                                                const __grid_constant__ DistConsts prior)
{
    using Writer = typename WriterFor<D, LAYOUT>::type;
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int32_t warp_chain0 = static_cast<int32_t>((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32;
    const int32_t chain = warp_chain0 + lane;
    const bool active = chain < R.n_chains;
    const int32_t cidx = active ? chain : R.n_chains - 1;   // tail lanes read a valid chain and never write
    const int NK = R.n_candidates;
    constexpr int kGroups = (2 * D + 3) / 4;
    float* lw_tab = smem + Writer::smem_floats_per_warp * (blockDim.x >> 5);   // [NK][blockDim]: candidate log-weights
    Writer writer(R, cidx, active, smem + Writer::smem_floats_per_warp * warp);

    // ---- carried state, float32 ----
    float* aux = R.aux + static_cast<int64_t>(cidx) * GLABC_AUX_SLOTS;
    double* s64 = R.state64 + static_cast<int64_t>(cidx) * GLABC_STATE64_SLOTS;
    bool local = aux[GLABC_AUX_LOCAL] != 0.0f, wide = aux[GLABC_AUX_WIDE] != 0.0f;
    bool lw_wide = aux[GLABC_AUX_LW_WIDE] != 0.0f, have_grad = aux[GLABC_AUX_HAVE_GRAD] != 0.0f;
    float theta[D], y[D], grad[D], lw_old = static_cast<float>(s64[GLABC_S64_LOGW]);
#pragma unroll
    for (int k = 0; k < D; ++k) {
        theta[k] = wide ? static_cast<float>(s64[GLABC_S64_THETA + k]) : R.theta[static_cast<int64_t>(cidx) * D + k];
        y[k] = wide ? static_cast<float>(s64[GLABC_S64_Y + k]) : R.y[static_cast<int64_t>(cidx) * D + k];
        grad[k] = static_cast<float>(s64[GLABC_S64_GRAD + k]);
    }
    if (R.write_row0) {
        writer.put(R, R.first_step - 1u, theta);
        writer.maybe_flush(R, R.first_step - 1u);
    }

    ChainStats<D> stats;
    const Stream stream = chain_stream(R, cidx);
    const float tau = K.tau_f, half_tau2 = 0.5f * K.tau_f * K.tau_f, inv_tau = 1.0f / K.tau_f;

    for (uint32_t i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
        const uint4 w0 = stream.block(R.rk, i, kSlotStep);
        const bool glob_coin = (step_block_ub(w0) < R.gf_thr_hi) || R.gf_all_global;   // GLMALA.py:151
        const bool is_global = active && glob_coin, is_local = active && !glob_coin;
        float prev[D];
#pragma unroll
        for (int k = 0; k < D; ++k) prev[k] = theta[k];
        bool changed = false;

        if (is_global) {
            // ================= iSIR global move, GLMALA.py:151-180 =================
            if (local) {  // :152-156 — the only place log_weight_old is computed from the state
                const float q_old = GIP ? dist_log_prob<D>(K.ipg, theta) : gauss_log_prob<D, false>(K.ip, theta);
                lw_old = (prior_log_prob<D, false, GPRIOR>(K.model, prior, theta) + model_log_kernel<D, false>(K.model, y)) - q_old;
                lw_wide = wide;
            }
            local = false;
            float m = lw_old == lw_old ? lw_old : -INFINITY;
            uint4 wfirst = make_uint4(0, 0, 0, 0);
GLABC_UNROLL(GLABC_MALA_KUNROLL)
            for (int j = 0; j < NK; ++j) {   // :158-165, candidate j
                float th_c[D], x_c[D], lw_c;
                if constexpr (GIP) {
                    WordStream ws(R.rk, stream, i, kSlotGeneric + 64u * static_cast<uint32_t>(j));
                    const float lq = dist_forward<D>(K.ipg, ws, th_c);
                    float eps_s[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) eps_s[k] = ws.normal();
                    model_simulate<D, false>(K.model, th_c, eps_s, x_c);
                    lw_c = (prior_log_prob<D, false, GPRIOR>(K.model, prior, th_c) + model_log_kernel<D, false>(K.model, x_c)) - lq;
                    if (j == 0) wfirst = stream.block(R.rk, i, kSlotNormal + 8u);
                } else {
                    float zc[kGroups * 4];
#pragma unroll
                    for (int g = 0; g < kGroups; ++g) {
                        const uint4 w = stream.block(R.rk, i, kSlotNormal + 8u + j * kGroups + g);
                        if (j == 0 && g == 0) wfirst = w;
                        box_muller(w.x, w.y, zc[4 * g], zc[4 * g + 1]);
                        box_muller(w.z, w.w, zc[4 * g + 2], zc[4 * g + 3]);
                    }
                    float eps_p[D], eps_s[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        eps_p[k] = zc[k];
                        eps_s[k] = zc[D + k];
                    }
                    const float lq = gauss_forward<D, false>(K.ip, eps_p, th_c);
                    model_simulate<D, false>(K.model, th_c, eps_s, x_c);
                    lw_c = (prior_log_prob<D, false, GPRIOR>(K.model, prior, th_c) + model_log_kernel<D, false>(K.model, x_c)) - lq;
                }
                lw_tab[j * blockDim.x + threadIdx.x] = lw_c;
                m = fmaxf(m, lw_c == lw_c ? lw_c : -INFINITY);
            }
            // 53-bit resampling uniform from spare bits of the step block and of candidate 0's first block
            const uint64_t m53 = (static_cast<uint64_t>(step_block_ua(w0)) << 29) | (static_cast<uint64_t>(step_block_ua(wfirst)) << 5) |
                                 static_cast<uint64_t>(step_block_ub(wfirst) >> 27);
            const double u64 = static_cast<double>(m53) * 0x1p-53;
            // weights: un-shifted float32 exp while the reference's are float32 (all-underflow => None => stay, B-1),
            // max-shifted once they are float64 there (no underflow near -104)
            // (a Gamma / GaussianMixture proposal draws in float64, so with it the reference's weights are float64 from the start)
            const bool w64 = lw_wide || (GIP && (K.ipg.kind == GLABC_DIST_GAMMA || K.ipg.kind == GLABC_DIST_GAUSSIAN_MIXTURE));
            const float shift = w64 ? m : 0.0f;
            auto weight = [&](float lw) {
                float w;
                asm("ex2.approx.f32 %0, %1;" : "=f"(w) : "f"((lw - shift) * 1.4426950408889634f));
                return (w != w || (w64 && m == -INFINITY)) ? 0.0f : w;
            };
            const float w_cur = weight(lw_old);
            float S = w_cur;
            for (int j = 0; j < NK; ++j) S += weight(lw_tab[j * blockDim.x + threadIdx.x]);
            const double thr = u64 * static_cast<double>(S);   // u < cumsum(w) / S  <=>  u * S < cumsum(w)
            double run = static_cast<double>(w_cur);
            int ind = thr < run ? 0 : -1;
            for (int j = 0; j < NK; ++j) {
                run += static_cast<double>(weight(lw_tab[j * blockDim.x + threadIdx.x]));
                if (ind < 0 && thr < run) ind = j + 1;
            }
            if (ind > 0) {   // :175-179 — rebuild the chosen candidate (a pure function of (chain, step, j)); the cached gradient is NOT refreshed (B-6)
                const int j = ind - 1;
                if constexpr (GIP) {
                    WordStream ws(R.rk, stream, i, kSlotGeneric + 64u * static_cast<uint32_t>(j));
                    (void)dist_forward<D>(K.ipg, ws, theta);
                    float eps_s[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) eps_s[k] = ws.normal();
                    model_simulate<D, false>(K.model, theta, eps_s, y);
                } else {
                    float zc[kGroups * 4];
#pragma unroll
                    for (int g = 0; g < kGroups; ++g) {
                        const uint4 w = stream.block(R.rk, i, kSlotNormal + 8u + j * kGroups + g);
                        box_muller(w.x, w.y, zc[4 * g], zc[4 * g + 1]);
                        box_muller(w.z, w.w, zc[4 * g + 2], zc[4 * g + 3]);
                    }
                    float eps_p[D], eps_s[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        eps_p[k] = zc[k];
                        eps_s[k] = zc[D + k];
                    }
                    gauss_forward<D, false>(K.ip, eps_p, theta);
                    model_simulate<D, false>(K.model, theta, eps_s, y);
                }
                lw_old = lw_tab[j * blockDim.x + threadIdx.x];
#pragma unroll
                for (int k = 0; k < D; ++k) changed |= theta[k] != prev[k];
            }
        }

        // ================= MALA local move, GLMALA.py:182-200 =================
        const unsigned pend = __ballot_sync(0xffffffffu, is_local);
        if (pend != 0u) {   // warp-uniform
            float z[D], eps_s[D], theta_p[D], grad_p[D];
            float u_a = 0.0f, lq_fwd = 0.0f;
            if (is_local) {
                float zz[kGroups * 4];
                box_muller(w0.x, w0.y, zz[0], zz[1]);
                box_muller(w0.z, w0.w, zz[2], zz[3]);
#pragma unroll
                for (int g = 1; g < kGroups; ++g) {
                    const uint4 w = stream.block(R.rk, i, kSlotNormal + g - 1);
                    box_muller(w.x, w.y, zz[4 * g], zz[4 * g + 1]);
                    box_muller(w.z, w.w, zz[4 * g + 2], zz[4 * g + 3]);
                }
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    z[k] = zz[k];
                    eps_s[k] = zz[D + k];
                }
                u_a = __uint2float_rn(step_block_ua(w0)) * 0x1p-24f;
                float zf[D];
                lq_fwd = gauss_forward<D, false>(K.unit, z, zf);   // Local_proposal_forward, :25-44
            }
#pragma unroll
            for (int k = 0; k < D; ++k) theta_p[k] = theta[k];
            // pass 0 (only chains whose grad_logABC_Theta_old is still None, :183-184): gradient at theta;
            // pass 1: theta' from the cached gradient (:186), gradient at theta' (:187) — one call site
            const unsigned need0 = __ballot_sync(0xffffffffu, is_local && !have_grad);
#pragma unroll 1
            for (int pass = need0 != 0u ? 0 : 1; pass < 2; ++pass) {
                if (pass == 1 && is_local) {
#pragma unroll
                    for (int k = 0; k < D; ++k) theta_p[k] = fmaf(grad[k], half_tau2, fmaf(z[k], tau, theta[k]));   // :43
                }
                unsigned todo = pass == 0 ? need0 : pend;
                float sums[D][4], cpm[D][2];
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    sums[k][0] = sums[k][1] = sums[k][2] = sums[k][3] = 0.0f;
                    cpm[k][0] = cpm[k][1] = 0.0f;
                }
                while (todo != 0u) {
                    const int src = __ffs(todo) - 1;
                    todo &= todo - 1u;
                    float th_s[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) th_s[k] = __shfl_sync(0xffffffffu, theta_p[k], src);
                    const Stream ss = chain_stream(R, warp_chain0 + src);
                    warp_gradient_sums<D, FAMILY>(K, R.rk, ss, i, pass == 0 ? kSlotGrad0 : kSlotGrad, th_s, lane, lane == src, sums, cpm);
                }
                const bool mine = pass == 0 ? (is_local && !have_grad) : is_local;
                if (mine) {
                    float gout[D];
                    gradient_from_sums<D, GPRIOR>(K, prior, theta_p, sums, cpm, gout);
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        if (pass == 0) grad[k] = gout[k];
                        grad_p[k] = gout[k];
                    }
                    have_grad = true;
                }
            }
            if (is_local) {
                float y_p[D], rr[D];
                model_simulate<D, false>(K.model, theta_p, eps_s, y_p);   // :188-189
#pragma unroll
                for (int k = 0; k < D; ++k) rr[k] = ((theta[k] - theta_p[k]) - grad_p[k] * half_tau2) * inv_tau;   // log_proposal, :97-116
                const float pp = prior_log_prob<D, false, GPRIOR>(K.model, prior, theta_p), kp = model_log_kernel<D, false>(K.model, y_p);
                const float lr = gauss_log_prob<D, false>(K.unit, rr);
                const float po = prior_log_prob<D, false, GPRIOR>(K.model, prior, theta), ko = model_log_kernel<D, false>(K.model, y);
                const float log_acc = ((pp + kp) - (po + ko)) + (lr - lq_fwd);   // :190-193
                if (log_approx(u_a) < log_acc) {   // :194-199
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        theta[k] = theta_p[k];
                        y[k] = y_p[k];
                        grad[k] = grad_p[k];
                    }
                    wide = true;
                    changed = true;
                }
            }
        }

        stats.update(is_global, changed, theta, prev);
        writer.put(R, i, theta);
        writer.maybe_flush(R, i);
    }
    writer.finish(R);

    if (active) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            R.theta[static_cast<int64_t>(chain) * D + k] = theta[k];
            R.y[static_cast<int64_t>(chain) * D + k] = y[k];
            s64[GLABC_S64_THETA + k] = static_cast<double>(theta[k]);
            s64[GLABC_S64_Y + k] = static_cast<double>(y[k]);
            s64[GLABC_S64_GRAD + k] = static_cast<double>(grad[k]);
        }
        s64[GLABC_S64_LOGW] = static_cast<double>(lw_old);
        aux[GLABC_AUX_LOCAL] = local ? 1.0f : 0.0f;
        aux[GLABC_AUX_WIDE] = wide ? 1.0f : 0.0f;
        aux[GLABC_AUX_LW_WIDE] = lw_wide ? 1.0f : 0.0f;
        aux[GLABC_AUX_HAVE_GRAD] = have_grad ? 1.0f : 0.0f;
        if (R.stats != nullptr)
            stats.store(R.stats + static_cast<int64_t>(chain) * GLABC_NSTATS(D), R.last_step + 1u - R.first_step);
    }
}

template <int D, int FAMILY, int LAYOUT, bool GIP>
static void launch_mala_fast_gip(const MalaConsts& K, const DistConsts& prior, const RunParams& R, int grid, int block, size_t smem,
                                 cudaStream_t st)
{
    if (generic_prior(prior)) k_mala_fast<D, FAMILY, LAYOUT, GIP, true><<<grid, block, smem, st>>>(K, R, prior);
    else k_mala_fast<D, FAMILY, LAYOUT, GIP, false><<<grid, block, smem, st>>>(K, R, prior);
}

template <int D, int FAMILY, int LAYOUT>
static cudaError_t launch_mala_fast_one(const MalaConsts& K, const DistConsts& prior, const RunParams& R, cudaStream_t st)
{
    using Writer = typename WriterFor<D, LAYOUT>::type;
    constexpr int block = GLABC_MALA_BLOCK;   // one chain per thread
    const int grid = (R.n_chains + block - 1) / block;
    const size_t smem = sizeof(float) * (static_cast<size_t>(Writer::smem_floats_per_warp) * (block / 32) +
                                         static_cast<size_t>(R.n_candidates) * block);
    if (K.ip_generic) launch_mala_fast_gip<D, FAMILY, LAYOUT, true>(K, prior, R, grid, block, smem, st);
    else launch_mala_fast_gip<D, FAMILY, LAYOUT, false>(K, prior, R, grid, block, smem, st);
    return cudaGetLastError();
}

template <int D, int FAMILY>
static cudaError_t launch_mala_fast(const MalaConsts& K, const DistConsts& prior, const RunParams& R, cudaStream_t st)
{
    switch (R.trace_layout) {
    case GLABC_TRACE_NONE: return launch_mala_fast_one<D, FAMILY, GLABC_TRACE_NONE>(K, prior, R, st);
    case GLABC_TRACE_TIME_MAJOR: return launch_mala_fast_one<D, FAMILY, GLABC_TRACE_TIME_MAJOR>(K, prior, R, st);
    case GLABC_TRACE_CHAIN_MAJOR: return launch_mala_fast_one<D, FAMILY, GLABC_TRACE_CHAIN_MAJOR>(K, prior, R, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace glabc
