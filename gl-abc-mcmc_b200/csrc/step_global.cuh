// K1 — the GlobalMCMC chain step, fused: branch draw, local random-walk / global independence
// proposal, simulator draw, discrepancy, Gaussian ABC log-kernel, prior, Metropolis–Hastings
// accept/reject, trace row and statistics.  Reference: GlobalMCMC.py:37-68 (SURVEY.md A.1).
//
// One thread = one chain; the chain state (theta, y, cached log-target) stays in registers for the
// whole launch.  The step is split in two phases:
//   prepare(i)  everything that does not depend on the chain state: Philox blocks, Box-Muller,
//               the branch coin, log(U_a), the global candidate / local increment, the simulator
//               noise, log q(theta') — pure ILP, no loop-carried dependence;
//   advance()   the short state-dependent chain: theta' -> y' -> log-target' -> accept -> select.
// The native-RNG loop is software-pipelined over batches of 4 steps: the prepare() of batch b+1 is
// issued in the same straight-line block as the advance() of batch b, so the scheduler overlaps
// the long RNG latency chains with the dependent chain even at 3-4 warps per scheduler
// (65,536 chains = 13.8 warps/SM).  Both branches differ only in how theta' is formed and in the
// proposal-density correction, so the step is branch-free (selects / a 0-1 mask).
#pragma once
#include "launch.cuh"
#include "sampler_common.cuh"

namespace glabc {

struct GlobalConsts {
    ModelConsts model;
    GaussConsts lp;  // Local_Proposal
    GaussConsts gp;  // Global_Proposal
};

// state-independent inputs of one step
template <int D>
struct StepInputs {
    bool is_global;   // STRICT path only (the FAST path works on the 0/1 masks below: no predicates
                      // to carry across the software pipeline, counters on the FMA pipe)
    float keep;       // 0 for a global move, 1 for a local one: theta' = keep*theta + cand
    float glob;       // 1 - keep
    float cand[D];    // global: Global_Proposal.forward() sample; local: Local_Proposal.sample()
    float noise[D];   // noise_loc + noise_scale*eps_sim   (Mixture.py:19-23)
    float lq_p;       // STRICT: log q_global(theta') from eps (distribution.py:171)
    float log_w;      // STRICT: log(U_a);  FAST: log(U_a) + glob*lq_p (the accept test with the
                      // state-independent part of the proposal correction moved to the left side)
    float raw[2 * D + 2];  // the draws themselves (tape layout) — only kept alive when dumped
};

template <int D, bool STRICT, bool KEEP_RAW>
__device__ __forceinline__ StepInputs<D> make_inputs(const GlobalConsts& K, bool is_global, float u_b, float u_a,
                                                    const float (&eps_p)[D], const float (&eps_s)[D])
{
    StepInputs<D> in;
    in.is_global = is_global;
    in.keep = is_global ? 0.0f : 1.0f;
    in.glob = 1.0f - in.keep;
    if constexpr (STRICT) {
        float th_g[D], th_l[D];
        in.lq_p = gauss_forward<D, true>(K.gp, eps_p, th_g);   // GlobalMCMC.py:40
        (void)gauss_forward<D, true>(K.lp, eps_p, th_l);        // GlobalMCMC.py:56 (sample part)
#pragma unroll
        for (int k = 0; k < D; ++k) {
            in.cand[k] = is_global ? th_g[k] : th_l[k];
            in.noise[k] = __fadd_rn(K.model.noise_loc[k], __fmul_rn(K.model.noise_scale[k], eps_s[k]));
        }
        in.log_w = logf(u_a);                                   // GlobalMCMC.py:47,62
    } else {
        // both candidates from the constant bank, then a select (prepare() still has the predicate)
        float q = 0.0f;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float cg = fmaf(K.gp.scale[k], eps_p[k], K.gp.loc[k]);
            const float cl = fmaf(K.lp.scale[k], eps_p[k], K.lp.loc[k]);
            in.cand[k] = is_global ? cg : cl;
            in.noise[k] = fmaf(K.model.noise_scale[k], eps_s[k], K.model.noise_loc[k]);
            q = fmaf(eps_p[k], eps_p[k], q);
        }
        in.lq_p = fmaf(-0.5f, q, K.gp.c_fast);
        in.log_w = fmaf(in.glob, in.lq_p, log_approx(u_a));
    }
    if constexpr (KEEP_RAW) {
        in.raw[0] = u_b;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            in.raw[1 + k] = eps_p[k];
            in.raw[1 + D + k] = eps_s[k];
        }
        in.raw[1 + 2 * D] = u_a;
    }
    return in;
}

// replay: the tape holds the reference's own draws, [step][slot][chain]
template <int D, bool STRICT>
__device__ __forceinline__ StepInputs<D> inputs_from_tape(const GlobalConsts& K, const RunParams& r,
                                                         uint32_t step_in_launch, int32_t chain)
{
    constexpr int kSlots = GLABC_TAPE_GLOBAL_SLOTS(D, D);
    const float* t = r.tape32 + (static_cast<int64_t>(step_in_launch) * kSlots) * r.n_chains + chain;
    float eps_p[D], eps_s[D];
    const float u_b = __ldg(t);
#pragma unroll
    for (int k = 0; k < D; ++k) eps_p[k] = __ldg(t + static_cast<int64_t>(1 + k) * r.n_chains);
#pragma unroll
    for (int k = 0; k < D; ++k) eps_s[k] = __ldg(t + static_cast<int64_t>(1 + D + k) * r.n_chains);
    const float u_a = __ldg(t + static_cast<int64_t>(1 + 2 * D) * r.n_chains);
    // GlobalMCMC.py:39 — float32 compare against the float32-rounded threshold, strict <
    return make_inputs<D, STRICT, false>(K, u_b < r.gf, u_b, u_a, eps_p, eps_s);
}

// native: ONE Philox block per step carries the four normals, U_b and U_a of a d<=2 step
// (bit budget in philox.cuh); d>2 draws its remaining normals from extra blocks.
template <int D, bool STRICT, bool KEEP_RAW>
__device__ __forceinline__ StepInputs<D> inputs_native(const GlobalConsts& K, const RunParams& r, const RoundKeys& rk,
                                                      const Stream& s, uint32_t step)
{
    constexpr int kGroups = (2 * D + 3) / 4;
    float z[kGroups * 4];
    const uint4 w0 = s.block(rk, step, kSlotStep);
    box_muller(w0.x, w0.y, z[0], z[1]);
    box_muller(w0.z, w0.w, z[2], z[3]);
#pragma unroll
    for (int g = 1; g < kGroups; ++g) {
        const uint4 w = s.block(rk, step, kSlotNormal + g - 1);
        box_muller(w.x, w.y, z[4 * g + 0], z[4 * g + 1]);
        box_muller(w.z, w.w, z[4 * g + 2], z[4 * g + 3]);
    }
    float eps_p[D], eps_s[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        eps_p[k] = z[k];
        eps_s[k] = z[D + k];
    }
    const uint32_t ub = step_block_ub(w0);  // 16-bit U_b in the top half: U_b < gf is an integer compare
    const bool is_global = (ub < r.gf_thr_hi) || r.gf_all_global;
    const float u_a = __uint2float_rn(step_block_ua(w0)) * 0x1p-24f;  // torch.rand's float32 grid (B-16)
    return make_inputs<D, STRICT, KEEP_RAW>(K, is_global, KEEP_RAW ? __uint2float_rn(ub >> 16) * 0x1p-16f : 0.0f, u_a, eps_p, eps_s);
}

template <int D>
struct ChainState {
    float theta[D], y[D];
    float prior, kern;  // cached log prior(theta), log kernel(y): the reference recomputes them every
                        // step from the same inputs (GlobalMCMC.py:46,61), so caching is bit-identical
};

struct StepRecord {  // replay-mode per-step quantities
    float prior_p, kern_p, log_acc;
    bool accept;
};

template <int D, int FAMILY, bool STRICT>
__device__ __forceinline__ StepRecord advance(const GlobalConsts& K, ChainState<D>& st, ChainStats<D>& stats,
                                              const StepInputs<D>& in)
{
    float theta_p[D], y_p[D];
    if constexpr (!STRICT) {
        // FAST: st.prior holds log prior + log kernel of the current state, st.kern is unused.
        float qp = 0.0f, sk = 0.0f, qo = 0.0f;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            theta_p[k] = fmaf(in.keep, st.theta[k], in.cand[k]);
            y_p[k] = (FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(theta_p[k]) : theta_p[k]) + in.noise[k];
            const float dy = y_p[k] - K.model.y_obs[k];
            sk = fmaf(dy, dy, sk);
            const float rp = fmaf(theta_p[k], K.model.prior.inv_scale[k], K.model.prior.nloc_inv[k]);
            qp = fmaf(rp, rp, qp);
            const float ro = fmaf(st.theta[k], K.gp.inv_scale[k], K.gp.nloc_inv[k]);
            qo = fmaf(ro, ro, qo);
        }
        // log target of the candidate, and log q_global(theta_old) for the independence correction
        const float tgt_p = fmaf(K.model.kern_fast_m, sk, fmaf(-0.5f, qp, K.model.prior.c_fast + K.model.kern_fast_c));
        const float lq_old = fmaf(-0.5f, qo, K.gp.c_fast);
        const float rhs = fmaf(in.glob, lq_old, tgt_p - st.prior);
        const bool accept = in.log_w < rhs;  // log U + glob*lq' < target' - target + glob*lq_old
        float prev[D];
#pragma unroll
        for (int k = 0; k < D; ++k) {
            prev[k] = st.theta[k];
            st.theta[k] = accept ? theta_p[k] : st.theta[k];
            st.y[k] = accept ? y_p[k] : st.y[k];
        }
        st.prior = accept ? tgt_p : st.prior;
        stats.update_masked(in.glob, accept ? 1.0f : 0.0f, st.theta, prev);
        // per-step record (replay only; dead code in the native kernels)
        return StepRecord{fmaf(-0.5f, qp, K.model.prior.c_fast), fmaf(K.model.kern_fast_m, sk, K.model.kern_fast_c),
                          fmaf(-in.glob, in.lq_p, rhs), accept};
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        theta_p[k] = in.is_global ? in.cand[k] : __fadd_rn(in.cand[k], st.theta[k]);  // :40 / :56
        const float mean = FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(theta_p[k]) : theta_p[k];
        y_p[k] = __fadd_rn(mean, in.noise[k]);                                         // :41 / :57
    }
    const float prior_p = model_prior<D, STRICT>(K.model, theta_p);         // :44 / :60
    const float kern_p = model_log_kernel<D, STRICT>(K.model, y_p);
    const float lq_old = gauss_log_prob<D, STRICT>(K.gp, st.theta);         // :45
    float log_acc;
    if constexpr (STRICT) {
        // left-to-right, exactly as written at GlobalMCMC.py:44-46 and :60-61
        const float base = __fadd_rn(prior_p, kern_p);
        const float g = __fsub_rn(__fsub_rn(__fsub_rn(__fadd_rn(base, lq_old), in.lq_p), st.prior), st.kern);
        const float l = __fsub_rn(__fsub_rn(base, st.prior), st.kern);
        log_acc = in.is_global ? g : l;
    } else {
        const float corr = in.is_global ? lq_old - in.lq_p : 0.0f;
        log_acc = (prior_p + kern_p) + (corr - (st.prior + st.kern));
    }
    const bool accept = in.log_w < log_acc;  // :49 strict <, NaN rejects (B-17)

    float prev[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        prev[k] = st.theta[k];
        st.theta[k] = accept ? theta_p[k] : st.theta[k];
        st.y[k] = accept ? y_p[k] : st.y[k];
    }
    st.prior = accept ? prior_p : st.prior;
    st.kern = accept ? kern_p : st.kern;
    stats.update(in.is_global, accept, st.theta, prev);
    return StepRecord{prior_p, kern_p, log_acc, accept};
}

template <int D, int FAMILY, bool STRICT, bool REPLAY, int LAYOUT, bool DUMP>
__global__ void __launch_bounds__(256) k_global_mcmc(const __grid_constant__ GlobalConsts K,
                                                     const __grid_constant__ RunParams R)
{
    using Writer = typename WriterFor<D, LAYOUT, true>::type;
    extern __shared__ float smem[];
    const int32_t chain = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = chain < R.n_chains;
    const int32_t cidx = active ? chain : R.n_chains - 1;  // tail lanes shadow the last chain, never store

    ChainState<D> st;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        st.theta[k] = R.theta[static_cast<int64_t>(cidx) * D + k];
        st.y[k] = R.y[static_cast<int64_t>(cidx) * D + k];
    }
    st.prior = model_prior<D, STRICT>(K.model, st.theta);
    st.kern = model_log_kernel<D, STRICT>(K.model, st.y);
    if constexpr (!STRICT) st.prior += st.kern;  // FAST carries the sum

    Writer writer(R, cidx, active, smem + (threadIdx.x >> 5) * Writer::smem_floats_per_warp);
    if (R.write_row0) {
        writer.put(R, R.first_step - 1u, st.theta);
        writer.maybe_flush(R, R.first_step - 1u);
    }
    ChainStats<D> stats;

    if constexpr (REPLAY) {
        for (uint32_t i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
            const StepInputs<D> in = inputs_from_tape<D, STRICT>(K, R, i - R.first_step, cidx);
            const StepRecord rec = advance<D, FAMILY, STRICT>(K, st, stats, in);
            writer.put(R, i, st.theta);  // :53 / :68
            writer.maybe_flush(R, i);
            if (R.debug != nullptr && active) {
                float* g = R.debug + static_cast<int64_t>(i - R.first_step) * GLABC_DEBUG_SLOTS * R.n_chains + chain;
                g[0] = static_cast<float>(static_cast<int>(in.is_global) | (static_cast<int>(rec.accept) << 1));
                g[static_cast<int64_t>(1) * R.n_chains] = rec.prior_p;
                g[static_cast<int64_t>(2) * R.n_chains] = rec.kern_p;
                g[static_cast<int64_t>(3) * R.n_chains] = rec.log_acc;
            }
        }
    } else {
        const Stream stream = chain_stream(R, cidx);
        auto dump = [&](uint32_t i, const StepInputs<D>& in) {
            if constexpr (DUMP) {
                if (R.tape_dump != nullptr && active) {
                    constexpr int kSlots = GLABC_TAPE_GLOBAL_SLOTS(D, D);
                    float* t = R.tape_dump + static_cast<int64_t>(i - R.first_step) * kSlots * R.n_chains + chain;
#pragma unroll
                    for (int k = 0; k < kSlots; ++k) t[static_cast<int64_t>(k) * R.n_chains] = in.raw[k];
                }
            }
        };
        auto single = [&](uint32_t i) {  // unpipelined step for the ragged head / tail of the range
            const StepInputs<D> in = inputs_native<D, STRICT, DUMP>(K, R, R.rk, stream, i);
            advance<D, FAMILY, STRICT>(K, st, stats, in);
            writer.put(R, i, st.theta);
            writer.maybe_flush(R, i);
            dump(i, in);
        };
        auto prepare4 = [&](uint32_t i, StepInputs<D> (&b)[4]) {
#pragma unroll
            for (int k = 0; k < 4; ++k) b[k] = inputs_native<D, STRICT, DUMP>(K, R, R.rk, stream, i + k);
        };
        // The steady loop runs whole trace tiles: 32 rows for the chain-major writers, whose tiles end on
        // absolute rows i % 32 == 31, one 8-step body for the others.  Inside a tile a row's slot is
        // the loop position, so the chain-major put is one shared-memory store at a fixed offset from
        // the body's base, with no row bookkeeping, and the tile ends in one unconditional flush.
        constexpr bool kTiled = LAYOUT == GLABC_TRACE_CHAIN_MAJOR;
        constexpr uint32_t kTile = kTiled ? 32u : 8u;
        auto advance4 = [&](uint32_t i, uint32_t slot, const StepInputs<D> (&b)[4]) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                advance<D, FAMILY, STRICT>(K, st, stats, b[k]);
                if constexpr (kTiled) writer.put_slot(slot + k, st.theta);
                else writer.put(R, i + k, st.theta);
                dump(i + k, b[k]);
            }
        };

        if (R.last_step >= R.first_step) {
            uint32_t i = R.first_step;
            while (i <= R.last_step && (i % kTile)) single(i++);  // head, up to the first tile boundary
            if (i + (kTile - 1u) <= R.last_step) {
                // ping-pong between two input buffers so no registers are copied between batches:
                // prepare() of the next batch is independent of the chain state and overlaps with the
                // dependent advance() chain of the current one, across tile edges too (the last
                // tile's look-ahead batch is computed and dropped)
                StepInputs<D> a[4], b[4];
                prepare4(i, a);
                do {
#pragma unroll 1
                    for (uint32_t s = 0; s < kTile; s += 8u) {
                        prepare4(i + s + 4u, b);
                        advance4(i + s, s, a);
                        prepare4(i + s + 8u, a);
                        advance4(i + s + 4u, s + 4u, b);
                    }
                    if constexpr (kTiled) writer.flush_tile(R, i);
                    i += kTile;
                } while (i + (kTile - 1u) <= R.last_step);
            }
            while (i <= R.last_step) single(i++);  // tail, < kTile steps
        }
    }
    writer.finish(R);

    if (active) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            R.theta[static_cast<int64_t>(chain) * D + k] = st.theta[k];
            R.y[static_cast<int64_t>(chain) * D + k] = st.y[k];
        }
        if (R.stats != nullptr)
            stats.store(R.stats + static_cast<int64_t>(chain) * GLABC_NSTATS(D), R.last_step + 1u - R.first_step);
    }
}

template <int D, int FAMILY, bool STRICT, bool REPLAY, int LAYOUT, bool DUMP>
static cudaError_t launch_one(const GlobalConsts& K, const RunParams& R, int block, cudaStream_t st)
{
    using Writer = typename WriterFor<D, LAYOUT, true>::type;
    const int grid = (R.n_chains + block - 1) / block;
    const size_t smem = sizeof(float) * Writer::smem_floats_per_warp * (block / 32);
    auto kern = k_global_mcmc<D, FAMILY, STRICT, REPLAY, LAYOUT, DUMP>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
    }
    RunParams P = R;
    P.trace_runs_16b = LAYOUT == GLABC_TRACE_CHAIN_MAJOR && D == 2 && chain_major_runs_16b(R);
    kern<<<grid, block, smem, st>>>(K, P);
    return cudaGetLastError();
}

template <int D, int FAMILY, bool STRICT>
static cudaError_t launch_mode(const GlobalConsts& K, const RunParams& R, bool replay, int layout, int block, cudaStream_t st)
{
    if (replay) {  // parity mode: time-major or chain-major trace, no dump
        switch (layout) {
        case GLABC_TRACE_NONE: return launch_one<D, FAMILY, STRICT, true, GLABC_TRACE_NONE, false>(K, R, block, st);
        case GLABC_TRACE_TIME_MAJOR: return launch_one<D, FAMILY, STRICT, true, GLABC_TRACE_TIME_MAJOR, false>(K, R, block, st);
        case GLABC_TRACE_CHAIN_MAJOR: return launch_one<D, FAMILY, STRICT, true, GLABC_TRACE_CHAIN_MAJOR, false>(K, R, block, st);
        }
        return cudaErrorInvalidValue;
    }
    if (R.tape_dump != nullptr) {  // diagnostic variant that also stores its draws
        if (layout != GLABC_TRACE_TIME_MAJOR) return cudaErrorInvalidValue;
        return launch_one<D, FAMILY, STRICT, false, GLABC_TRACE_TIME_MAJOR, true>(K, R, block, st);
    }
    switch (layout) {
    case GLABC_TRACE_NONE: return launch_one<D, FAMILY, STRICT, false, GLABC_TRACE_NONE, false>(K, R, block, st);
    case GLABC_TRACE_TIME_MAJOR: return launch_one<D, FAMILY, STRICT, false, GLABC_TRACE_TIME_MAJOR, false>(K, R, block, st);
    case GLABC_TRACE_CHAIN_MAJOR: return launch_one<D, FAMILY, STRICT, false, GLABC_TRACE_CHAIN_MAJOR, false>(K, R, block, st);
    case GLABC_TRACE_EVENTS: return launch_one<D, FAMILY, STRICT, false, GLABC_TRACE_EVENTS, false>(K, R, block, st);
    }
    return cudaErrorInvalidValue;
}

template <int D>
cudaError_t launch_global_mcmc_dim(const ModelConsts& model, const GaussConsts& lp, const GaussConsts& gp,
                                   const RunParams& R, bool strict, bool replay, int layout, int block, cudaStream_t st)
{
    GlobalConsts K{model, lp, gp};
    return with_family(model.family, [&](auto f) {
        return strict ? launch_mode<D, f, true>(K, R, replay, layout, block, st)
                      : launch_mode<D, f, false>(K, R, replay, layout, block, st);
    });
}

}  // namespace glabc
