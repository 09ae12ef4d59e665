// K2 — the GLMCMC chain step: with probability gf an iSIR global move (K fresh candidates from the
// importance proposal + the current state, un-shifted importance weights, inverse-CDF resample),
// otherwise a local random-walk Metropolis–Hastings move.  Reference: GLMCMC.py:58-104 and
// weight_sampling GLMCMC.py:7-22 (SURVEY.md A.2).
//
// One thread = one chain.  The K candidates of a step are independent of the chain state and of
// each other, so they are generated two at a time (ILP) and parked in shared memory as
// [slot][field][thread] (conflict-free: consecutive lanes), which also makes "take candidate ind"
// a plain indexed load instead of a K-way select chain.  K is a run-time parameter (1..16).
// The global/local choice is a per-thread coin and a warp almost always contains both kinds
// (gf = 0.9: P(all 32 lanes agree) = 3 %), so both arms are evaluated branch-free and the state
// update is predicated.
#pragma once
#include "launch.cuh"
#include "sampler_common.cuh"

namespace glabc {

struct IsirConsts {
    ModelConsts model;
    GaussConsts lp;  // Local_Proposal
    GaussConsts ip;  // Importance_Proposal
};

// per-thread view of the shared-memory candidate table: slot s in [0, K], fields: 0 weight,
// 1 log-weight, 2 log prior, 3 log kernel, 4.. theta[D], 4+D.. x[D]
template <int D>
struct CandTable {
    static constexpr int kFields = 4 + 2 * D;
    float* base;      // + threadIdx.x already applied
    uint32_t stride;  // blockDim.x
    __device__ __forceinline__ float& at(int slot, int field) const { return base[(slot * kFields + field) * stride]; }
};

// exp of a log-weight, un-shifted, denormal results kept (GLMCMC.py:78, SURVEY.md B-1: during burn-in
// every weight of a row can sit below 1e-38 and the reference still resamples among them; only a row
// that underflows to exact zeros gives `None`).  STRICT = expf; FAST = MUFU.EX2 without .ftz.
template <bool STRICT>
__device__ __forceinline__ float weight_exp(float lw)
{
    float w;
    if constexpr (STRICT) {
        w = expf(lw);
    } else {
        asm("ex2.approx.f32 %0, %1;" : "=f"(w) : "f"(lw * 1.4426950408889634f));
    }
    return (w != w) ? 0.0f : w;  // GLMCMC.py:80-81 NaN -> 0
}

// torch.sum over n contiguous float32 read from the table (field 0 of slots 0..n-1): ATen row_sum
// (four interleaved partials) for n < 16, the 16-lane vectorised path for n >= 16 (SURVEY.md B-3)
template <int D>
__device__ __forceinline__ float torch_sum_table(const CandTable<D>& t, int n)
{
    if (n >= 16) {
        float lane[16];
#pragma unroll
        for (int l = 0; l < 16; ++l) lane[l] = t.at(l, 0);  // one full vector (n <= 17 here)
        float acc = 0.0f;
        for (int i = 16; i < n; ++i) acc = __fadd_rn(acc, t.at(i, 0));
#pragma unroll
        for (int l = 0; l < 16; ++l) acc = __fadd_rn(acc, lane[l]);
        return acc;
    }
    float p[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    const int rows = n >> 2;
    for (int r = 0; r < rows; ++r)
#pragma unroll
        for (int k = 0; k < 4; ++k) p[k] = __fadd_rn(p[k], t.at(r * 4 + k, 0));
    for (int i = rows * 4; i < n; ++i) p[0] = __fadd_rn(p[0], t.at(i, 0));
#pragma unroll
    for (int k = 1; k < 4; ++k) p[0] = __fadd_rn(p[0], p[k]);
    return p[0];
}

// one importance candidate from its normals: theta_j, x_j, log-weight, weight -> table slot
template <int D, int FAMILY, bool STRICT>
__device__ __forceinline__ void make_candidate(const IsirConsts& K, const float (&eps_p)[D], const float (&eps_s)[D],
                                               const CandTable<D>& tab, int slot)
{
    float th[D], x[D];
    const float lq = gauss_forward<D, STRICT>(K.ip, eps_p, th);  // GLMCMC.py:66
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const float mean = FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(th[k]) : th[k];
        if constexpr (STRICT) {
            x[k] = __fadd_rn(mean, __fadd_rn(K.model.noise_loc[k], __fmul_rn(K.model.noise_scale[k], eps_s[k])));
        } else {
            x[k] = mean + fmaf(K.model.noise_scale[k], eps_s[k], K.model.noise_loc[k]);  // GLMCMC.py:71
        }
    }
    const float prior = model_prior<D, STRICT>(K.model, th);
    const float kern = model_log_kernel<D, STRICT>(K.model, x);
    const float lw = STRICT ? __fsub_rn(__fadd_rn(prior, kern), lq) : (prior + kern) - lq;  // GLMCMC.py:72-74
    tab.at(slot, 0) = weight_exp<STRICT>(lw);
    tab.at(slot, 1) = lw;
    tab.at(slot, 2) = prior;
    tab.at(slot, 3) = kern;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        tab.at(slot, 4 + k) = th[k];
        tab.at(slot, 4 + D + k) = x[k];
    }
}


// ---- software-pipelined form of the native FAST loop (NKT > 0) --------------------------------------------------
// Everything of step i + 1 that does not depend on the chain state — the step's Philox blocks, the K candidates, the
// local proposal's increment and simulator noise, log U — is computed IN REGISTERS in the same straight-line block as
// the short dependent part of step i (weight of the current state, resample, local MH test, state update), so the
// scheduler fills the dependent chain's latency holes at 3-4 warps per scheduler.  The candidates' weights stay in
// registers; the fields a switch needs (theta, x, log-weight, prior + kernel) are parked in a single-buffered
// shared-memory table AFTER step i has read its own row, which keeps "take candidate ind" one indexed load and the
// table small enough (7.5 KB per 64 chains) for every CTA of a 65,536-chain launch to be resident at once.
template <int D, int NK>
struct IsirStepIn {
    bool is_global;
    float log_w;      // log U_a of the local MH test
    float z_l[D];     // Local_Proposal increment (state-independent)
    float n_l[D];     // simulator noise of the local candidate
    double u64;       // resampling uniform
    float w[NK];      // importance weights of the K candidates
};

template <int D, int NK>
struct IsirCands {    // what a switch to candidate j needs
    float lw[NK], pk[NK], th[NK][D], x[NK][D];
};

// pipelined table: slot j in [0, K), fields 0 log-weight, 1 prior + kernel, 2.. theta[D], 2+D.. x[D]
template <int D>
struct TakeTable {
    static constexpr int kFields = 2 + 2 * D;
    float* base;      // + threadIdx.x already applied
    uint32_t stride;  // blockDim.x
    __device__ __forceinline__ float& at(int slot, int field) const { return base[(slot * kFields + field) * stride]; }
};

template <int D, int FAMILY, int NK>
__device__ __forceinline__ void isir_prepare(const IsirConsts& K, const RunParams& R, const Stream& stream, uint32_t i,
                                             IsirStepIn<D, NK>& in, IsirCands<D, NK>& c)
{
    constexpr int kGroups = (2 * D + 3) / 4;
    const uint4 w0 = stream.block(R.rk, i, kSlotStep);
    float z[kGroups * 4];
    box_muller(w0.x, w0.y, z[0], z[1]);
    box_muller(w0.z, w0.w, z[2], z[3]);
#pragma unroll
    for (int g = 1; g < kGroups; ++g) {
        const uint4 w = stream.block(R.rk, i, kSlotNormal + g - 1);
        box_muller(w.x, w.y, z[4 * g], z[4 * g + 1]);
        box_muller(w.z, w.w, z[4 * g + 2], z[4 * g + 3]);
    }
    float eps_lp[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        eps_lp[k] = z[k];
        in.n_l[k] = fmaf(K.model.noise_scale[k], z[D + k], K.model.noise_loc[k]);
    }
    (void)gauss_forward<D, false>(K.lp, eps_lp, in.z_l);
    in.is_global = (step_block_ub(w0) < R.gf_thr_hi) || R.gf_all_global;
    const uint32_t ua24 = step_block_ua(w0);
    in.log_w = log_approx(__uint2float_rn(ua24) * 0x1p-24f);
#pragma unroll
    for (int j = 0; j < NK; ++j) {
        float zz[kGroups * 4], eps_p[D];
        uint4 wj[kGroups];
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            wj[g] = stream.block(R.rk, i, kSlotNormal + 8u + j * kGroups + g);
            box_muller(wj[g].x, wj[g].y, zz[4 * g], zz[4 * g + 1]);
            box_muller(wj[g].z, wj[g].w, zz[4 * g + 2], zz[4 * g + 3]);
        }
        if (j == 0) {  // 53-bit resampling uniform: see the plain loop
            const uint64_t m53 = (static_cast<uint64_t>(ua24) << 29) | (static_cast<uint64_t>(step_block_ua(wj[0])) << 5) |
                                 static_cast<uint64_t>(step_block_ub(wj[0]) >> 27);
            in.u64 = static_cast<double>(m53) * 0x1p-53;
        }
#pragma unroll
        for (int k = 0; k < D; ++k) eps_p[k] = zz[k];
        const float lq = gauss_forward<D, false>(K.ip, eps_p, c.th[j]);  // GLMCMC.py:66
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float mean = FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(c.th[j][k]) : c.th[j][k];
            c.x[j][k] = mean + fmaf(K.model.noise_scale[k], zz[D + k], K.model.noise_loc[k]);  // GLMCMC.py:71
        }
        c.pk[j] = model_prior<D, false>(K.model, c.th[j]) + model_log_kernel<D, false>(K.model, c.x[j]);
        c.lw[j] = c.pk[j] - lq;                                          // GLMCMC.py:72-74
        in.w[j] = weight_exp<false>(c.lw[j]);
    }
}

template <int D, int NK>
__device__ __forceinline__ void isir_park(const IsirCands<D, NK>& c, const TakeTable<D>& tab)
{
#pragma unroll
    for (int j = 0; j < NK; ++j) {
        tab.at(j, 0) = c.lw[j];
        tab.at(j, 1) = c.pk[j];
#pragma unroll
        for (int k = 0; k < D; ++k) {
            tab.at(j, 2 + k) = c.th[j][k];
            tab.at(j, 2 + D + k) = c.x[j][k];
        }
    }
}

template <int D>
struct IsirState {
    float theta[D], y[D];
    float pk_old, lw_old;   // prior + kernel of the current state, its cached log-weight
    bool local;
};

template <int D, int FAMILY, int NK, class Writer>
__device__ __forceinline__ void isir_advance(const IsirConsts& K, const RunParams& R, uint32_t i, const IsirStepIn<D, NK>& in,
                                             const TakeTable<D>& tab, IsirState<D>& s, ChainStats<D>& stats, Writer& writer)
{
    // iSIR arm: weight of the current state, resample (GLMCMC.py:60-64,78-84)
    float lw_cur = s.lw_old;
    if (s.local) lw_cur = s.pk_old - gauss_log_prob<D, false>(K.ip, s.theta);
    const float w0 = weight_exp<false>(lw_cur);
    float S = w0;
#pragma unroll
    for (int j = 0; j < NK; ++j) S += in.w[j];
    const double thr = in.u64 * static_cast<double>(S);   // u < cumsum(w) / S  <=>  u * S < cumsum(w), in float64
    double run = static_cast<double>(w0);
    int ind = thr < run ? 0 : -1;
#pragma unroll
    for (int j = 0; j < NK; ++j) {
        run += static_cast<double>(in.w[j]);
        if (ind < 0 && thr < run) ind = j + 1;
    }
    const bool switch_g = in.is_global && ind > 0;
    const int take = switch_g ? ind - 1 : 0;   // always a valid row: the loads are unconditional, their use predicated
    float tk[TakeTable<D>::kFields];
#pragma unroll
    for (int f = 0; f < TakeTable<D>::kFields; ++f) tk[f] = tab.at(take, f);

    // local arm (GLMCMC.py:90-104)
    float th_l[D], y_l[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        th_l[k] = in.z_l[k] + s.theta[k];
        y_l[k] = (FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(th_l[k]) : th_l[k]) + in.n_l[k];
    }
    const float pk_l = model_prior<D, false>(K.model, th_l) + model_log_kernel<D, false>(K.model, y_l);
    const bool accept_l = !in.is_global && (in.log_w < pk_l - s.pk_old);

    float prev[D];
#pragma unroll
    for (int k = 0; k < D; ++k) prev[k] = s.theta[k];
    if (switch_g) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            s.theta[k] = tk[2 + k];
            s.y[k] = tk[2 + D + k];
        }
        lw_cur = tk[0];      // GLMCMC.py:86: cached log-weight of the taken candidate
        s.pk_old = tk[1];
    }
    if (accept_l) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            s.theta[k] = th_l[k];
            s.y[k] = y_l[k];
        }
        s.pk_old = pk_l;
    }
    if (in.is_global) {
        s.lw_old = lw_cur;
        s.local = false;     // GLMCMC.py:65
    }
    s.local = s.local || accept_l;  // GLMCMC.py:100
    stats.update(in.is_global, switch_g || accept_l, s.theta, prev);
    writer.put(R, i, s.theta);
    writer.maybe_flush(R, i);
}

// NKT > 0: K is a compile-time constant — the candidate loops unroll, so the K independent Philox / Box-Muller /
// log-weight chains of a global move interleave (ILP K) instead of running one after the other.
template <int D, int FAMILY, bool STRICT, bool REPLAY, int LAYOUT, bool DUMP, int NKT = 0>
__global__ void __launch_bounds__(256, 2) k_isir(const __grid_constant__ IsirConsts K, const __grid_constant__ RunParams R)
{
    using Writer = typename WriterFor<D, LAYOUT>::type;
    extern __shared__ float smem[];
    const int32_t chain = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = chain < R.n_chains;
    const int32_t cidx = active ? chain : R.n_chains - 1;
    const int NK = NKT > 0 ? NKT : R.n_candidates;

    // shared memory: [trace staging of every warp][candidate table of the block]
    float* stage = smem + (threadIdx.x >> 5) * Writer::smem_floats_per_warp;
    CandTable<D> tab{smem + (blockDim.x >> 5) * Writer::smem_floats_per_warp + threadIdx.x, blockDim.x};

    float theta[D], y[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        theta[k] = R.theta[static_cast<int64_t>(cidx) * D + k];
        y[k] = R.y[static_cast<int64_t>(cidx) * D + k];
    }
    float prior_old = model_prior<D, STRICT>(K.model, theta);
    float kern_old = model_log_kernel<D, STRICT>(K.model, y);
    float lw_old = R.aux[static_cast<int64_t>(cidx) * GLABC_AUX_SLOTS + GLABC_AUX_LOGW];
    bool local = R.aux[static_cast<int64_t>(cidx) * GLABC_AUX_SLOTS + GLABC_AUX_LOCAL] != 0.0f;

    Writer writer(R, cidx, active, stage);
    if (R.write_row0) {
        writer.put(R, R.first_step - 1u, theta);
        writer.maybe_flush(R, R.first_step - 1u);
    }
    ChainStats<D> stats;
    const Stream stream = chain_stream(R, cidx);
    const int tape_slots = 2 + NK * 2 * D;
    constexpr int kGroups = (2 * D + 3) / 4;  // Philox blocks per candidate

    constexpr bool PIPE = !STRICT && !REPLAY && !DUMP && NKT > 0;
    if constexpr (PIPE) {
        constexpr int NKC = NKT > 0 ? NKT : 1;
        const TakeTable<D> take{tab.base, blockDim.x};
        IsirState<D> s;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            s.theta[k] = theta[k];
            s.y[k] = y[k];
        }
        s.pk_old = prior_old + kern_old; s.lw_old = lw_old; s.local = local;
        if (R.last_step >= R.first_step) {
            IsirStepIn<D, NKC> cur, nxt;
            IsirCands<D, NKC> cands;
            isir_prepare<D, FAMILY, NKC>(K, R, stream, R.first_step, cur, cands);
            isir_park<D, NKC>(cands, take);
            for (uint32_t i = R.first_step; i <= R.last_step; ++i) {
                // (the prepare past the last step is wasted work; its rows are never read)
                isir_prepare<D, FAMILY, NKC>(K, R, stream, i + 1u, nxt, cands);
                isir_advance<D, FAMILY, NKC>(K, R, i, cur, take, s, stats, writer);
                isir_park<D, NKC>(cands, take);
                cur = nxt;
            }
        }
#pragma unroll
        for (int k = 0; k < D; ++k) {
            theta[k] = s.theta[k];
            y[k] = s.y[k];
        }
        lw_old = s.lw_old; local = s.local;
    } else
    for (uint32_t i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
        // ---------------- draws ----------------
        bool is_global;
        float u_a, eps_lp[D], eps_ls[D];
        double u64;
        const float* tp = nullptr;
        if constexpr (REPLAY) {
            tp = R.tape32 + (static_cast<int64_t>(i - R.first_step) * tape_slots) * R.n_chains + cidx;
            is_global = __ldg(tp) < R.gf;  // GLMCMC.py:59
#pragma unroll
            for (int k = 0; k < D; ++k) {  // a local step's draws sit in the first candidate's slots
                eps_lp[k] = __ldg(tp + static_cast<int64_t>(1 + k) * R.n_chains);
                eps_ls[k] = __ldg(tp + static_cast<int64_t>(1 + NK * D + k) * R.n_chains);
            }
            u_a = __ldg(tp + static_cast<int64_t>(1 + 2 * NK * D) * R.n_chains);
            u64 = R.tape64[static_cast<int64_t>(i - R.first_step) * R.n_chains + cidx];
        } else {
            const uint4 w0 = stream.block(R.rk, i, kSlotStep);
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
                eps_lp[k] = z[k];
                eps_ls[k] = z[D + k];
            }
            is_global = (step_block_ub(w0) < R.gf_thr_hi) || R.gf_all_global;
            const uint32_t ua24 = step_block_ua(w0);
            u_a = __uint2float_rn(ua24) * 0x1p-24f;
            // 53-bit resampling uniform: the step block's U_a field (unused on a global move) on top
            // of the spare U_a / U_b fields of candidate 0's first block
            const uint4 c0 = stream.block(R.rk, i, kSlotNormal + 8u);
            const uint64_t m53 = (static_cast<uint64_t>(ua24) << 29) | (static_cast<uint64_t>(step_block_ua(c0)) << 5) |
                                 static_cast<uint64_t>(step_block_ub(c0) >> 27);
            u64 = static_cast<double>(m53) * 0x1p-53;
        }

        // ---------------- iSIR arm: K candidates into the table (state-independent) ----------------
#pragma unroll
        for (int j = 0; j < NK; ++j) {
            float eps_p[D], eps_s[D];
            if constexpr (REPLAY) {
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    eps_p[k] = __ldg(tp + static_cast<int64_t>(1 + j * D + k) * R.n_chains);
                    eps_s[k] = __ldg(tp + static_cast<int64_t>(1 + NK * D + j * D + k) * R.n_chains);
                }
            } else {
                float z[kGroups * 4];
#pragma unroll
                for (int g = 0; g < kGroups; ++g) {
                    const uint4 w = stream.block(R.rk, i, kSlotNormal + 8u + j * kGroups + g);
                    box_muller(w.x, w.y, z[4 * g], z[4 * g + 1]);
                    box_muller(w.z, w.w, z[4 * g + 2], z[4 * g + 3]);
                }
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    eps_p[k] = z[k];
                    eps_s[k] = z[D + k];
                }
            }
            make_candidate<D, FAMILY, STRICT>(K, eps_p, eps_s, tab, j + 1);
            if constexpr (DUMP) {
                if (R.tape_dump != nullptr && active && is_global) {
                    float* t = R.tape_dump + (static_cast<int64_t>(i - R.first_step) * tape_slots) * R.n_chains + chain;
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        t[static_cast<int64_t>(1 + j * D + k) * R.n_chains] = eps_p[k];
                        t[static_cast<int64_t>(1 + NK * D + j * D + k) * R.n_chains] = eps_s[k];
                    }
                }
            }
        }

        // ---------------- iSIR arm: weight of the current state, resample ----------------
        float lw_cur = lw_old;
        if (local) {  // GLMCMC.py:60-64 (predicated: cheap, state-dependent)
            const float lq = gauss_log_prob<D, STRICT>(K.ip, theta);
            lw_cur = STRICT ? __fsub_rn(__fadd_rn(prior_old, kern_old), lq) : (prior_old + kern_old) - lq;
        }
        tab.at(0, 0) = weight_exp<STRICT>(lw_cur);
        int ind = -1;  // None
        float S;
        if constexpr (STRICT) {
            S = torch_sum_table<D>(tab, NK + 1);  // GLMCMC.py:82
            double run = 0.0;                     // GLMCMC.py:18-22: float64 running sum of float32 quotients
            for (int j = 0; j <= NK; ++j) {
                run += static_cast<double>(__fdiv_rn(tab.at(j, 0), S));
                if (ind < 0 && u64 < run) ind = j;
            }
        } else {
            S = 0.0f;
#pragma unroll
            for (int j = 0; j <= NK; ++j) S += tab.at(j, 0);
            // u < sum_{i<=j} w_i / S  <=>  u * S < sum_{i<=j} w_i, evaluated in float64
            const double thr = u64 * static_cast<double>(S);
            double run = 0.0;
#pragma unroll
            for (int j = 0; j <= NK; ++j) {
                run += static_cast<double>(tab.at(j, 0));
                if (ind < 0 && thr < run) ind = j;
            }
        }
        const bool switch_g = is_global && ind > 0;  // GLMCMC.py:84
        const int take = switch_g ? ind : 0;

        // ---------------- local arm: random-walk MH (GLMCMC.py:90-104) ----------------
        float th_l[D], y_l[D], z_l[D];
        (void)gauss_forward<D, STRICT>(K.lp, eps_lp, z_l);
#pragma unroll
        for (int k = 0; k < D; ++k) {
            th_l[k] = STRICT ? __fadd_rn(z_l[k], theta[k]) : z_l[k] + theta[k];
            const float mean = FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(th_l[k]) : th_l[k];
            if constexpr (STRICT) {
                y_l[k] = __fadd_rn(mean, __fadd_rn(K.model.noise_loc[k], __fmul_rn(K.model.noise_scale[k], eps_ls[k])));
            } else {
                y_l[k] = mean + fmaf(K.model.noise_scale[k], eps_ls[k], K.model.noise_loc[k]);
            }
        }
        const float prior_l = model_prior<D, STRICT>(K.model, th_l);
        const float kern_l = model_log_kernel<D, STRICT>(K.model, y_l);
        const float log_acc = STRICT ? __fsub_rn(__fsub_rn(__fadd_rn(prior_l, kern_l), prior_old), kern_old)
                                     : (prior_l + kern_l) - (prior_old + kern_old);
        const float log_w = STRICT ? logf(u_a) : log_approx(u_a);
        const bool accept_l = !is_global && (log_w < log_acc);

        // ---------------- state update ----------------
        float prev[D];
#pragma unroll
        for (int k = 0; k < D; ++k) prev[k] = theta[k];
        const float lw0 = lw_cur;  // log-weight the current state entered the resampling with
        if (switch_g) {
#pragma unroll
            for (int k = 0; k < D; ++k) {
                theta[k] = tab.at(take, 4 + k);
                y[k] = tab.at(take, 4 + D + k);
            }
            lw_cur = tab.at(take, 1);  // GLMCMC.py:86: cached log-weight of the taken candidate
            prior_old = tab.at(take, 2);  // same values the reference recomputes from (theta, y) later
            kern_old = tab.at(take, 3);
        }
        if (accept_l) {
#pragma unroll
            for (int k = 0; k < D; ++k) {
                theta[k] = th_l[k];
                y[k] = y_l[k];
            }
            prior_old = prior_l;
            kern_old = kern_l;
        }
        if (is_global) {
            lw_old = lw_cur;
            local = false;  // GLMCMC.py:65
        }
        local = local || accept_l;  // GLMCMC.py:100
        const bool moved = switch_g || accept_l;
        stats.update(is_global, moved, theta, prev);
        writer.put(R, i, theta);
        writer.maybe_flush(R, i);

        if constexpr (REPLAY) {
            if (R.debug != nullptr && active) {
                float* g = R.debug + static_cast<int64_t>(i - R.first_step) * GLABC_DEBUG_SLOTS * R.n_chains + chain;
                const int64_t n = R.n_chains;
                g[0] = static_cast<float>(static_cast<int>(is_global) | (static_cast<int>(moved) << 1) |
                                          ((is_global ? ind + 1 : 0) << 8));
                if (is_global) {
                    g[1 * n] = lw0;
                    g[2 * n] = S;
                    g[3 * n] = STRICT ? __fdiv_rn(tab.at(0, 0), S) : tab.at(0, 0) / S;
                    for (int j = 0; j < NK; ++j) g[(4 + j) * n] = tab.at(j + 1, 1);
                } else {
                    g[1 * n] = prior_l;
                    g[2 * n] = kern_l;
                    g[3 * n] = log_acc;
                    for (int j = 0; j < NK; ++j) g[(4 + j) * n] = 0.0f;
                }
            }
        }
        if constexpr (DUMP) {
            if (R.tape_dump != nullptr && active) {  // the uniforms + local normals this step consumed (replay layout;
                                                     // the candidates' normals are dumped inside the candidate loop)
                float* t = R.tape_dump + (static_cast<int64_t>(i - R.first_step) * tape_slots) * R.n_chains + chain;
                const int64_t n = R.n_chains;
                t[0] = is_global ? 0.0f : 1.0f;  // any value on the right side of gf reproduces the branch
                if (!is_global) {
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        t[(1 + k) * n] = eps_lp[k];
                        t[(1 + NK * D + k) * n] = eps_ls[k];
                    }
                }
                t[(1 + 2 * NK * D) * n] = u_a;
                if (R.tape64_dump != nullptr) R.tape64_dump[static_cast<int64_t>(i - R.first_step) * n + chain] = u64;
            }
        }
    }
    writer.finish(R);

    if (active) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            R.theta[static_cast<int64_t>(chain) * D + k] = theta[k];
            R.y[static_cast<int64_t>(chain) * D + k] = y[k];
        }
        R.aux[static_cast<int64_t>(chain) * GLABC_AUX_SLOTS + GLABC_AUX_LOGW] = lw_old;
        R.aux[static_cast<int64_t>(chain) * GLABC_AUX_SLOTS + GLABC_AUX_LOCAL] = local ? 1.0f : 0.0f;
        if (R.stats != nullptr)
            stats.store(R.stats + static_cast<int64_t>(chain) * GLABC_NSTATS(D), R.last_step + 1u - R.first_step);
    }
}

template <int D, int FAMILY, bool STRICT, bool REPLAY, int LAYOUT, bool DUMP, int NKT = 0>
static cudaError_t launch_isir_one(const IsirConsts& K, const RunParams& R, int block, cudaStream_t st)
{
    using Writer = typename WriterFor<D, LAYOUT>::type;
    const int grid = (R.n_chains + block - 1) / block;
    constexpr bool PIPE = !STRICT && !REPLAY && !DUMP && NKT > 0;   // pipelined loop: the smaller take-table
    const size_t table = PIPE ? static_cast<size_t>(R.n_candidates) * TakeTable<D>::kFields
                              : static_cast<size_t>(R.n_candidates + 1) * CandTable<D>::kFields;
    const size_t smem = sizeof(float) * (static_cast<size_t>(Writer::smem_floats_per_warp) * (block / 32) + table * block);
    auto kern = k_isir<D, FAMILY, STRICT, REPLAY, LAYOUT, DUMP, NKT>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
    }
    kern<<<grid, block, smem, st>>>(K, R);
    return cudaGetLastError();
}

template <int D, int FAMILY, bool STRICT>
static cudaError_t launch_isir_mode(const IsirConsts& K, const RunParams& R, bool replay, int layout, int block, cudaStream_t st)
{
    if (replay) {
        switch (layout) {
        case GLABC_TRACE_NONE: return launch_isir_one<D, FAMILY, STRICT, true, GLABC_TRACE_NONE, false>(K, R, block, st);
        case GLABC_TRACE_TIME_MAJOR: return launch_isir_one<D, FAMILY, STRICT, true, GLABC_TRACE_TIME_MAJOR, false>(K, R, block, st);
        case GLABC_TRACE_CHAIN_MAJOR: return launch_isir_one<D, FAMILY, STRICT, true, GLABC_TRACE_CHAIN_MAJOR, false>(K, R, block, st);
        }
        return cudaErrorInvalidValue;
    }
    if (R.tape_dump != nullptr) {
        if (layout != GLABC_TRACE_TIME_MAJOR) return cudaErrorInvalidValue;
        return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_TIME_MAJOR, true>(K, R, block, st);
    }
    if constexpr (!STRICT && D == 2) {  // the README / BASELINE configuration: batch_size = 5 (Mixture.py:73, README.md:125)
        if (R.n_candidates == 5) {
            switch (layout) {
            case GLABC_TRACE_NONE: return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_NONE, false, 5>(K, R, block, st);
            case GLABC_TRACE_TIME_MAJOR: return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_TIME_MAJOR, false, 5>(K, R, block, st);
            case GLABC_TRACE_CHAIN_MAJOR: return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_CHAIN_MAJOR, false, 5>(K, R, block, st);
            case GLABC_TRACE_EVENTS: return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_EVENTS, false, 5>(K, R, block, st);
            }
        }
    }
    switch (layout) {
    case GLABC_TRACE_NONE: return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_NONE, false>(K, R, block, st);
    case GLABC_TRACE_TIME_MAJOR: return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_TIME_MAJOR, false>(K, R, block, st);
    case GLABC_TRACE_CHAIN_MAJOR: return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_CHAIN_MAJOR, false>(K, R, block, st);
    case GLABC_TRACE_EVENTS: return launch_isir_one<D, FAMILY, STRICT, false, GLABC_TRACE_EVENTS, false>(K, R, block, st);
    }
    return cudaErrorInvalidValue;
}

template <int D>
cudaError_t launch_isir_dim(const ModelConsts& model, const GaussConsts& lp, const GaussConsts& ip, const RunParams& R,
                            bool strict, bool replay, int layout, int block, cudaStream_t st)
{
    IsirConsts K{model, lp, ip};
    return with_family(model.family, [&](auto f) {
        return strict ? launch_isir_mode<D, f, true>(K, R, replay, layout, block, st)
                      : launch_isir_mode<D, f, false>(K, R, replay, layout, block, st);
    });
}

}  // namespace glabc
