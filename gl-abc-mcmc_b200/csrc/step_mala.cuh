// K3 — the GLMALA chain step: with probability gf the iSIR global move of K2 (GLMALA.py:151-180),
// otherwise a MALA local move (GLMALA.py:182-200) whose drift is numberical_gradient_logABC
// (GLMALA.py:46-95): a central finite difference of a Gaussian synthetic log-likelihood of the
// discrepancy, estimated from 2*d*num_grad simulator draws with common random numbers, plus a
// float32 finite-difference prior gradient.  SURVEY.md A.3, quirks B-5..B-8.
//
// One WARP = one chain.  A local step is ~100x heavier than a global one (d*num_grad Philox/Box-Muller
// draws, each simulated at theta+h and theta-h), so the draws of a gradient are spread over the 32
// lanes (lane l owns Philox blocks l, l+32, ...) and the float64 mean / variance sums are folded with
// xor-shuffles; in a global step lane j < K evaluates candidate j and the K+1 weights are gathered
// with shuffles.  Everything that depends on the chain state is warp-uniform, so the global / local
// coin is a real (non-divergent) branch.  Carried state is float64 where the reference's is: the
// reference's MALA proposal adds a float64 gradient, so theta / y (and, if the first global move
// came later, the iSIR weights) become float64 tensors after the first accepted local move — the
// `wide` / `lw_wide` flags reproduce that dtype promotion because it changes decisions (float64 exp
// does not underflow at -104, SURVEY.md B-1).
#pragma once
#include "launch.cuh"
#include "sampler_common.cuh"
#include "step_generic.cuh"

namespace glabc {

struct MalaConsts {
    ModelConsts model;
    GaussConsts ip;    // Importance_Proposal
    GaussConsts unit;  // DiagGaussian(d, [0], [0]) of Local_proposal_forward / log_proposal (GLMALA.py:40,113)
    double eps2;       // ABCset.epsilon ** 2 (Python float, GLMALA.py:90)
    double tau;        // the Python float tau
    float tau_f;       // z * tau is a float32 product
    int32_t num_grad;
    int32_t ip_generic;   // the Importance_Proposal is a Uniform / Gamma / GaussianMixture: `ipg` (k_mala_fast only), else `ip`
    DistConsts ipg;
};

constexpr uint32_t kSlotGrad = 0x10000u;   // gradient normals of theta' (native mode)
constexpr uint32_t kSlotGrad0 = 0x20000u;  // gradient normals of the first gradient (grad_old is None)
constexpr double kLog2Pi = 1.8378770664093453;

__device__ __forceinline__ double shfl_xor_f64(double v, int off)
{
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_xor_sync(0xffffffffu, lo, off);
    hi = __shfl_xor_sync(0xffffffffu, hi, off);
    return __hiloint2double(hi, lo);
}

__device__ __forceinline__ double shfl_f64(double v, int src)
{
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_sync(0xffffffffu, lo, src);
    hi = __shfl_sync(0xffffffffu, hi, src);
    return __hiloint2double(hi, lo);
}

__device__ __forceinline__ double warp_sum_f64(double v)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += shfl_xor_f64(v, off);
    return v;
}

// torch.sum over n < 16 (four interleaved partials) / n >= 16 (16-lane vector path), float64 flavour
template <int N>
__device__ __forceinline__ double torch_sum64(const double (&v)[N])
{
    double p[4] = {0.0, 0.0, 0.0, 0.0};
    constexpr int rows = N / 4;
#pragma unroll
    for (int r = 0; r < rows; ++r)
#pragma unroll
        for (int k = 0; k < 4; ++k) p[k] += v[r * 4 + k];
#pragma unroll
    for (int i = rows * 4; i < N; ++i) p[0] += v[i];
#pragma unroll
    for (int k = 1; k < 4; ++k) p[0] += p[k];
    return p[0];
}

// DiagGaussian.log_prob on a float64 tensor with float32 parameters (torch type promotion)
template <int D>
__device__ __forceinline__ double gauss_log_prob64(const GaussConsts& g, const double (&z)[D])
{
    double t[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        const double r = (z[i] - static_cast<double>(g.loc[i])) / static_cast<double>(g.scale[i]);
        t[i] = static_cast<double>(g.log_scale[i]) + 0.5 * (r * r);
    }
    return -0.5 * D * kLog2Pi - torch_sum64<D>(t);
}

template <int D>
__device__ __forceinline__ double model_log_kernel64(const ModelConsts& m, const double (&y)[D])
{
    double t[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        const double dy = y[i] - static_cast<double>(m.y_obs[i]);
        t[i] = dy * dy;
    }
    const double dis = sqrt(torch_sum64<D>(t));
    const double r = (dis - 0.0) / static_cast<double>(m.eps_scale);
    return -0.5 * kLog2Pi - (static_cast<double>(m.eps_log_scale) + 0.5 * (r * r));
}

// discrepancy of one simulator draw at theta (float32; Mixture.py:13-26,33-36)
template <int D, int FAMILY, bool STRICT>
__device__ __forceinline__ float sim_discrepancy(const ModelConsts& m, const float (&theta)[D], const float (&eps)[D])
{
    float t[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        const float mean = FAMILY == GLABC_MODEL_ABS_NORMAL ? fabsf(theta[i]) : theta[i];
        if constexpr (STRICT) {
            const float yv = __fadd_rn(mean, __fadd_rn(m.noise_loc[i], __fmul_rn(m.noise_scale[i], eps[i])));
            const float dy = __fsub_rn(yv, m.y_obs[i]);
            t[i] = __fmul_rn(dy, dy);
        } else {
            const float dy = fmaf(m.noise_scale[i], eps[i], mean + m.noise_loc[i]) - m.y_obs[i];
            t[i] = dy * dy;
        }
    }
    if constexpr (STRICT) {
        return __fsqrt_rn(torch_sum_strict<D>(t));
    } else {
        float s = t[0];
#pragma unroll
        for (int i = 1; i < D; ++i) s += t[i];
        float r;
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(s));
        return r;
    }
}

// Where the normals of a gradient come from: a Philox slot base (native) or a tape column (replay),
// and where to dump them (native tape dump for the oracle cross-check).
struct GradSource {
    const float* tape;   // replay: &tape[first gradient slot][chain], stride n_chains between normals
    float* dump;         // native + dump: same layout, or nullptr
    uint32_t slot0;      // native: Philox slot base
    uint32_t step;
    int64_t stride;
};

// numberical_gradient_logABC(theta, num) -> grad[D]  (GLMALA.py:46-95)
// The k loop is deliberately NOT unrolled and the function is called from one site only: the kernel's
// instruction footprint is what limits it (warps of a block sit in different phases of the step).
template <int D, int FAMILY, bool STRICT, bool REPLAY>
__device__ __forceinline__ void mala_gradient(const MalaConsts& K, const RoundKeys& rk, const Stream& stream,
                                              const GradSource& src, const double (&theta_in)[D], int lane,
                                              double (&grad)[D], double* gstat)
{
    constexpr int kDpb = D == 3 ? 1 : 4 / D;  // draws per Philox block
    const int num = K.num_grad;
    const int nblk = (num + kDpb - 1) / kDpb;
    float th[D];
    const float zero[D] = {};
#pragma unroll
    for (int i = 0; i < D; ++i) th[i] = __double2float_rn(theta_in[i]);  // theta.float(), :60

#pragma unroll 1
    for (int k = 0; k < D; ++k) {
        float tp[D], tm[D], ta[D], tb[D];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            tp[i] = i == k ? __fadd_rn(th[i], 0.1f) : th[i];  // d * torch.eye in float32, :63-67
            tm[i] = i == k ? __fsub_rn(th[i], 0.1f) : th[i];
            ta[i] = i == k ? __fadd_rn(th[i], 0.00001f) : th[i];  // :84-85
            tb[i] = i == k ? __fsub_rn(th[i], 0.00001f) : th[i];
        }
        // sums are taken around the noise-free discrepancy (numerically robust one-pass variance)
        const float cpf = sim_discrepancy<D, FAMILY, STRICT>(K.model, tp, zero);
        const float cmf = sim_discrepancy<D, FAMILY, STRICT>(K.model, tm, zero);
        double s1p = 0.0, s2p = 0.0, s1m = 0.0, s2m = 0.0;
        float f1p = 0.0f, f2p = 0.0f, f1m = 0.0f, f2m = 0.0f;  // FAST: float32 sums (deviations from c are O(0.3))
#pragma unroll 1
        for (int g = lane; g < nblk; g += 32) {
            float z[4];
            if constexpr (!REPLAY) {
                const uint4 w = stream.block(rk, src.step, src.slot0 + static_cast<uint32_t>(k * nblk + g));
                box_muller(w.x, w.y, z[0], z[1]);
                box_muller(w.z, w.w, z[2], z[3]);
            }
#pragma unroll
            for (int t = 0; t < kDpb; ++t) {
                const int j = g * kDpb + t;
                if (j < num) {
                    float eps[D];
#pragma unroll
                    for (int q = 0; q < D; ++q) {
                        const int64_t idx = (static_cast<int64_t>(k) * num + j) * D + q;
                        if constexpr (REPLAY) {
                            eps[q] = __ldg(src.tape + idx * src.stride);
                        } else {
                            eps[q] = z[t * D + q];
                            if (src.dump != nullptr) src.dump[idx * src.stride] = eps[q];
                        }
                    }
                    const float dp = sim_discrepancy<D, FAMILY, STRICT>(K.model, tp, eps);  // :78-79
                    const float dm = sim_discrepancy<D, FAMILY, STRICT>(K.model, tm, eps);  // :80-83 (same draws)
                    if constexpr (STRICT) {
                        const double xp = static_cast<double>(dp) - static_cast<double>(cpf);
                        const double xm = static_cast<double>(dm) - static_cast<double>(cmf);
                        s1p += xp;
                        s2p = fma(xp, xp, s2p);
                        s1m += xm;
                        s2m = fma(xm, xm, s2m);
                    } else {
                        const float xp = dp - cpf, xm = dm - cmf;
                        f1p += xp;
                        f2p = fmaf(xp, xp, f2p);
                        f1m += xm;
                        f2m = fmaf(xm, xm, f2m);
                    }
                }
            }
        }
        // finite-difference prior gradient, h = 1e-5, in float32 (:84-85; ulp-noise dominated, B-8) — always
        // in the reference's exact operation order: it is the one piece whose rounding is visible
        const float gprior = __fdiv_rn(__fsub_rn(model_prior<D, true>(K.model, ta), model_prior<D, true>(K.model, tb)),
                                       static_cast<float>(2 * 0.00001));
        double gk;
        if constexpr (STRICT) {
            s1p = warp_sum_f64(s1p);
            s2p = warp_sum_f64(s2p);
            s1m = warp_sum_f64(s1m);
            s2m = warp_sum_f64(s2m);
            const double n = static_cast<double>(num);
            const double mup = static_cast<double>(cpf) + s1p / n, mum = static_cast<double>(cmf) + s1m / n;  // :86-87
            const double sp = (s2p - s1p * s1p / n) / (n - 1.0), sm = (s2m - s1m * s1m / n) / (n - 1.0);     // :88-89
            if (gstat != nullptr && k < 4) {   // replay debug record (glabc.h: debug64 slots 20..35)
                gstat[k] = mup;
                gstat[4 + k] = mum;
                gstat[8 + k] = sp;
                gstat[12 + k] = sm;
            }
            const double vp = sp + K.eps2, vm = sm + K.eps2;
            const double lpp = -0.5 * log(vp) - 0.5 * (mup * mup) / vp;  // :90-93
            const double lpm = -0.5 * log(vm) - 0.5 * (mum * mum) / vm;
            gk = (lpp - lpm) / (2 * 1e-1) + static_cast<double>(gprior);  // :94-95
        } else {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                f1p += __shfl_xor_sync(0xffffffffu, f1p, off);
                f2p += __shfl_xor_sync(0xffffffffu, f2p, off);
                f1m += __shfl_xor_sync(0xffffffffu, f1m, off);
                f2m += __shfl_xor_sync(0xffffffffu, f2m, off);
            }
            // the drift only has to be the same function of (theta, draws) on both sides of the MH ratio;
            // float32 here perturbs it by ~1e-5 relative
            const float rn = 1.0f / static_cast<float>(num), rn1 = 1.0f / static_cast<float>(num - 1);
            const float e2 = static_cast<float>(K.eps2);
            const float mup = fmaf(f1p, rn, cpf), mum = fmaf(f1m, rn, cmf);
            const float vp = fmaf(fmaf(-f1p * rn, f1p, f2p), rn1, e2), vm = fmaf(fmaf(-f1m * rn, f1m, f2m), rn1, e2);
            // lpp - lpm = -0.5 * (log(vp / vm) + mup^2 / vp - mum^2 / vm)
            const float ivp = __fdividef(1.0f, vp), ivm = __fdividef(1.0f, vm);
            const float dl = 0.69314718055994531f * lg2_approx(vp * ivm) + (mup * mup * ivp - mum * mum * ivm);
            gk = static_cast<double>(fmaf(dl, -2.5f, gprior));  // -0.5 / (2 * 0.1)
        }
#pragma unroll
        for (int i = 0; i < D; ++i) grad[i] = i == k ? gk : grad[i];
    }
}

// The K+1 iSIR weights live one per lane: lane 0 = the current state, lane j = candidate j (1 <= j <= K).
// torch.sum over them in ATen's order (SURVEY.md B-3): four interleaved partials for n < 16, the 16-lane
// vector path (tail first, then lanes 0..15) for n >= 16.
__device__ __forceinline__ float torch_sum_lanes(float w, int n)
{
    if (n >= 16) {
        float acc = 0.0f;
        for (int i = 16; i < n; ++i) acc = __fadd_rn(acc, __shfl_sync(0xffffffffu, w, i));
        for (int l = 0; l < 16; ++l) acc = __fadd_rn(acc, __shfl_sync(0xffffffffu, w, l));
        return acc;
    }
    float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
    const int body = n & ~3;
    for (int i = 0; i < n; ++i) {
        const float v = __shfl_sync(0xffffffffu, w, i);
        const int slot = i < body ? (i & 3) : 0;
        // x + 0 == x exactly for the non-negative weights, so the unselected partials are untouched
        p0 = __fadd_rn(p0, slot == 0 ? v : 0.0f);
        p1 = __fadd_rn(p1, slot == 1 ? v : 0.0f);
        p2 = __fadd_rn(p2, slot == 2 ? v : 0.0f);
        p3 = __fadd_rn(p3, slot == 3 ? v : 0.0f);
    }
    return __fadd_rn(__fadd_rn(__fadd_rn(p0, p1), p2), p3);
}

__device__ __forceinline__ double torch_sum_lanes64(double w, int n)
{
    double p0 = 0.0, p1 = 0.0, p2 = 0.0, p3 = 0.0;
    const int body = n & ~3;
    for (int i = 0; i < n; ++i) {
        const double v = shfl_f64(w, i);
        const int slot = i < body ? (i & 3) : 0;
        p0 += slot == 0 ? v : 0.0;
        p1 += slot == 1 ? v : 0.0;
        p2 += slot == 2 ? v : 0.0;
        p3 += slot == 3 ? v : 0.0;
    }
    return ((p0 + p1) + p2) + p3;
}

// inclusive prefix sum over lanes (float64), Hillis-Steele
__device__ __forceinline__ double warp_scan_f64(double v, int lane)
{
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        int lo = __double2loint(v), hi = __double2hiint(v);
        lo = __shfl_up_sync(0xffffffffu, lo, off);
        hi = __shfl_up_sync(0xffffffffu, hi, off);
        const double u = __hiloint2double(hi, lo);
        if (lane >= off) v += u;
    }
    return v;
}

template <int D, int FAMILY, bool STRICT, bool REPLAY, bool DUMP>
__global__ void __launch_bounds__(128, 6) k_mala(const __grid_constant__ MalaConsts K, const __grid_constant__ RunParams R)
{
    const int lane = threadIdx.x & 31;
    const int32_t chain = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (chain >= R.n_chains) return;  // warp-uniform
    const int NK = R.n_candidates;
    const int64_t C = R.n_chains;
    const int num = K.num_grad;
    const int tape_slots = 2 + NK * 2 * D + D * num * D;
    const int gslot0 = 2 + NK * 2 * D;
    constexpr int kGroups = (2 * D + 3) / 4;

    // ---- carried state (warp-uniform) ----
    float* aux = R.aux + static_cast<int64_t>(chain) * GLABC_AUX_SLOTS;
    double* s64 = R.state64 + static_cast<int64_t>(chain) * GLABC_STATE64_SLOTS;
    bool local = aux[GLABC_AUX_LOCAL] != 0.0f, wide = aux[GLABC_AUX_WIDE] != 0.0f;
    bool lw_wide = aux[GLABC_AUX_LW_WIDE] != 0.0f, have_grad = aux[GLABC_AUX_HAVE_GRAD] != 0.0f;
    double theta[D], y[D], grad[D], lw_old = s64[GLABC_S64_LOGW];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        theta[k] = wide ? s64[GLABC_S64_THETA + k] : static_cast<double>(R.theta[static_cast<int64_t>(chain) * D + k]);
        y[k] = wide ? s64[GLABC_S64_Y + k] : static_cast<double>(R.y[static_cast<int64_t>(chain) * D + k]);
        grad[k] = s64[GLABC_S64_GRAD + k];
    }

    // ---- trace: lane (row & 31) keeps row `row`; a 32-row window is flushed as one coalesced run ----
    float keep[D];
#pragma unroll
    for (int k = 0; k < D; ++k) keep[k] = 0.0f;
    const uint32_t first_row = R.write_row0 ? R.first_step - 1u : R.first_step;
    auto flush = [&](uint32_t last_row) {
        if (R.trace == nullptr) return;
        const uint32_t wb = last_row & ~31u;
        const uint32_t row = wb + lane;
        if (row >= first_row && row <= last_row) {
            const int64_t rr = static_cast<int64_t>(row) - R.trace_row_base;
            float* dst = R.trace_layout == GLABC_TRACE_CHAIN_MAJOR
                             ? R.trace + ((R.trace_chain_off + chain) * R.trace_rows + rr) * D
                             : R.trace + (rr * R.trace_chains + R.trace_chain_off + chain) * D;
#pragma unroll
            for (int k = 0; k < D; ++k) dst[k] = keep[k];
        }
    };
    if (R.write_row0 && lane == static_cast<int>((R.first_step - 1u) & 31u)) {
#pragma unroll
        for (int k = 0; k < D; ++k) keep[k] = __double2float_rn(theta[k]);
    }
    if (R.write_row0 && ((R.first_step & 31u) == 0u)) flush(R.first_step - 1u);

    ChainStats<D> stats;
    const Stream stream = chain_stream(R, chain);

    // FAST native mode: a run of consecutive GLOBAL moves is resolved in one batch.  The branch coins and the K candidates of
    // a step are state-independent (Philox), so lane (s, j) = s * (K + 1) + j builds candidate j - 1 of step i + s for up to five
    // steps at once (30 of 32 lanes busy instead of 6); only the short dependent part — the weight of the current state, the
    // max-shifted float32 weights, the scan against the 53-bit uniform, the switch — then runs step by step.
    const int G1 = NK + 1;
    const int slots = 32 / G1 < 5 ? 32 / G1 : 5;
    constexpr bool kBatch = !STRICT && !REPLAY && !DUMP;

    for (uint32_t i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
        if constexpr (kBatch) {
            if (slots >= 2) {
                const int s_mine = lane / G1, j_mine = lane - s_mine * G1;
                const uint32_t step_mine = i + static_cast<uint32_t>(s_mine);
                const bool in_use = s_mine < slots && step_mine <= R.last_step && step_mine >= i;
                const uint4 w0s = stream.block(R.rk, in_use ? step_mine : i, kSlotStep);
                const bool glob_mine = in_use && ((step_block_ub(w0s) < R.gf_thr_hi) || R.gf_all_global);
                const unsigned bal = __ballot_sync(0xffffffffu, glob_mine && j_mine == 0);
                int L = 0;
                while (L < slots && ((bal >> (L * G1)) & 1u)) ++L;
                if (L >= 1) {
                    // ---- state-independent part, all slots at once: candidate cj of step `step_mine` (GLMALA.py:158-165) ----
                    const int cj = j_mine > 0 ? j_mine - 1 : 0;   // lane (s, 0) shadows candidate 0: it needs that block's spare bits
                    float zc[kGroups * 4];
                    uint4 wfirst = make_uint4(0, 0, 0, 0);
#pragma unroll
                    for (int g = 0; g < kGroups; ++g) {
                        const uint4 w = stream.block(R.rk, in_use ? step_mine : i, kSlotNormal + 8u + cj * kGroups + g);
                        if (g == 0) wfirst = w;
                        box_muller(w.x, w.y, zc[4 * g], zc[4 * g + 1]);
                        box_muller(w.z, w.w, zc[4 * g + 2], zc[4 * g + 3]);
                    }
                    float eps_p[D], eps_s[D], th_c[D], x_c[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        eps_p[k] = zc[k];
                        eps_s[k] = zc[D + k];
                    }
                    const float lq = gauss_forward<D, false>(K.ip, eps_p, th_c);
                    model_simulate<D, false>(K.model, th_c, eps_s, x_c);
                    const float lw_c = (model_prior<D, false>(K.model, th_c) + model_log_kernel<D, false>(K.model, x_c)) - lq;
                    const uint64_t m53 = (static_cast<uint64_t>(step_block_ua(w0s)) << 29) |
                                         (static_cast<uint64_t>(step_block_ua(wfirst)) << 5) |
                                         static_cast<uint64_t>(step_block_ub(wfirst) >> 27);
                    const double u64_mine = static_cast<double>(m53) * 0x1p-53;   // valid in lane (s, 0)
                    // ---- the dependent part, step by step ----
                    for (int sidx = 0; sidx < L; ++sidx) {
                        const uint32_t step = i + static_cast<uint32_t>(sidx);
                        const int base = sidx * G1;
                        float prev[D];
#pragma unroll
                        for (int k = 0; k < D; ++k) prev[k] = __double2float_rn(theta[k]);
                        if (local) {  // GLMALA.py:152-156
                            if (wide) {
                                lw_old = (gauss_log_prob64<D>(K.model.prior, theta) + model_log_kernel64<D>(K.model, y)) -
                                         gauss_log_prob64<D>(K.ip, theta);
                            } else {
                                float tf[D], yf[D];
#pragma unroll
                                for (int k = 0; k < D; ++k) {
                                    tf[k] = __double2float_rn(theta[k]);
                                    yf[k] = __double2float_rn(y[k]);
                                }
                                lw_old = static_cast<double>((model_prior<D, false>(K.model, tf) + model_log_kernel<D, false>(K.model, yf)) -
                                                             gauss_log_prob<D, false>(K.ip, tf));
                            }
                            lw_wide = wide;
                        }
                        local = false;
                        const bool in_grp = lane >= base && lane < base + G1;
                        const float lw_f = lane == base ? static_cast<float>(lw_old) : lw_c;
                        float m = (in_grp && lw_f == lw_f) ? lw_f : -INFINITY;
#pragma unroll
                        for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
                        float w;
                        asm("ex2.approx.f32 %0, %1;" : "=f"(w) : "f"((lw_f - m) * 1.4426950408889634f));
                        if (w != w || !in_grp || m == -INFINITY) w = 0.0f;
                        double S = 0.0;   // summed in candidate order: the result does not depend on which slot the step sits in
                        for (int j = 0; j <= NK; ++j) S += static_cast<double>(__shfl_sync(0xffffffffu, w, base + j));
                        const double thr = shfl_f64(u64_mine, base) * S;
                        double run = 0.0;
                        int ind = -1;
                        for (int j = 0; j <= NK; ++j) {
                            run += static_cast<double>(__shfl_sync(0xffffffffu, w, base + j));
                            if (ind < 0 && thr < run) ind = j;
                        }
                        const int src = base + (ind > 0 ? ind : 1);
                        float th_t[D], x_t[D];
#pragma unroll
                        for (int k = 0; k < D; ++k) {
                            th_t[k] = __shfl_sync(0xffffffffu, th_c[k], src);
                            x_t[k] = __shfl_sync(0xffffffffu, x_c[k], src);
                        }
                        const float lw_t = __shfl_sync(0xffffffffu, lw_c, src);
                        if (ind > 0) {  // GLMALA.py:175-179: the cached gradient is NOT refreshed (B-6)
#pragma unroll
                            for (int k = 0; k < D; ++k) {
                                theta[k] = static_cast<double>(th_t[k]);
                                y[k] = static_cast<double>(x_t[k]);
                            }
                            lw_old = static_cast<double>(lw_t);
                        }
                        bool changed = false;
                        float now[D];
#pragma unroll
                        for (int k = 0; k < D; ++k) {
                            now[k] = __double2float_rn(theta[k]);
                            changed |= now[k] != prev[k];
                        }
                        stats.update(true, changed, now, prev);
                        if (lane == static_cast<int>(step & 31u)) {
#pragma unroll
                            for (int k = 0; k < D; ++k) keep[k] = now[k];
                        }
                        if (((step + 1u) & 31u) == 0u || step == R.last_step) flush(step);
                    }
                    i += static_cast<uint32_t>(L - 1);
                    continue;
                }
            }
        }
        const int64_t srow = static_cast<int64_t>(i - R.first_step);
        const float* tp = nullptr;
        uint4 w0 = make_uint4(0, 0, 0, 0);
        bool is_global;
        if constexpr (REPLAY) {
            tp = R.tape32 + (srow * tape_slots) * C + chain;
            is_global = __ldg(tp) < R.gf;  // GLMALA.py:151
        } else {
            w0 = stream.block(R.rk, i, kSlotStep);
            is_global = (step_block_ub(w0) < R.gf_thr_hi) || R.gf_all_global;
        }
        float* dump = nullptr;
        if constexpr (DUMP) {
            if (R.tape_dump != nullptr) dump = R.tape_dump + (srow * tape_slots) * C + chain;
            if (dump != nullptr && lane == 0) dump[0] = is_global ? 0.0f : 1.0f;  // any value on the right side of gf
        }
        float prev[D];
#pragma unroll
        for (int k = 0; k < D; ++k) prev[k] = __double2float_rn(theta[k]);
        bool changed = false;
        int ind = -1;
        double dbg[GLABC_DEBUG64_SLOTS];
        if constexpr (REPLAY) {
#pragma unroll
            for (int k = 0; k < GLABC_DEBUG64_SLOTS; ++k) dbg[k] = 0.0;
        }

        if (is_global) {
            // ================= iSIR global move, GLMALA.py:151-180 =================
            // lane 0 carries the current state's weight, lane j (1..K) candidate j-1; other lanes shadow
            double u64;
            const int cj = min(max(lane - 1, 0), NK - 1);
            const bool is_cand = lane >= 1 && lane <= NK;
            float eps_p[D], eps_s[D];
            if constexpr (REPLAY) {
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    eps_p[k] = __ldg(tp + static_cast<int64_t>(1 + cj * D + k) * C);
                    eps_s[k] = __ldg(tp + static_cast<int64_t>(1 + NK * D + cj * D + k) * C);
                }
                u64 = R.tape64[srow * C + chain];
            } else {
                float z[kGroups * 4];
                uint4 wfirst = make_uint4(0, 0, 0, 0);
#pragma unroll
                for (int g = 0; g < kGroups; ++g) {
                    const uint4 w = stream.block(R.rk, i, kSlotNormal + 8u + cj * kGroups + g);
                    if (g == 0) wfirst = w;
                    box_muller(w.x, w.y, z[4 * g], z[4 * g + 1]);
                    box_muller(w.z, w.w, z[4 * g + 2], z[4 * g + 3]);
                }
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    eps_p[k] = z[k];
                    eps_s[k] = z[D + k];
                }
                // 53-bit resampling uniform from spare bits of the step block and of candidate 0's first block
                // (lane 0 shadows candidate 0, so it holds that block)
                const uint64_t m53 = (static_cast<uint64_t>(step_block_ua(w0)) << 29) |
                                     (static_cast<uint64_t>(step_block_ua(wfirst)) << 5) |
                                     static_cast<uint64_t>(step_block_ub(wfirst) >> 27);
                u64 = shfl_f64(static_cast<double>(m53) * 0x1p-53, 0);
                if constexpr (DUMP) {
                    if (dump != nullptr && is_cand) {
#pragma unroll
                        for (int k = 0; k < D; ++k) {
                            dump[static_cast<int64_t>(1 + cj * D + k) * C] = eps_p[k];
                            dump[static_cast<int64_t>(1 + NK * D + cj * D + k) * C] = eps_s[k];
                        }
                    }
                    if (R.tape64_dump != nullptr && lane == 0) R.tape64_dump[srow * C + chain] = u64;
                }
            }
            // candidate cj (float32, GLMALA.py:158-165)
            float th_c[D], x_c[D];
            const float lq = gauss_forward<D, STRICT>(K.ip, eps_p, th_c);
            model_simulate<D, STRICT>(K.model, th_c, eps_s, x_c);
            const float prior_c = model_prior<D, STRICT>(K.model, th_c);
            const float kern_c = model_log_kernel<D, STRICT>(K.model, x_c);
            const float lw_c = STRICT ? __fsub_rn(__fadd_rn(prior_c, kern_c), lq) : (prior_c + kern_c) - lq;

            if (local) {  // GLMALA.py:152-156 — the only place log_weight_old is computed from the state
                if (wide) {
                    lw_old = (gauss_log_prob64<D>(K.model.prior, theta) + model_log_kernel64<D>(K.model, y)) -
                             gauss_log_prob64<D>(K.ip, theta);
                } else {
                    float tf[D], yf[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        tf[k] = __double2float_rn(theta[k]);
                        yf[k] = __double2float_rn(y[k]);
                    }
                    const float a = model_prior<D, STRICT>(K.model, tf), b = model_log_kernel<D, STRICT>(K.model, yf);
                    const float q = gauss_log_prob<D, STRICT>(K.ip, tf);
                    lw_old = static_cast<double>(STRICT ? __fsub_rn(__fadd_rn(a, b), q) : (a + b) - q);
                }
                lw_wide = wide;
            }
            local = false;

            double S, w0n;
            if (!STRICT && lw_wide) {
                // FAST: the promoted (float64) weights only matter because float32 exp underflows near -104; exponentiating
                // max-shifted in float32 gives the same resampling law without the double-precision exp, divide and scan
                const float lw_f = lane == 0 ? static_cast<float>(lw_old) : lw_c;
                float m = (lane <= NK && lw_f == lw_f) ? lw_f : -INFINITY;
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
                float w;
                asm("ex2.approx.f32 %0, %1;" : "=f"(w) : "f"((lw_f - m) * 1.4426950408889634f));
                if (w != w || lane > NK || m == -INFINITY) w = 0.0f;
                float Sf = w;
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) Sf += __shfl_xor_sync(0xffffffffu, Sf, off);
                const double thr = u64 * static_cast<double>(Sf);
                double run = 0.0;
                for (int j = 0; j <= NK; ++j) {
                    run += static_cast<double>(__shfl_sync(0xffffffffu, w, j));
                    if (ind < 0 && thr < run) ind = j;
                }
                S = static_cast<double>(Sf) * exp(static_cast<double>(m));   // un-shifted, for the debug record only (dead otherwise)
                w0n = static_cast<double>(__fdiv_rn(__shfl_sync(0xffffffffu, w, 0), Sf));
            } else if (lw_wide) {  // float64 weights (no underflow near -104)
                double w = exp(lane == 0 ? lw_old : static_cast<double>(lw_c));
                if (w != w || lane > NK) w = 0.0;
                S = torch_sum_lanes64(w, NK + 1);
                const double q = w / S;
                double run = 0.0;
                for (int j = 0; j <= NK; ++j) {
                    run += shfl_f64(q, j);
                    if (ind < 0 && u64 < run) ind = j;
                }
                w0n = shfl_f64(q, 0);
            } else {
                const float lw_f = lane == 0 ? __double2float_rn(lw_old) : lw_c;
                float w;
                if constexpr (STRICT) {
                    w = expf(lw_f);
                } else {
                    asm("ex2.approx.f32 %0, %1;" : "=f"(w) : "f"(lw_f * 1.4426950408889634f));
                }
                if (w != w || lane > NK) w = 0.0f;
                float Sf;
                double run = 0.0;
                if constexpr (STRICT) {
                    Sf = torch_sum_lanes(w, NK + 1);
                    const float q = __fdiv_rn(w, Sf);
                    for (int j = 0; j <= NK; ++j) {
                        run += static_cast<double>(__shfl_sync(0xffffffffu, q, j));
                        if (ind < 0 && u64 < run) ind = j;
                    }
                } else {
                    Sf = w;
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) Sf += __shfl_xor_sync(0xffffffffu, Sf, off);
                    const double thr = u64 * static_cast<double>(Sf);  // u < cumsum(w)/S  <=>  u*S < cumsum(w)
                    for (int j = 0; j <= NK; ++j) {
                        run += static_cast<double>(__shfl_sync(0xffffffffu, w, j));
                        if (ind < 0 && thr < run) ind = j;
                    }
                }
                S = static_cast<double>(Sf);
                w0n = static_cast<double>(__fdiv_rn(__shfl_sync(0xffffffffu, w, 0), Sf));
            }
            if constexpr (REPLAY) {
                dbg[1] = lw_old;
                dbg[2] = S;
                dbg[3] = w0n;
#pragma unroll
                for (int j = 0; j < GLABC_MAX_K; ++j) {
                    const float v = __shfl_sync(0xffffffffu, lw_c, j + 1);
                    if (j < NK) dbg[4 + j] = static_cast<double>(v);
                }
            }
            const int src = ind > 0 ? ind : 1;
            float th_t[D], x_t[D];
#pragma unroll
            for (int k = 0; k < D; ++k) {
                th_t[k] = __shfl_sync(0xffffffffu, th_c[k], src);
                x_t[k] = __shfl_sync(0xffffffffu, x_c[k], src);
            }
            const float lw_t = __shfl_sync(0xffffffffu, lw_c, src);
            if (ind > 0) {  // GLMALA.py:175-179: the cached gradient is NOT refreshed (B-6)
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    theta[k] = static_cast<double>(th_t[k]);
                    y[k] = static_cast<double>(x_t[k]);
                }
                lw_old = static_cast<double>(lw_t);
            }
#pragma unroll
            for (int k = 0; k < D; ++k) changed |= (__double2float_rn(theta[k]) != prev[k]);
        } else {
            // ================= MALA local move, GLMALA.py:182-200 =================
            float z[D], eps_s[D], u_a;
            if constexpr (REPLAY) {
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    z[k] = __ldg(tp + static_cast<int64_t>(1 + k) * C);
                    eps_s[k] = __ldg(tp + static_cast<int64_t>(1 + NK * D + k) * C);
                }
                u_a = __ldg(tp + static_cast<int64_t>(1 + 2 * NK * D) * C);
            } else {
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
                if constexpr (DUMP) {
                    if (dump != nullptr && lane == 0) {
#pragma unroll
                        for (int k = 0; k < D; ++k) {
                            dump[static_cast<int64_t>(1 + k) * C] = z[k];
                            dump[static_cast<int64_t>(1 + NK * D + k) * C] = eps_s[k];
                        }
                        dump[static_cast<int64_t>(1 + 2 * NK * D) * C] = u_a;
                    }
                }
            }
            float zf[D];
            const float lq_fwd = gauss_forward<D, true>(K.unit, z, zf);  // Local_proposal_forward, :25-44
            double theta_p[D], grad_p[D], y_p[D];
            // pass 0 (only while grad_logABC_Theta_old is None, :183-184): gradient at theta;
            // pass 1: proposal theta' from the cached gradient (:186), gradient at theta' (:187) — one call site
#pragma unroll 1
            for (int pass = have_grad ? 1 : 0; pass < 2; ++pass) {
                double tgt[D];
                GradSource gs{};
                gs.stride = C;
                gs.step = i;
                if (pass == 0) {
                    gs.slot0 = kSlotGrad0;
                    if constexpr (REPLAY) gs.tape = R.tape_grad0 + chain;
                    if constexpr (DUMP) gs.dump = R.tape_grad0_dump != nullptr ? R.tape_grad0_dump + chain : nullptr;
#pragma unroll
                    for (int k = 0; k < D; ++k) tgt[k] = theta[k];
                } else {
                    gs.slot0 = kSlotGrad;
                    if constexpr (REPLAY) gs.tape = tp + static_cast<int64_t>(gslot0) * C;
                    if constexpr (DUMP) gs.dump = dump != nullptr ? dump + static_cast<int64_t>(gslot0) * C : nullptr;
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        const float zt = __fmul_rn(zf[k], K.tau_f);
                        const double a = wide ? static_cast<double>(zt) + theta[k]
                                              : static_cast<double>(__fadd_rn(zt, __double2float_rn(theta[k])));
                        theta_p[k] = a + grad[k] * (K.tau * K.tau) / 2.0;  // :43
                        tgt[k] = theta_p[k];
                    }
                }
                double gout[D];
#pragma unroll
                for (int k = 0; k < D; ++k) gout[k] = 0.0;
                double* gstat = nullptr;
                if constexpr (REPLAY) gstat = pass == 1 ? dbg + 20 : nullptr;
                mala_gradient<D, FAMILY, STRICT, REPLAY>(K, R.rk, stream, gs, tgt, lane, gout, gstat);
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    if (pass == 0) grad[k] = gout[k];
                    grad_p[k] = gout[k];
                }
            }
            have_grad = true;
#pragma unroll
            for (int k = 0; k < D; ++k) {  // :188-189: |theta'| (float64) + likelihood.sample() (float32)
                const float noise = __fadd_rn(K.model.noise_loc[k], __fmul_rn(K.model.noise_scale[k], eps_s[k]));
                const double mean = FAMILY == GLABC_MODEL_ABS_NORMAL ? fabs(theta_p[k]) : theta_p[k];
                y_p[k] = mean + static_cast<double>(noise);
            }
            double prior_p, kern_p, lq_rev, log_acc;
            if constexpr (STRICT) {
                prior_p = gauss_log_prob64<D>(K.model.prior, theta_p);
                kern_p = model_log_kernel64<D>(K.model, y_p);
                double rr[D];  // log_proposal(Theta_prop, grad_prop, Theta_old, tau), :97-116
#pragma unroll
                for (int k = 0; k < D; ++k) rr[k] = (theta[k] - theta_p[k] - grad_p[k] * (K.tau * K.tau) / 2.0) / K.tau;
                lq_rev = gauss_log_prob64<D>(K.unit, rr);
                double prior_o, kern_o;
                if (wide) {
                    prior_o = gauss_log_prob64<D>(K.model.prior, theta);
                    kern_o = model_log_kernel64<D>(K.model, y);
                } else {
                    float tf[D], yf[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        tf[k] = __double2float_rn(theta[k]);
                        yf[k] = __double2float_rn(y[k]);
                    }
                    prior_o = static_cast<double>(model_prior<D, STRICT>(K.model, tf));
                    kern_o = static_cast<double>(model_log_kernel<D, STRICT>(K.model, yf));
                }
                log_acc = prior_p + kern_p + lq_rev - prior_o - kern_o - static_cast<double>(lq_fwd);  // :190-193
            } else {
                // FAST: the five log-densities in float32 (the reference's are float64 only because theta was promoted); the
                // state itself stays float64 so the chain's arithmetic on theta is unchanged
                float tpf[D], ypf[D], tf[D], yf[D], rrf[D];
                const float inv_tau = 1.0f / K.tau_f, half_tau2 = 0.5f * K.tau_f * K.tau_f;
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    tpf[k] = static_cast<float>(theta_p[k]);
                    ypf[k] = static_cast<float>(y_p[k]);
                    tf[k] = static_cast<float>(theta[k]);
                    yf[k] = static_cast<float>(y[k]);
                    rrf[k] = (static_cast<float>(theta[k] - theta_p[k]) - static_cast<float>(grad_p[k]) * half_tau2) * inv_tau;
                }
                const float pp = model_prior<D, false>(K.model, tpf), kp = model_log_kernel<D, false>(K.model, ypf);
                const float lr = gauss_log_prob<D, false>(K.unit, rrf);
                const float po = model_prior<D, false>(K.model, tf), ko = model_log_kernel<D, false>(K.model, yf);
                prior_p = static_cast<double>(pp);
                kern_p = static_cast<double>(kp);
                lq_rev = static_cast<double>(lr);
                log_acc = static_cast<double>(((pp + kp) - (po + ko)) + (lr - lq_fwd));
            }
            const float log_w = STRICT ? logf(u_a) : log_approx(u_a);
            const bool accept = static_cast<double>(log_w) < log_acc;
            if constexpr (REPLAY) {
                dbg[1] = log_acc;
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    dbg[2 + k] = theta_p[k];
                    dbg[6 + k] = y_p[k];
                    dbg[10 + k] = grad_p[k];
                }
                dbg[14] = prior_p;
                dbg[15] = kern_p;
                dbg[16] = lq_rev;
                dbg[17] = static_cast<double>(lq_fwd);
            }
            if (accept) {  // :195-199
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

        float now[D];
#pragma unroll
        for (int k = 0; k < D; ++k) now[k] = __double2float_rn(theta[k]);  // Theta_Re[i,:] = Theta_old (float32 buffer)
        stats.update(is_global, changed, now, prev);
        if (lane == static_cast<int>(i & 31u)) {
#pragma unroll
            for (int k = 0; k < D; ++k) keep[k] = now[k];
        }
        if (((i + 1u) & 31u) == 0u || i == R.last_step) flush(i);

        if constexpr (REPLAY) {
            if (R.debug64 != nullptr && lane == 0) {
                dbg[0] = static_cast<double>(static_cast<int>(is_global) | (static_cast<int>(changed) << 1) |
                                             ((is_global ? ind + 1 : 0) << 8) | (static_cast<int>(is_global && lw_wide) << 16));
                double* g = R.debug64 + srow * GLABC_DEBUG64_SLOTS * C + chain;
#pragma unroll
                for (int k = 0; k < GLABC_DEBUG64_SLOTS; ++k) g[static_cast<int64_t>(k) * C] = dbg[k];
            }
        }
    }

    if (R.last_step < R.first_step && R.write_row0) flush(R.first_step - 1u);

    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            R.theta[static_cast<int64_t>(chain) * D + k] = __double2float_rn(theta[k]);
            R.y[static_cast<int64_t>(chain) * D + k] = __double2float_rn(y[k]);
            s64[GLABC_S64_THETA + k] = theta[k];
            s64[GLABC_S64_Y + k] = y[k];
            s64[GLABC_S64_GRAD + k] = grad[k];
        }
        s64[GLABC_S64_LOGW] = lw_old;
        aux[GLABC_AUX_LOCAL] = local ? 1.0f : 0.0f;
        aux[GLABC_AUX_WIDE] = wide ? 1.0f : 0.0f;
        aux[GLABC_AUX_LW_WIDE] = lw_wide ? 1.0f : 0.0f;
        aux[GLABC_AUX_HAVE_GRAD] = have_grad ? 1.0f : 0.0f;
        if (R.stats != nullptr)
            stats.store(R.stats + static_cast<int64_t>(chain) * GLABC_NSTATS(D), R.last_step + 1u - R.first_step);
    }
}

template <int D, int FAMILY, bool STRICT, bool REPLAY, bool DUMP>
static cudaError_t launch_mala_one(const MalaConsts& K, const RunParams& R, int block, cudaStream_t st)
{
    if (block > 128) block = 128;   // __launch_bounds__(128, 6): 80 registers, six CTAs (24 chains) per SM
    const int warps_per_block = block / 32;
    const int grid = (R.n_chains + warps_per_block - 1) / warps_per_block;
    k_mala<D, FAMILY, STRICT, REPLAY, DUMP><<<grid, block, 0, st>>>(K, R);
    return cudaGetLastError();
}

// the throughput path (step_mala_fast.cuh): FAST arithmetic, native Philox, no tape dump
template <int D, int FAMILY>
static cudaError_t launch_mala_fast(const MalaConsts& K, const DistConsts& prior, const RunParams& R, cudaStream_t st);

template <int D, int FAMILY>
static cudaError_t launch_mala_family(const MalaConsts& K, const DistConsts& prior, const RunParams& R, bool strict, bool replay,
                                      int block, cudaStream_t st)
{
    const bool dump = R.tape_dump != nullptr;
    // block_threads == 96 keeps the warp-per-chain kernel for FAST runs too (tests compare the two layouts)
    if (K.ip_generic || generic_prior(prior)) {   // host side has checked: FAST arithmetic, native RNG, no tape dump
        if (strict || replay || dump) return cudaErrorInvalidValue;
        return launch_mala_fast<D, FAMILY>(K, prior, R, st);
    }
    if (!strict && !replay && !dump && block != 96) return launch_mala_fast<D, FAMILY>(K, prior, R, st);
    if (replay)
        return strict ? launch_mala_one<D, FAMILY, true, true, false>(K, R, block, st)
                      : launch_mala_one<D, FAMILY, false, true, false>(K, R, block, st);
    if (dump)
        return strict ? launch_mala_one<D, FAMILY, true, false, true>(K, R, block, st)
                      : launch_mala_one<D, FAMILY, false, false, true>(K, R, block, st);
    return strict ? launch_mala_one<D, FAMILY, true, false, false>(K, R, block, st)
                  : launch_mala_one<D, FAMILY, false, false, false>(K, R, block, st);
}

template <int D>
cudaError_t launch_mala_dim(const MalaConsts& K, const DistConsts& prior, const RunParams& R, bool strict, bool replay, int block,
                            cudaStream_t st)
{
    return with_family(K.model.family, [&](auto f) { return launch_mala_family<D, f>(K, prior, R, strict, replay, block, st); });
}

}  // namespace glabc
