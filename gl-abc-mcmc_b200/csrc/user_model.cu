// User-supplied ABC models compiled at run time into the fused GlobalMCMC step kernel (SURVEY.md 8(f) n1).
//
// The reference's plugin surface is a duck-typed Python object (generate_samples / prior_log_prob / discrepancy,
// examples/Mixture.py:13-36, README.md:66-104); an arbitrary Python simulator cannot run inside a kernel.  Here the
// three model functions arrive as CUDA C++ device-function source, are concatenated between a prelude (Philox4x32-10,
// Box-Muller) and the step kernel below, and compiled with NVRTC for the device's architecture — the simulator is
// inlined into the same single kernel as the proposal, the Gaussian ABC kernel and the MH test (GlobalMCMC.py:37-68).
//
// libnvrtc / libcuda are dlopen'ed on first use: libglabc.so itself keeps no link-time dependency on them, so it
// still loads (and exports every symbol) on a machine without a driver.
#include <dlfcn.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>
#include <nvrtc.h>

#include "user_model.cuh"

namespace glabc {

namespace {

// ---- the kernel's source: prelude + (user source) + step kernel.  D, YD, NN and the two proposal kinds GLABC_LP_KIND,
// GLABC_GP_KIND arrive as -D macros; the prelude includes dist_device.cuh, whose text build.py embeds here. ----
const char kDistDevice[] =
#include "dist_device_src.inc"
    ;

const char* kPrelude = R"GLABC(
typedef unsigned int u32;
typedef unsigned long long u64;
// NVRTC compiles without the host's <cmath>: the usual constants a model may want
#ifndef INFINITY
#define INFINITY __int_as_float(0x7f800000)
#endif
#ifndef NAN
#define NAN __int_as_float(0x7fffffff)
#endif
#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif
#include "dist_device.cuh"
using glabc::UserRun;
using glabc::UserEval;
// A prior may return exactly this value to say "outside the support: draw the local proposal again" — the reference's
// `while prior_log_prob(theta') == 7 * np.log(1e-10)` (GLMCMC.py:92-93; the float32 tensor is compared with the float64
// scalar cast down to float32)
#define GLABC_PRIOR_SENTINEL (-161.18095397949219f)
__device__ __forceinline__ uint4 glabc_philox(u32 c0, u32 c1, u32 c2, u32 c3, u32 k0, u32 k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const u64 p0 = (u64)0xD2511F53u * c0;
        const u64 p1 = (u64)0xCD9E8D57u * c2;
        const u32 n0 = (u32)(p1 >> 32) ^ c1 ^ k0, n2 = (u32)(p0 >> 32) ^ c3 ^ k1;
        c1 = (u32)p1; c3 = (u32)p0; c0 = n0; c2 = n2;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ void glabc_box_muller(u32 w0, u32 w1, float& n0, float& n1)
{
    const float u1 = fmaf(__uint2float_rn(w0 >> 8), 0x1p-24f, 0x1p-25f);
    const float r = sqrtf(-2.0f * __logf(u1));
    const float a = __uint2float_rn(w1 >> 8) * (6.28318530717958647692f * 0x1p-24f);
    float s, c;
    __sincosf(a, &s, &c);
    n0 = r * c;
    n1 = r * s;
}
// dist_forward's word source: successive 32-bit words of the Philox blocks (chain, step, slot0), (.., slot0 + 1), ..
struct GlabcWords {
    u32 g0, g1, step, slot, k0, k1;
    uint4 cur;
    int used;
    float spare;
    bool has_spare;
    __device__ __forceinline__ GlabcWords(u32 c0, u32 c1, u32 i, u32 slot0, u32 key0, u32 key1)
        : g0(c0), g1(c1), step(i), slot(slot0), k0(key0), k1(key1), cur(make_uint4(0, 0, 0, 0)), used(4), spare(0.f), has_spare(false) {}
    __device__ __forceinline__ u32 next()
    {
        if (used == 4) {
            cur = glabc_philox(g0, g1, step, slot++, k0, k1);
            used = 0;
        }
        const u32 w = used == 0 ? cur.x : used == 1 ? cur.y : used == 2 ? cur.z : cur.w;
        ++used;
        return w;
    }
    __device__ __forceinline__ float uniform() { return __uint2float_rn(next() >> 8) * 0x1p-24f; }                 // [0, 1)
    __device__ __forceinline__ float uniform_open() { return fmaf(__uint2float_rn(next() >> 8), 0x1p-24f, 0x1p-25f); }  // (0, 1)
    __device__ __forceinline__ float normal()
    {
        if (has_spare) {
            has_spare = false;
            return spare;
        }
        const u32 w0 = next(), w1 = next();
        float n0;
        glabc_box_muller(w0, w1, n0, spare);
        has_spare = true;
        return n0;
    }
};
// Philox slots (the counter's last word) the user kernels draw from, per (chain, step):
//   step 0, 2 ..             glabc_k_eval_user's SIMULATE: ceil(NN / 4) blocks of the simulator's normals for row
//                            row_base + r.  The step kernels draw only at steps step_base + 1 .. (the loop index i >= 1),
//                            so step 0 is never used by a run, and y0 of chain c is the SIMULATE row chain_id_base + c.
//   1                        the step's coin and MH uniform
//   2 ..                     NB blocks of normals: a DiagGaussian proposal's D, then the simulator's NN
//   0x100 + j NB ..          the same for iSIR candidate j < GLABC_MAX_K
//   0x10000 .., 0x20000 ..   GLMALA's gradient draws
//   0x40000000 + r ..        redraw r < 64 of a DiagGaussian local proposal the prior answered with GLABC_PRIOR_SENTINEL
//   0x80000000               the iSIR resampling uniform
//   GLABC_SLOT_PROP ..       a Uniform / Gamma / GaussianMixture local or global draw; sentinel redraws continue its stream
//   GLABC_SLOT_CAND + j GLABC_CAND_BLOCKS ..   iSIR candidate j from a Uniform / Gamma / GaussianMixture importance proposal
// A non-Gaussian proposal only moves the proposal's draws: the simulator keeps its blocks.  One dist_forward takes at most
// 386 blocks at D = 8 (Gamma: 8 x (64 squeeze iterations x 3 words + 1) words, dist_device.cuh), so a candidate's range
// of 0x200 blocks holds it, and the 65 draws of a local move with every redraw (25090 blocks) fit under GLABC_SLOT_CAND.
#define GLABC_SLOT_PROP 0x60000000u
#define GLABC_SLOT_CAND 0x60010000u
#define GLABC_CAND_BLOCKS 0x200u
)GLABC";

const char* kKernel = R"GLABC(
__device__ __forceinline__ float glabc_target(const UserRun& R, const float* th, const float* y)
{
    const float dis = glabc_user_discrepancy(y, R.params);
    return glabc_user_prior_log_prob(th, R.params) + fmaf(R.kern_m, dis * dis, R.kern_c);
}
extern "C" __global__ void __launch_bounds__(128) glabc_k_global_user(const __grid_constant__ UserRun R)
{
    const int chain = blockIdx.x * blockDim.x + threadIdx.x;
    if (chain >= R.n_chains) return;
    const u64 gid = ((u64)R.chain_hi0 << 32 | R.chain_lo0) + (u64)chain;
    const u32 g0 = (u32)gid, g1 = (u32)(gid >> 32);
    float th[D], y[YD];
#pragma unroll
    for (int k = 0; k < D; ++k) th[k] = R.theta[(long long)chain * D + k];
#pragma unroll
    for (int k = 0; k < YD; ++k) y[k] = R.y[(long long)chain * YD + k];
    float tgt = glabc_target(R, th, y);
    float n_glob = 0.f, acc_l = 0.f, acc_g = 0.f, sum[D], sumsq[D], gram[D * (D + 1) / 2];
#pragma unroll
    for (int k = 0; k < D; ++k) sum[k] = sumsq[k] = 0.f;
#pragma unroll
    for (int k = 0; k < D * (D + 1) / 2; ++k) gram[k] = 0.f;
    // trace rows: row index = loop index i, row 0 = initial theta (GlobalMCMC.py:34-35)
    const long long cstride = R.trace_layout == 2 ? (long long)D : R.trace_chains * D;   // per ROW
    float* row = nullptr;
    if (R.trace_layout != 0) {
        const long long r0 = (long long)R.first_step - (R.write_row0 ? 1 : 0) - R.trace_row_base;
        row = R.trace_layout == 2 ? R.trace + ((R.trace_chain_off + chain) * R.trace_rows + r0) * D
                                  : R.trace + (r0 * R.trace_chains + R.trace_chain_off + chain) * D;
        if (R.write_row0) {
#pragma unroll
            for (int k = 0; k < D; ++k) row[k] = th[k];
            row += cstride;
        }
    }
    constexpr int NZ = D + NN;                 // normals per step
    constexpr int NB = (NZ + 3) / 4;           // extra Philox blocks carrying them
    for (u32 i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
        const uint4 w0 = glabc_philox(g0, g1, i, 1u, R.key0, R.key1);
        const bool is_global = R.gf_all_global || (w0.x < R.gf_thr);              // GlobalMCMC.py:38-39
        const float log_u = __logf(__uint2float_rn(w0.y >> 8) * 0x1p-24f);         // :47,61 (log 0 = -inf accepts, as torch's)
        float z[NB * 4 + 4];
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const uint4 w = glabc_philox(g0, g1, i, 2u + b, R.key0, R.key1);
            glabc_box_muller(w.x, w.y, z[4 * b], z[4 * b + 1]);
            glabc_box_muller(w.z, w.w, z[4 * b + 2], z[4 * b + 3]);
        }
        float thp[D], yp[YD], corr = 0.f;
        if (is_global) {                       // independence proposal q = Global_Proposal, :40-46
#if GLABC_GP_KIND == GLABC_DIST_DIAG_GAUSSIAN
            float qn = 0.f, qo = 0.f;
#pragma unroll
            for (int k = 0; k < D; ++k) {
                thp[k] = fmaf(R.gp_scale[k], z[k], R.gp_loc[k]);
                const float r = (th[k] - R.gp_loc[k]) * R.gp_inv_scale[k];
                qn = fmaf(z[k], z[k], qn);
                qo = fmaf(r, r, qo);
            }
            corr = 0.5f * (qn - qo);           // log q(theta) - log q(theta'): the constants cancel
#else
            GlabcWords ws(g0, g1, i, GLABC_SLOT_PROP, R.key0, R.key1);
            const float lq_p = glabc::dist_forward<D>(R.gq, ws, thp);
            corr = glabc::dist_log_prob<D>(R.gq, th) - lq_p;
#endif
        } else {                               // random walk theta + z, z ~ Local_Proposal, :56-60 (no q term)
#if GLABC_LP_KIND == GLABC_DIST_DIAG_GAUSSIAN
#pragma unroll
            for (int k = 0; k < D; ++k) thp[k] = th[k] + fmaf(R.lp_scale[k], z[k], R.lp_loc[k]);
#else
            GlabcWords ws(g0, g1, i, GLABC_SLOT_PROP, R.key0, R.key1);
            float zl[D];
            (void)glabc::dist_forward<D>(R.lq, ws, zl);
#pragma unroll
            for (int k = 0; k < D; ++k) thp[k] = th[k] + zl[k];
#endif
        }
        glabc_user_simulate(thp, z + D, R.params, yp);
        const float tgt_p = glabc_target(R, thp, yp);
        const bool acc = log_u < (tgt_p - tgt) + corr;
        float dl[D];
#pragma unroll
        for (int k = 0; k < D; ++k) {
            dl[k] = acc ? thp[k] - th[k] : 0.f;
            th[k] = acc ? thp[k] : th[k];
            sum[k] += th[k];
            sumsq[k] = fmaf(th[k], th[k], sumsq[k]);
        }
        if (acc) {
#pragma unroll
            for (int k = 0; k < YD; ++k) y[k] = yp[k];
            tgt = tgt_p;
        }
        int t = 0;
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = a; b < D; ++b, ++t) gram[t] = fmaf(dl[a], dl[b], gram[t]);
        n_glob += is_global ? 1.f : 0.f;
        acc_g += (acc && is_global) ? 1.f : 0.f;
        acc_l += (acc && !is_global) ? 1.f : 0.f;
        if (row != nullptr) {
#pragma unroll
            for (int k = 0; k < D; ++k) row[k] = th[k];
            row += cstride;
        }
    }
#pragma unroll
    for (int k = 0; k < D; ++k) R.theta[(long long)chain * D + k] = th[k];
#pragma unroll
    for (int k = 0; k < YD; ++k) R.y[(long long)chain * YD + k] = y[k];
    if (R.stats != nullptr) {
        float* st = R.stats + (long long)chain * (4 + 2 * D + D * (D + 1) / 2);
        st[0] += R.last_step >= R.first_step ? (float)(R.last_step + 1u - R.first_step) : 0.f;
        st[1] += n_glob;
        st[2] += acc_l;
        st[3] += acc_g;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            st[4 + k] += sum[k];
            st[4 + D + k] += sumsq[k];
        }
#pragma unroll
        for (int k = 0; k < D * (D + 1) / 2; ++k) st[4 + 2 * D + k] += gram[k];
    }
}

// ---- GLMCMC (iSIR) step for a user model: GLMCMC.py:58-104 with weight_sampling :7-22 --------------------------------
// gp_* (gq when it is not a DiagGaussian) hold the Importance_Proposal here.  Candidate j of step i is a pure function of (chain, i, j) through Philox, so
// the K weights are computed first and only the selected candidate is rebuilt — no per-candidate storage.
__device__ __forceinline__ float glabc_candidate(const UserRun& R, u32 g0, u32 g1, u32 i, int j, float* th, float* y, float& pk)
{
    constexpr int NZ = D + NN, NB = (NZ + 3) / 4;
    float z[NB * 4];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const uint4 w = glabc_philox(g0, g1, i, 0x100u + (u32)(j * NB + b), R.key0, R.key1);
        glabc_box_muller(w.x, w.y, z[4 * b], z[4 * b + 1]);
        glabc_box_muller(w.z, w.w, z[4 * b + 2], z[4 * b + 3]);
    }
#if GLABC_GP_KIND == GLABC_DIST_DIAG_GAUSSIAN
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        th[k] = fmaf(R.gp_scale[k], z[k], R.gp_loc[k]);     // Importance_Proposal.forward, GLMCMC.py:66
        q = fmaf(z[k], z[k], q);
    }
    glabc_user_simulate(th, z + D, R.params, y);            // :71
    pk = glabc_target(R, th, y);                            // log prior + log kernel
    return pk + 0.5f * q;                                   // log-weight up to the proposal's constant (it cancels in the ratio)
#else
    GlabcWords ws(g0, g1, i, GLABC_SLOT_CAND + (u32)j * GLABC_CAND_BLOCKS, R.key0, R.key1);
    float tj[D];
    const float lq = glabc::dist_forward<D>(R.gq, ws, tj);
#pragma unroll
    for (int k = 0; k < D; ++k) th[k] = tj[k];
    glabc_user_simulate(th, z + D, R.params, y);
    pk = glabc_target(R, th, y);
    return pk - lq;                                         // log prior + log K - log q, GLMCMC.py:66-74
#endif
}
#if GLABC_GP_KIND != GLABC_DIST_DIAG_GAUSSIAN
// log-weight of the current state, GLMCMC.py:60-64: +inf outside the support of q, so that global move selects nothing
// (the reference's resample after inf / inf); a NaN weight counts as 0, as the candidates'
__device__ __forceinline__ float glabc_state_logw(const UserRun& R, const float (&th)[D], float pk)
{
    const float lw = pk - glabc::dist_log_prob<D>(R.gq, th);
    return lw == lw ? lw : -INFINITY;
}
#endif
extern "C" __global__ void __launch_bounds__(128) glabc_k_isir_user(const __grid_constant__ UserRun R)
{
    const int chain = blockIdx.x * blockDim.x + threadIdx.x;
    if (chain >= R.n_chains) return;
    const u64 gid = ((u64)R.chain_hi0 << 32 | R.chain_lo0) + (u64)chain;
    const u32 g0 = (u32)gid, g1 = (u32)(gid >> 32);
    const int NK = R.n_candidates;
    float th[D], y[YD];
#pragma unroll
    for (int k = 0; k < D; ++k) th[k] = R.theta[(long long)chain * D + k];
#pragma unroll
    for (int k = 0; k < YD; ++k) y[k] = R.y[(long long)chain * YD + k];
    float pk = glabc_target(R, th, y);
    float lw_old = R.aux[(long long)chain * 8 + 0];
    bool local = R.aux[(long long)chain * 8 + 1] != 0.f;
    float n_glob = 0.f, acc_l = 0.f, acc_g = 0.f, sum[D], sumsq[D], gram[D * (D + 1) / 2];
#pragma unroll
    for (int k = 0; k < D; ++k) sum[k] = sumsq[k] = 0.f;
#pragma unroll
    for (int k = 0; k < D * (D + 1) / 2; ++k) gram[k] = 0.f;
    const long long cstride = R.trace_layout == 2 ? (long long)D : R.trace_chains * D;
    float* row = nullptr;
    if (R.trace_layout != 0) {
        const long long r0 = (long long)R.first_step - (R.write_row0 ? 1 : 0) - R.trace_row_base;
        row = R.trace_layout == 2 ? R.trace + ((R.trace_chain_off + chain) * R.trace_rows + r0) * D
                                  : R.trace + (r0 * R.trace_chains + R.trace_chain_off + chain) * D;
        if (R.write_row0) {
#pragma unroll
            for (int k = 0; k < D; ++k) row[k] = th[k];
            row += cstride;
        }
    }
    for (u32 i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
        const uint4 w0 = glabc_philox(g0, g1, i, 1u, R.key0, R.key1);
        const bool is_global = R.gf_all_global || (w0.x < R.gf_thr);              // GLMCMC.py:59
        float dl[D];
#pragma unroll
        for (int k = 0; k < D; ++k) dl[k] = 0.f;
        bool moved = false;
        if (is_global) {
            if (local) {                                                          // :60-64: log-weight of the current state
#if GLABC_GP_KIND == GLABC_DIST_DIAG_GAUSSIAN
                float qo = 0.f;
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    const float r = (th[k] - R.gp_loc[k]) * R.gp_inv_scale[k];
                    qo = fmaf(r, r, qo);
                }
                lw_old = pk + 0.5f * qo;
#else
                lw_old = glabc_state_logw(R, th, pk);
#endif
            }
            local = false;
            // shifted weights (the reference exponentiates un-shifted in float32, :78; the shift only removes underflow)
            float lw[17], thc[D], yc[YD], pkc, mx = lw_old;
            lw[0] = lw_old;
            for (int j = 0; j < NK; ++j) {
                lw[j + 1] = glabc_candidate(R, g0, g1, i, j, thc, yc, pkc);
                if (!(lw[j + 1] == lw[j + 1])) lw[j + 1] = -INFINITY;             // :80-81 NaN weight -> 0
                mx = fmaxf(mx, lw[j + 1]);
            }
            if (mx > -INFINITY) {
                double S = 0.0;
                for (int j = 0; j <= NK; ++j) S += (double)__expf(lw[j] - mx);
                const uint4 wu = glabc_philox(g0, g1, i, 0x80000000u, R.key0, R.key1);
                const double u = ((double)wu.x * 4294967296.0 + (double)wu.y) * (1.0 / 18446744073709551616.0);
                const double thr = u * S;                                         // weight_sampling, :7-22
                double run = 0.0;
                int ind = -1;
                for (int j = 0; j <= NK; ++j) {
                    run += (double)__expf(lw[j] - mx);
                    if (ind < 0 && thr < run) ind = j;
                }
                if (ind > 0) {                                                    // :84-88
                    const float lwn = glabc_candidate(R, g0, g1, i, ind - 1, thc, yc, pkc);
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        dl[k] = thc[k] - th[k];
                        th[k] = thc[k];
                    }
#pragma unroll
                    for (int k = 0; k < YD; ++k) y[k] = yc[k];
                    pk = pkc;
                    lw_old = lwn;
                    moved = true;
                }
            }
        } else {                                                                  // local random walk, :90-104
            constexpr int NZ = D + NN, NB = (NZ + 3) / 4;
            float z[NB * 4], thp[D], yp[YD];
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const uint4 w = glabc_philox(g0, g1, i, 2u + b, R.key0, R.key1);
                glabc_box_muller(w.x, w.y, z[4 * b], z[4 * b + 1]);
                glabc_box_muller(w.z, w.w, z[4 * b + 2], z[4 * b + 3]);
            }
#if GLABC_LP_KIND == GLABC_DIST_DIAG_GAUSSIAN
#pragma unroll
            for (int k = 0; k < D; ++k) thp[k] = th[k] + fmaf(R.lp_scale[k], z[k], R.lp_loc[k]);
            // GLMCMC.py:92-93: while the prior answers with the sentinel, draw the local proposal again (fresh normals from
            // further Philox blocks of the same step; 64 redraws at most, then the proposal stands and is rejected)
            for (u32 redraw = 0; redraw < 64u && glabc_user_prior_log_prob(thp, R.params) == GLABC_PRIOR_SENTINEL; ++redraw) {
                float zr[((D + 3) / 4) * 4];
#pragma unroll
                for (int b = 0; b < (D + 3) / 4; ++b) {
                    const uint4 w = glabc_philox(g0, g1, i, 0x40000000u + redraw * (u32)((D + 3) / 4) + b, R.key0, R.key1);
                    glabc_box_muller(w.x, w.y, zr[4 * b], zr[4 * b + 1]);
                    glabc_box_muller(w.z, w.w, zr[4 * b + 2], zr[4 * b + 3]);
                }
#pragma unroll
                for (int k = 0; k < D; ++k) thp[k] = th[k] + fmaf(R.lp_scale[k], zr[k], R.lp_loc[k]);
            }
#else
            GlabcWords ws(g0, g1, i, GLABC_SLOT_PROP, R.key0, R.key1);
            float zl[D];
            (void)glabc::dist_forward<D>(R.lq, ws, zl);
#pragma unroll
            for (int k = 0; k < D; ++k) thp[k] = th[k] + zl[k];
            for (u32 redraw = 0; redraw < 64u && glabc_user_prior_log_prob(thp, R.params) == GLABC_PRIOR_SENTINEL; ++redraw) {
                (void)glabc::dist_forward<D>(R.lq, ws, zl);   // GLMCMC.py:92-93, from the stream's next words
#pragma unroll
                for (int k = 0; k < D; ++k) thp[k] = th[k] + zl[k];
            }
#endif
            glabc_user_simulate(thp, z + D, R.params, yp);
            const float pkp = glabc_target(R, thp, yp);
            const float log_u = __logf(__uint2float_rn(w0.y >> 8) * 0x1p-24f);
            if (log_u < pkp - pk) {
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    dl[k] = thp[k] - th[k];
                    th[k] = thp[k];
                }
#pragma unroll
                for (int k = 0; k < YD; ++k) y[k] = yp[k];
                pk = pkp;
                local = true;                                                     // :100
                moved = true;
            }
        }
#pragma unroll
        for (int k = 0; k < D; ++k) {
            sum[k] += th[k];
            sumsq[k] = fmaf(th[k], th[k], sumsq[k]);
        }
        int t = 0;
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = a; b < D; ++b, ++t) gram[t] = fmaf(dl[a], dl[b], gram[t]);
        n_glob += is_global ? 1.f : 0.f;
        acc_g += (moved && is_global) ? 1.f : 0.f;
        acc_l += (moved && !is_global) ? 1.f : 0.f;
        if (row != nullptr) {
#pragma unroll
            for (int k = 0; k < D; ++k) row[k] = th[k];
            row += cstride;
        }
    }
#pragma unroll
    for (int k = 0; k < D; ++k) R.theta[(long long)chain * D + k] = th[k];
#pragma unroll
    for (int k = 0; k < YD; ++k) R.y[(long long)chain * YD + k] = y[k];
    R.aux[(long long)chain * 8 + 0] = lw_old;
    R.aux[(long long)chain * 8 + 1] = local ? 1.f : 0.f;
    if (R.stats != nullptr) {
        float* st = R.stats + (long long)chain * (4 + 2 * D + D * (D + 1) / 2);
        st[0] += R.last_step >= R.first_step ? (float)(R.last_step + 1u - R.first_step) : 0.f;
        st[1] += n_glob;
        st[2] += acc_l;
        st[3] += acc_g;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            st[4 + k] += sum[k];
            st[4 + D + k] += sumsq[k];
        }
#pragma unroll
        for (int k = 0; k < D * (D + 1) / 2; ++k) st[4 + 2 * D + k] += gram[k];
    }
}

// ---- GLMALA step for a user model: GLMALA.py:150-200, gradient :46-95 ------------------------------------------------
// A thread per chain for the iSIR global move and the tail of the MALA move; the WARP for the gradient
// (numberical_gradient_logABC): the chains of a warp that drew a local move are served one after the other, the num_grad
// common-random-number draws of a dimension dealt over the 32 lanes.  gp_* hold the Importance_Proposal.
__device__ __forceinline__ void glabc_grad_sums(const UserRun& R, u32 g0, u32 g1, u32 i, u32 slot0, const float* th, int lane,
                                                bool mine, float (*sums)[4], float (*cpm)[2])
{
    constexpr int NB = (NN + 3) / 4 > 0 ? (NN + 3) / 4 : 1;
    for (int k = 0; k < D; ++k) {
        float tp[D], tm[D], yy[YD], zero[NB * 4];
#pragma unroll
        for (int q = 0; q < D; ++q) {
            tp[q] = q == k ? th[q] + 0.1f : th[q];          // GLMALA.py:63-67
            tm[q] = q == k ? th[q] - 0.1f : th[q];
        }
#pragma unroll
        for (int q = 0; q < NB * 4; ++q) zero[q] = 0.f;
        glabc_user_simulate(tp, zero, R.params, yy);
        const float cp = glabc_user_discrepancy(yy, R.params);
        glabc_user_simulate(tm, zero, R.params, yy);
        const float cm = glabc_user_discrepancy(yy, R.params);
        float f1p = 0.f, f2p = 0.f, f1m = 0.f, f2m = 0.f;
        for (int j = lane; j < R.num_grad; j += 32) {
            float z[NB * 4];
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const uint4 w = glabc_philox(g0, g1, i, slot0 + (u32)((k * R.num_grad + j) * NB + b), R.key0, R.key1);
                glabc_box_muller(w.x, w.y, z[4 * b], z[4 * b + 1]);
                glabc_box_muller(w.z, w.w, z[4 * b + 2], z[4 * b + 3]);
            }
            glabc_user_simulate(tp, z, R.params, yy);        // :78-79
            const float xp = glabc_user_discrepancy(yy, R.params) - cp;
            glabc_user_simulate(tm, z, R.params, yy);        // :80-83: the same draws (common random numbers)
            const float xm = glabc_user_discrepancy(yy, R.params) - cm;
            f1p += xp; f2p = fmaf(xp, xp, f2p);
            f1m += xm; f2m = fmaf(xm, xm, f2m);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            f1p += __shfl_xor_sync(0xffffffffu, f1p, off);
            f2p += __shfl_xor_sync(0xffffffffu, f2p, off);
            f1m += __shfl_xor_sync(0xffffffffu, f1m, off);
            f2m += __shfl_xor_sync(0xffffffffu, f2m, off);
        }
        if (mine) {
            sums[k][0] = f1p; sums[k][1] = f2p; sums[k][2] = f1m; sums[k][3] = f2m;
            cpm[k][0] = cp; cpm[k][1] = cm;
        }
    }
}
extern "C" __global__ void __launch_bounds__(64) glabc_k_mala_user(const __grid_constant__ UserRun R)
{
    const int lane = threadIdx.x & 31;
    const int chain = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = chain < R.n_chains;
    const int cidx = active ? chain : R.n_chains - 1;
    const u64 gid = ((u64)R.chain_hi0 << 32 | R.chain_lo0) + (u64)cidx;
    const u32 g0 = (u32)gid, g1 = (u32)(gid >> 32);
    const u64 gid0 = ((u64)R.chain_hi0 << 32 | R.chain_lo0) + (u64)(chain - lane);   // the warp's first chain, the same on every lane (tail lanes included)
    const int NK = R.n_candidates;
    float th[D], y[YD], grad[D];
#pragma unroll
    for (int k = 0; k < D; ++k) th[k] = R.theta[(long long)cidx * D + k];
#pragma unroll
    for (int k = 0; k < YD; ++k) y[k] = R.y[(long long)cidx * YD + k];
    float pk = glabc_target(R, th, y);
    float lw_old = R.aux[(long long)cidx * 8 + 0];
    bool local = R.aux[(long long)cidx * 8 + 1] != 0.f, have_grad = R.aux[(long long)cidx * 8 + 2] != 0.f;
#pragma unroll
    for (int k = 0; k < D; ++k) grad[k] = R.aux[(long long)cidx * 8 + 3 + k];
    float n_glob = 0.f, acc_l = 0.f, acc_g = 0.f, sum[D], sumsq[D], gram[D * (D + 1) / 2];
#pragma unroll
    for (int k = 0; k < D; ++k) sum[k] = sumsq[k] = 0.f;
#pragma unroll
    for (int k = 0; k < D * (D + 1) / 2; ++k) gram[k] = 0.f;
    const long long cstride = R.trace_layout == 2 ? (long long)D : R.trace_chains * D;
    float* row = nullptr;
    if (R.trace_layout != 0 && active) {
        const long long r0 = (long long)R.first_step - (R.write_row0 ? 1 : 0) - R.trace_row_base;
        row = R.trace_layout == 2 ? R.trace + ((R.trace_chain_off + chain) * R.trace_rows + r0) * D
                                  : R.trace + (r0 * R.trace_chains + R.trace_chain_off + chain) * D;
        if (R.write_row0) {
#pragma unroll
            for (int k = 0; k < D; ++k) row[k] = th[k];
            row += cstride;
        }
    }
    const float tau = R.tau, half_tau2 = 0.5f * R.tau * R.tau, inv_tau = 1.0f / R.tau;
    const float rn = 1.0f / (float)R.num_grad, rn1 = 1.0f / (float)(R.num_grad - 1);
    auto grad_from = [&](const float* tt, float (*sums)[4], float (*cpm)[2], float* out) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            float ta[D], tb[D];
#pragma unroll
            for (int q = 0; q < D; ++q) {
                ta[q] = q == k ? __fadd_rn(tt[q], 0.00001f) : tt[q];      // GLMALA.py:84-85, float32 finite difference
                tb[q] = q == k ? __fsub_rn(tt[q], 0.00001f) : tt[q];
            }
            const float gprior = __fdiv_rn(__fsub_rn(glabc_user_prior_log_prob(ta, R.params), glabc_user_prior_log_prob(tb, R.params)), 2e-5f);
            const float mup = fmaf(sums[k][0], rn, cpm[k][0]), mum = fmaf(sums[k][2], rn, cpm[k][1]);
            const float vp = fmaf(fmaf(-sums[k][0] * rn, sums[k][0], sums[k][1]), rn1, R.eps2);
            const float vm = fmaf(fmaf(-sums[k][2] * rn, sums[k][2], sums[k][3]), rn1, R.eps2);
            const float dl = __logf(vp / vm) + (mup * mup / vp - mum * mum / vm);   // :90-93: -2 (log p+ - log p-)
            out[k] = fmaf(dl, -2.5f, gprior);                                     // :94-95
        }
    };
    for (u32 i = R.first_step; i <= R.last_step && R.last_step >= R.first_step; ++i) {
        const uint4 w0 = glabc_philox(g0, g1, i, 1u, R.key0, R.key1);
        const bool coin = R.gf_all_global || (w0.x < R.gf_thr);                   // GLMALA.py:151
        const bool is_global = active && coin, is_local = active && !coin;
        float dl[D];
#pragma unroll
        for (int k = 0; k < D; ++k) dl[k] = 0.f;
        bool moved = false;
        if (is_global) {                                                          // :151-180, as glabc_k_isir_user
            if (local) {
#if GLABC_GP_KIND == GLABC_DIST_DIAG_GAUSSIAN
                float qo = 0.f;
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    const float r = (th[k] - R.gp_loc[k]) * R.gp_inv_scale[k];
                    qo = fmaf(r, r, qo);
                }
                lw_old = pk + 0.5f * qo;
#else
                lw_old = glabc_state_logw(R, th, pk);
#endif
            }
            local = false;
            float lw[17], thc[D], yc[YD], pkc, mx = lw_old;
            lw[0] = lw_old;
            for (int j = 0; j < NK; ++j) {
                lw[j + 1] = glabc_candidate(R, g0, g1, i, j, thc, yc, pkc);
                if (!(lw[j + 1] == lw[j + 1])) lw[j + 1] = -INFINITY;
                mx = fmaxf(mx, lw[j + 1]);
            }
            if (mx > -INFINITY) {
                double S = 0.0;
                for (int j = 0; j <= NK; ++j) S += (double)__expf(lw[j] - mx);
                const uint4 wu = glabc_philox(g0, g1, i, 0x80000000u, R.key0, R.key1);
                const double u = ((double)wu.x * 4294967296.0 + (double)wu.y) * (1.0 / 18446744073709551616.0);
                const double thr = u * S;
                double run = 0.0;
                int ind = -1;
                for (int j = 0; j <= NK; ++j) {
                    run += (double)__expf(lw[j] - mx);
                    if (ind < 0 && thr < run) ind = j;
                }
                if (ind > 0) {                                                    // :175-179: the cached gradient is NOT refreshed (B-6)
                    const float lwn = glabc_candidate(R, g0, g1, i, ind - 1, thc, yc, pkc);
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        dl[k] = thc[k] - th[k];
                        th[k] = thc[k];
                    }
#pragma unroll
                    for (int k = 0; k < YD; ++k) y[k] = yc[k];
                    pk = pkc;
                    lw_old = lwn;
                    moved = true;
                }
            }
        }
        const unsigned pend = __ballot_sync(0xffffffffu, is_local);
        if (pend != 0u) {                                                         // :182-200
            constexpr int NZ = D + NN, NB = (NZ + 3) / 4;
            float z[NB * 4], thp[D], gp[D], lq_fwd = 0.f;
#pragma unroll
            for (int q = 0; q < NB * 4; ++q) z[q] = 0.f;
            if (is_local) {
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const uint4 w = glabc_philox(g0, g1, i, 2u + b, R.key0, R.key1);
                    glabc_box_muller(w.x, w.y, z[4 * b], z[4 * b + 1]);
                    glabc_box_muller(w.z, w.w, z[4 * b + 2], z[4 * b + 3]);
                }
#pragma unroll
                for (int k = 0; k < D; ++k) lq_fwd = fmaf(z[k], z[k], lq_fwd);
                lq_fwd *= -0.5f;                                                  // log N(z; 0, I) up to the constant (it cancels)
            }
#pragma unroll
            for (int k = 0; k < D; ++k) thp[k] = th[k];
            const unsigned need0 = __ballot_sync(0xffffffffu, is_local && !have_grad);
            for (int pass = need0 != 0u ? 0 : 1; pass < 2; ++pass) {
                if (pass == 1 && is_local) {
#pragma unroll
                    for (int k = 0; k < D; ++k) thp[k] = fmaf(grad[k], half_tau2, fmaf(z[k], tau, th[k]));   // :43
                }
                unsigned todo = pass == 0 ? need0 : pend;
                float sums[D][4], cpm[D][2];
                while (todo != 0u) {
                    const int src = __ffs(todo) - 1;
                    todo &= todo - 1u;
                    float ts[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) ts[k] = __shfl_sync(0xffffffffu, thp[k], src);
                    const u64 gs = gid0 + (u64)src;
                    glabc_grad_sums(R, (u32)gs, (u32)(gs >> 32), i, pass == 0 ? 0x20000u : 0x10000u, ts, lane, lane == src, sums, cpm);
                }
                if (pass == 0 ? (is_local && !have_grad) : is_local) {
                    float gout[D];
                    grad_from(thp, sums, cpm, gout);
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        if (pass == 0) grad[k] = gout[k];
                        gp[k] = gout[k];
                    }
                    have_grad = true;
                }
            }
            if (is_local) {
                float yp[YD], lr = 0.f;
                glabc_user_simulate(thp, z + D, R.params, yp);                    // :188-189
                const float pkp = glabc_target(R, thp, yp);
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    const float r = ((th[k] - thp[k]) - gp[k] * half_tau2) * inv_tau;   // log_proposal, :97-116
                    lr = fmaf(r, r, lr);
                }
                lr *= -0.5f;
                const float log_u = __logf(__uint2float_rn(w0.y >> 8) * 0x1p-24f);
                if (log_u < (pkp - pk) + (lr - lq_fwd)) {                         // :190-199
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        dl[k] = thp[k] - th[k];
                        th[k] = thp[k];
                        grad[k] = gp[k];
                    }
#pragma unroll
                    for (int k = 0; k < YD; ++k) y[k] = yp[k];
                    pk = pkp;
                    moved = true;
                }
            }
        }
#pragma unroll
        for (int k = 0; k < D; ++k) {
            sum[k] += th[k];
            sumsq[k] = fmaf(th[k], th[k], sumsq[k]);
        }
        int t = 0;
#pragma unroll
        for (int a = 0; a < D; ++a)
#pragma unroll
            for (int b = a; b < D; ++b, ++t) gram[t] = fmaf(dl[a], dl[b], gram[t]);
        n_glob += is_global ? 1.f : 0.f;
        acc_g += (moved && is_global) ? 1.f : 0.f;
        acc_l += (moved && !is_global) ? 1.f : 0.f;
        if (row != nullptr) {
#pragma unroll
            for (int k = 0; k < D; ++k) row[k] = th[k];
            row += cstride;
        }
    }
    if (!active) return;
#pragma unroll
    for (int k = 0; k < D; ++k) R.theta[(long long)chain * D + k] = th[k];
#pragma unroll
    for (int k = 0; k < YD; ++k) R.y[(long long)chain * YD + k] = y[k];
    R.aux[(long long)chain * 8 + 0] = lw_old;
    R.aux[(long long)chain * 8 + 1] = local ? 1.f : 0.f;
    R.aux[(long long)chain * 8 + 2] = have_grad ? 1.f : 0.f;
#pragma unroll
    for (int k = 0; k < D; ++k) R.aux[(long long)chain * 8 + 3 + k] = grad[k];
    if (R.stats != nullptr) {
        float* st = R.stats + (long long)chain * (4 + 2 * D + D * (D + 1) / 2);
        st[0] += R.last_step >= R.first_step ? (float)(R.last_step + 1u - R.first_step) : 0.f;
        st[1] += n_glob;
        st[2] += acc_l;
        st[3] += acc_g;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            st[4 + k] += sum[k];
            st[4 + D + k] += sumsq[k];
        }
#pragma unroll
        for (int k = 0; k < D * (D + 1) / 2; ++k) st[4 + 2 * D + k] += gram[k];
    }
}

// ---- the model's functions outside a run: generate_samples / prior_log_prob / discrepancy / calculate_log_kernel ------
// One row per thread, grid-stride.  SIMULATE row r draws its NN normals as a step kernel draws its simulator noise, from the
// Philox blocks (row_base + r, step 0, slot 2 + b): step 0 is no step's, see the slot table.
extern "C" __global__ void __launch_bounds__(256) glabc_k_eval_user(const __grid_constant__ UserEval E)
{
    const u64 row0 = (u64)E.row_hi << 32 | E.row_lo;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (E.op == GLABC_USER_SIMULATE) {
        constexpr int NB = (NN + 3) / 4;
        for (long long r = first; r < E.n; r += stride) {
            float th[D], y[YD], z[NB > 0 ? NB * 4 : 4];
#pragma unroll
            for (int k = 0; k < D; ++k) th[k] = E.in[r * D + k];
            const u64 gid = row0 + (u64)r;
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const uint4 w = glabc_philox((u32)gid, (u32)(gid >> 32), 0u, 2u + b, E.key0, E.key1);
                glabc_box_muller(w.x, w.y, z[4 * b], z[4 * b + 1]);
                glabc_box_muller(w.z, w.w, z[4 * b + 2], z[4 * b + 3]);
            }
            glabc_user_simulate(th, z, E.params, y);
#pragma unroll
            for (int k = 0; k < YD; ++k) E.out[r * YD + k] = y[k];
        }
    } else if (E.op == GLABC_USER_PRIOR) {
        for (long long r = first; r < E.n; r += stride) {
            float th[D];
#pragma unroll
            for (int k = 0; k < D; ++k) th[k] = E.in[r * D + k];
            E.out[r] = glabc_user_prior_log_prob(th, E.params);
        }
    } else {                                   // DISCREPANCY, LOG_KERNEL (the kernel term of glabc_target)
        const bool log_kernel = E.op == GLABC_USER_LOG_KERNEL;
        for (long long r = first; r < E.n; r += stride) {
            float y[YD];
#pragma unroll
            for (int k = 0; k < YD; ++k) y[k] = E.in[r * YD + k];
            const float dis = glabc_user_discrepancy(y, E.params);
            E.out[r] = log_kernel ? fmaf(E.kern_m, dis * dis, E.kern_c) : dis;
        }
    }
}
)GLABC";

// ---- lazily bound NVRTC / driver entry points --------------------------------------------------------------------
struct Dyn {
    bool tried = false, rt_ok = false, ok = false;   // rt_ok: NVRTC usable (compile checks need no driver); ok: + driver
    std::string why;
    decltype(&nvrtcCreateProgram) createProgram = nullptr;
    decltype(&nvrtcCompileProgram) compileProgram = nullptr;
    decltype(&nvrtcGetProgramLogSize) getLogSize = nullptr;
    decltype(&nvrtcGetProgramLog) getLog = nullptr;
    decltype(&nvrtcGetCUBINSize) getCubinSize = nullptr;
    decltype(&nvrtcGetCUBIN) getCubin = nullptr;
    decltype(&nvrtcDestroyProgram) destroyProgram = nullptr;
    decltype(&nvrtcGetErrorString) errString = nullptr;
    CUresult (*moduleLoadData)(CUmodule*, const void*) = nullptr;
    CUresult (*moduleGetFunction)(CUfunction*, CUmodule, const char*) = nullptr;
    CUresult (*launchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream, void**,
                             void**) = nullptr;
    CUresult (*getErrorString)(CUresult, const char**) = nullptr;
};

Dyn& dyn()
{
    static Dyn d;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    if (d.tried) return d;
    d.tried = true;
    void* rt = nullptr;
    for (const char* name : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"}) {
        rt = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
        if (rt) break;
    }
    if (!rt) {
        d.why = "libnvrtc.so.12 could not be loaded (needed to compile a user model)";
        return d;
    }
#define GLABC_SYM(lib, field, sym)                                             \
    d.field = reinterpret_cast<decltype(d.field)>(dlsym(lib, sym));           \
    if (!d.field) {                                                           \
        d.why = std::string("symbol ") + sym + " not found";                  \
        return d;                                                             \
    }
    GLABC_SYM(rt, createProgram, "nvrtcCreateProgram")
    GLABC_SYM(rt, compileProgram, "nvrtcCompileProgram")
    GLABC_SYM(rt, getLogSize, "nvrtcGetProgramLogSize")
    GLABC_SYM(rt, getLog, "nvrtcGetProgramLog")
    GLABC_SYM(rt, getCubinSize, "nvrtcGetCUBINSize")
    GLABC_SYM(rt, getCubin, "nvrtcGetCUBIN")
    GLABC_SYM(rt, destroyProgram, "nvrtcDestroyProgram")
    GLABC_SYM(rt, errString, "nvrtcGetErrorString")
    d.rt_ok = true;
    void* cu = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!cu) {
        d.why = "libcuda.so.1 could not be loaded";
        return d;
    }
    GLABC_SYM(cu, moduleLoadData, "cuModuleLoadData")
    GLABC_SYM(cu, moduleGetFunction, "cuModuleGetFunction")
    GLABC_SYM(cu, launchKernel, "cuLaunchKernel")
    GLABC_SYM(cu, getErrorString, "cuGetErrorString")
#undef GLABC_SYM
    d.ok = true;
    return d;
}

struct Compiled {
    CUmodule mod = nullptr;
    CUfunction fn = nullptr;        // glabc_k_global_user
    CUfunction fn_isir = nullptr;   // glabc_k_isir_user
    CUfunction fn_mala = nullptr;   // glabc_k_mala_user (models with theta_dim <= 5: the gradient is cached in the aux slots)
    CUfunction fn_eval = nullptr;   // glabc_k_eval_user
};
std::mutex g_cache_mu;
// key: model_key() + proposal kinds, so the modules of one model are adjacent in the map
std::map<std::string, Compiled> g_cache;

// device | arch | dims | n_noise | source length | source: names a model, whatever the proposal kinds it was compiled for
std::string model_key(int device, int cc, const glabc_user_model_t& um)
{
    const size_t len = strlen(um.source);
    char head[160];
    snprintf(head, sizeof(head), "%d|%d|%d|%d|%d|%zu|", device, cc, um.theta_dim, um.y_dim, um.n_noise, len);
    return std::string(head) + std::string(um.source, len);
}

std::string cu_err(Dyn& d, CUresult r)
{
    const char* s = nullptr;
    d.getErrorString(r, &s);
    return s ? s : "unknown driver error";
}

}  // namespace

// NVRTC: prelude + user source + step kernel -> cubin for sm_<cc>, the Local / Global-or-Importance proposal kinds fixed
static int compile_to_cubin(Dyn& d, int cc, const glabc_user_model_t& um, int lp_kind, int gp_kind, std::vector<char>& cubin,
                            std::string& err)
{
    const std::string src = std::string(kPrelude) + "\n// ---- user model ----\n" + um.source + "\n// ---- step kernel ----\n" + kKernel;
    nvrtcProgram prog = nullptr;
    const char* hdr_src[] = {kDistDevice};
    const char* hdr_name[] = {"dist_device.cuh"};
    nvrtcResult r = d.createProgram(&prog, src.c_str(), "glabc_user_model.cu", 1, hdr_src, hdr_name);
    if (r != NVRTC_SUCCESS) {
        err = std::string("nvrtcCreateProgram: ") + d.errString(r);
        return GLABC_ERR_CUDA;
    }
    char arch[48], dD[24], dY[24], dN[24], dLP[32], dGP[32];
    snprintf(arch, sizeof(arch), "--gpu-architecture=sm_%d%s", cc, cc >= 90 ? "a" : "");
    snprintf(dD, sizeof(dD), "-DD=%d", um.theta_dim);
    snprintf(dY, sizeof(dY), "-DYD=%d", um.y_dim);
    snprintf(dN, sizeof(dN), "-DNN=%d", um.n_noise);
    snprintf(dLP, sizeof(dLP), "-DGLABC_LP_KIND=%d", lp_kind);
    snprintf(dGP, sizeof(dGP), "-DGLABC_GP_KIND=%d", gp_kind);
    // dist_device.cuh's constants, from include/glabc.h
    char kinds[4][48], sizes[3][40];
    snprintf(kinds[0], sizeof(kinds[0]), "-DGLABC_DIST_DIAG_GAUSSIAN=%d", GLABC_DIST_DIAG_GAUSSIAN);
    snprintf(kinds[1], sizeof(kinds[1]), "-DGLABC_DIST_UNIFORM=%d", GLABC_DIST_UNIFORM);
    snprintf(kinds[2], sizeof(kinds[2]), "-DGLABC_DIST_GAMMA=%d", GLABC_DIST_GAMMA);
    snprintf(kinds[3], sizeof(kinds[3]), "-DGLABC_DIST_GAUSSIAN_MIXTURE=%d", GLABC_DIST_GAUSSIAN_MIXTURE);
    snprintf(sizes[0], sizeof(sizes[0]), "-DGLABC_MAX_DIM=%d", GLABC_MAX_DIM);
    snprintf(sizes[1], sizeof(sizes[1]), "-DGLABC_MAX_MODES=%d", GLABC_MAX_MODES);
    snprintf(sizes[2], sizeof(sizes[2]), "-DGLABC_USER_MAX_PARAMS=%d", GLABC_USER_MAX_PARAMS);
    char ops[4][40];   // glabc_k_eval_user's operations
    snprintf(ops[0], sizeof(ops[0]), "-DGLABC_USER_SIMULATE=%d", GLABC_USER_SIMULATE);
    snprintf(ops[1], sizeof(ops[1]), "-DGLABC_USER_PRIOR=%d", GLABC_USER_PRIOR);
    snprintf(ops[2], sizeof(ops[2]), "-DGLABC_USER_DISCREPANCY=%d", GLABC_USER_DISCREPANCY);
    snprintf(ops[3], sizeof(ops[3]), "-DGLABC_USER_LOG_KERNEL=%d", GLABC_USER_LOG_KERNEL);
    const char* opts[] = {arch, dD, dY, dN, dLP, dGP, kinds[0], kinds[1], kinds[2], kinds[3], sizes[0], sizes[1], sizes[2],
                          ops[0], ops[1], ops[2], ops[3], "--std=c++17", "--use_fast_math", "-lineinfo"};
    r = d.compileProgram(prog, static_cast<int>(sizeof(opts) / sizeof(opts[0])), opts);
    if (r != NVRTC_SUCCESS) {
        size_t n = 0;
        d.getLogSize(prog, &n);
        std::string log(n, '\0');
        if (n) d.getLog(prog, &log[0]);
        d.destroyProgram(&prog);
        err = std::string("user model does not compile: ") + log.c_str();
        return GLABC_ERR_INVALID;
    }
    size_t nb = 0;
    d.getCubinSize(prog, &nb);
    cubin.resize(nb);
    d.getCubin(prog, cubin.data());
    d.destroyProgram(&prog);
    return GLABC_OK;
}

int user_model_check(int cc, const glabc_user_model_t& um, int lp_kind, int gp_kind, std::string& err)
{
    Dyn& d = dyn();
    if (!d.rt_ok) {
        err = d.why;
        return GLABC_ERR_UNSUPPORTED;
    }
    std::vector<char> cubin;
    return compile_to_cubin(d, cc, um, lp_kind, gp_kind, cubin, err);
}

// the module of (model, proposal kinds): from the cache, or compiled and loaded.  Called with g_cache_mu held.
static int load_module(Dyn& d, int device, int cc, const glabc_user_model_t& um, int lp_kind, int gp_kind, const Compiled** out,
                       std::string& err)
{
    char kinds[32];
    snprintf(kinds, sizeof(kinds), "|%d|%d", lp_kind, gp_kind);
    const std::string key = model_key(device, cc, um) + kinds;
    auto it = g_cache.find(key);
    if (it != g_cache.end()) {
        *out = &it->second;
        return GLABC_OK;
    }
    std::vector<char> cubin;
    int st = compile_to_cubin(d, cc, um, lp_kind, gp_kind, cubin, err);
    if (st) return st;
    Compiled c;
    CUresult cr = d.moduleLoadData(&c.mod, cubin.data());
    if (cr != CUDA_SUCCESS) {
        err = "cuModuleLoadData: " + cu_err(d, cr);
        return GLABC_ERR_CUDA;
    }
    const std::pair<CUfunction*, const char*> fns[] = {{&c.fn, "glabc_k_global_user"}, {&c.fn_isir, "glabc_k_isir_user"},
                                                       {&c.fn_mala, "glabc_k_mala_user"}, {&c.fn_eval, "glabc_k_eval_user"}};
    for (const auto& f : fns) {
        cr = d.moduleGetFunction(f.first, c.mod, f.second);
        if (cr != CUDA_SUCCESS) {
            err = "cuModuleGetFunction: " + cu_err(d, cr);
            return GLABC_ERR_CUDA;
        }
    }
    *out = &(g_cache[key] = c);
    return GLABC_OK;
}

int user_model_compile(int device, int cc, const glabc_user_model_t& um, int lp_kind, int gp_kind, int kind, void** fn_out,
                       std::string& err)
{
    Dyn& d = dyn();
    if (!d.ok) {
        err = d.why;
        return GLABC_ERR_UNSUPPORTED;
    }
    std::lock_guard<std::mutex> lock(g_cache_mu);
    const Compiled* c = nullptr;
    const int st = load_module(d, device, cc, um, lp_kind, gp_kind, &c, err);
    if (st) return st;
    *fn_out = kind == 2 ? c->fn_mala : kind == 1 ? c->fn_isir : c->fn;
    return GLABC_OK;
}

int user_model_eval_fn(int device, int cc, const glabc_user_model_t& um, void** fn_out, std::string& err)
{
    Dyn& d = dyn();
    if (!d.ok) {
        err = d.why;
        return GLABC_ERR_UNSUPPORTED;
    }
    std::lock_guard<std::mutex> lock(g_cache_mu);
    const std::string prefix = model_key(device, cc, um) + "|";   // then only the proposal kinds follow
    auto it = g_cache.lower_bound(prefix);
    if (it != g_cache.end() && it->first.compare(0, prefix.size(), prefix) == 0) {
        *fn_out = it->second.fn_eval;
        return GLABC_OK;
    }
    const Compiled* c = nullptr;
    const int st = load_module(d, device, cc, um, GLABC_DIST_DIAG_GAUSSIAN, GLABC_DIST_DIAG_GAUSSIAN, &c, err);
    if (st) return st;
    *fn_out = c->fn_eval;
    return GLABC_OK;
}

static int launch(void* fn, void* param, unsigned grid, int block, cudaStream_t st, std::string& err)
{
    Dyn& d = dyn();
    if (!d.ok) {
        err = d.why;
        return GLABC_ERR_UNSUPPORTED;
    }
    void* args[] = {param};
    const CUresult cr = d.launchKernel(static_cast<CUfunction>(fn), grid, 1, 1, static_cast<unsigned>(block), 1, 1, 0,
                                       reinterpret_cast<CUstream>(st), args, nullptr);
    if (cr != CUDA_SUCCESS) {
        err = "cuLaunchKernel: " + cu_err(d, cr);
        return GLABC_ERR_CUDA;
    }
    return GLABC_OK;
}

int user_model_launch(void* fn, const UserRun& R, int block, cudaStream_t st, std::string& err)
{
    if (R.n_chains <= 0) return GLABC_OK;
    UserRun copy = R;
    return launch(fn, &copy, static_cast<unsigned>((R.n_chains + block - 1) / block), block, st, err);
}

int user_model_eval_launch(void* fn, const UserEval& E, int sm_count, cudaStream_t st, std::string& err)
{
    if (E.n <= 0) return GLABC_OK;
    constexpr int block = 256;   // glabc_k_eval_user's __launch_bounds__
    // a grid-stride loop: enough blocks to fill every SM several times over, fewer for a small n
    const long long want = (E.n + block - 1) / block, cap = 32LL * (sm_count > 0 ? sm_count : 1);
    UserEval copy = E;
    return launch(fn, &copy, static_cast<unsigned>(want < cap ? want : cap), block, st, err);
}

}  // namespace glabc
