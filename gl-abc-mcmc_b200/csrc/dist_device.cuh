// Device versions of the reference's proposal distributions (distribution.py: Uniform :50-86, Gamma :90-137,
// DiagGaussian :143-181, GaussianMixture :206-293), and the kernel parameter of the run-time compiled user-model kernels.
// One text for both compilers: nvcc builds the general kernels from it (step_generic.cuh), and build.py embeds it in
// libglabc.so for NVRTC, which compiles it into every user model (user_model.cu).  So it includes nothing: the
// GLABC_DIST_* kinds, GLABC_MAX_MODES, GLABC_MAX_DIM and GLABC_USER_MAX_PARAMS come from include/glabc.h (nvcc) or as
// -D options built from its constants (NVRTC); INFINITY and NAN from the CUDA headers or the NVRTC prelude.
//   Uniform          z = low + (high - low) * U                         log p = -log prod(high - low), -inf outside
//   Gamma            Marsaglia-Tsang squeeze per coordinate (+ the U^(1/a) boost for shape < 1)
//                                                                        log p = sum a log b - lgamma(a) + (a-1) log z - b z
//   GaussianMixture  mode by inverse CDF of the soft-maxed weights, then a diagonal Gaussian; log p = logsumexp over modes
#pragma once
// (ND, not D, names a dimension here: the user-model source defines D, YD and NN as macros.)
#if !defined(GLABC_MAX_MODES) || !defined(GLABC_MAX_DIM) || !defined(GLABC_USER_MAX_PARAMS)
#error "dist_device.cuh needs the size macros and GLABC_DIST_* kinds of include/glabc.h"
#endif

namespace glabc {

// MAXD: the widest distribution a kernel takes.  DistConsts (= DistConstsT<4>) for the built-in kernels,
// DistConstsT<GLABC_MAX_DIM> for the user-model kernels.
template <int MAXD>
struct DistConstsT {
    int kind, dim, n_modes;
    float a[MAXD], b[MAXD], c[MAXD];  // Gauss: loc, log_scale, scale; Uniform: low, high, c[0] = log p;
                                      // Gamma: shape, rate, c = a log b - lgamma(a)
    float half_log_2pi;               // float32(-0.5 d log 2 pi)
    float mix_loc[GLABC_MAX_MODES][MAXD], mix_inv_scale[GLABC_MAX_MODES][MAXD], mix_scale[GLABC_MAX_MODES][MAXD];
    float mix_c[GLABC_MAX_MODES];    // -0.5 d log 2 pi + log w_m - sum log_scale_m
    float mix_cdf[GLABC_MAX_MODES];  // inclusive prefix sums of the weights
};

template <int ND, int MAXD>
__device__ __forceinline__ float dist_log_prob(const DistConstsT<MAXD>& q, const float (&z)[ND])
{
    switch (q.kind) {
    case GLABC_DIST_DIAG_GAUSSIAN: {
        float s = 0.0f;
#pragma unroll
        for (int i = 0; i < ND; ++i) {
            const float r = (z[i] - q.a[i]) / q.c[i];
            s += q.b[i] + 0.5f * (r * r);
        }
        return q.half_log_2pi - s;
    }
    case GLABC_DIST_UNIFORM: {
        bool out = false;
#pragma unroll
        for (int i = 0; i < ND; ++i) out |= (z[i] < q.a[i]) || (z[i] > q.b[i]);  // distribution.py:82-85
        return out ? -INFINITY : q.c[0];
    }
    case GLABC_DIST_GAMMA: {
        float s = 0.0f;
#pragma unroll
        for (int i = 0; i < ND; ++i) {
            float lp;
            if (z[i] > 0.0f) lp = q.c[i] + (q.a[i] - 1.0f) * logf(z[i]) - q.b[i] * z[i];
            else if (z[i] == 0.0f && q.a[i] == 1.0f) lp = q.c[i];   // pdf(0) = b for shape 1
            else lp = -INFINITY;                                     // pdf == 0 -> -inf, distribution.py:133-136
            s += lp;
        }
        return s;
    }
    case GLABC_DIST_GAUSSIAN_MIXTURE: {
        float t[GLABC_MAX_MODES], mx = -INFINITY;
        for (int m = 0; m < q.n_modes; ++m) {
            float s = 0.0f;
#pragma unroll
            for (int i = 0; i < ND; ++i) {
                const float r = (z[i] - q.mix_loc[m][i]) * q.mix_inv_scale[m][i];
                s = fmaf(r, r, s);
            }
            t[m] = fmaf(-0.5f, s, q.mix_c[m]);  // distribution.py:283-288
            mx = fmaxf(mx, t[m]);
        }
        if (mx == -INFINITY) return -INFINITY;
        float acc = 0.0f;
        for (int m = 0; m < q.n_modes; ++m) acc += expf(t[m] - mx);
        return mx + logf(acc);
    }
    }
    return NAN;
}

// forward(): one draw and its log-density.  WS is the word source of one (chain, step): uniform() in [0, 1),
// uniform_open() in (0, 1) and normal(), each a function of the words consumed so far.
// Words one draw consumes at most (normal() takes two words per pair of normals, uniform() / uniform_open() one):
// DiagGaussian 2 ND, Uniform ND, GaussianMixture 1 + 2 ND, Gamma ND (64 (2 + 1) + 1) -- 64 squeeze iterations of a
// normal and a uniform, then the shape < 1 boost -- i.e. 1544 words = 386 Philox blocks at ND = 8.
template <int ND, int MAXD, class WS>
__device__ __forceinline__ float dist_forward(const DistConstsT<MAXD>& q, WS& ws, float (&z)[ND])
{
    switch (q.kind) {
    case GLABC_DIST_DIAG_GAUSSIAN: {
        float s = 0.0f;
#pragma unroll
        for (int i = 0; i < ND; ++i) {
            const float e = ws.normal();
            z[i] = fmaf(q.c[i], e, q.a[i]);
            s += q.b[i] + 0.5f * (e * e);  // log p from eps, distribution.py:171-173
        }
        return q.half_log_2pi - s;
    }
    case GLABC_DIST_UNIFORM: {
#pragma unroll
        for (int i = 0; i < ND; ++i) z[i] = fmaf(q.b[i] - q.a[i], ws.uniform(), q.a[i]);  // distribution.py:73-77
        return q.c[0];
    }
    case GLABC_DIST_GAMMA: {
#pragma unroll
        for (int i = 0; i < ND; ++i) {
            // Marsaglia & Tsang (2000): Gamma(a >= 1) by squeeze-rejection from a cubed normal; shape < 1 via Gamma(a + 1) * U^(1/a)
            const float a0 = q.a[i];
            const float a = a0 < 1.0f ? a0 + 1.0f : a0;
            const float dd = a - (1.0f / 3.0f), cc = rsqrtf(9.0f * dd);
            float g = dd;
            for (int it = 0; it < 64; ++it) {
                const float x = ws.normal();
                const float t = fmaf(cc, x, 1.0f);
                if (t <= 0.0f) continue;
                const float v = t * t * t;
                const float u = ws.uniform_open();
                if (logf(u) < 0.5f * x * x + dd - dd * v + dd * logf(v)) {
                    g = dd * v;
                    break;
                }
            }
            if (a0 < 1.0f) g *= powf(ws.uniform_open(), 1.0f / a0);
            z[i] = g / q.b[i];  // scale = 1 / rate, distribution.py:118
        }
        return dist_log_prob<ND>(q, z);
    }
    case GLABC_DIST_GAUSSIAN_MIXTURE: {
        const float u = ws.uniform();
        int m = q.n_modes - 1;
        for (int j = q.n_modes - 2; j >= 0; --j)
            if (u < q.mix_cdf[j]) m = j;  // torch.multinomial(weights, 1): first mode whose cumulative weight exceeds u
#pragma unroll
        for (int i = 0; i < ND; ++i) z[i] = fmaf(ws.normal(), q.mix_scale[m][i], q.mix_loc[m][i]);  // distribution.py:258-260
        return dist_log_prob<ND>(q, z);
    }
    }
    return NAN;
}

// kernel parameter of the user-model kernels glabc_k_{global,isir,mala}_user (user_model.cu)
struct UserRun {
    int n_chains;
    unsigned first_step, last_step, chain_lo0, chain_hi0, key0, key1, gf_thr;
    int gf_all_global, write_row0, trace_layout, pad;
    long long trace_rows, trace_chains, trace_chain_off, trace_row_base;
    float *theta, *y, *trace, *stats;
    float lp_loc[GLABC_MAX_DIM], lp_scale[GLABC_MAX_DIM], gp_loc[GLABC_MAX_DIM], gp_scale[GLABC_MAX_DIM], gp_inv_scale[GLABC_MAX_DIM];
    float kern_c, kern_m;     // log K(dis) = kern_c + kern_m * dis^2   (Mixture.py:38-53)
    float params[GLABC_USER_MAX_PARAMS];
    float* aux;               // iSIR: [C][8] carried state (slot 0 cached log-weight, slot 1 `local` flag;
                              // GLMALA adds slot 2 = gradient cached, slots 3.. = the cached gradient)
    int n_candidates, pad2;
    float tau, eps2;          // GLMALA: step size, ABCset.epsilon ** 2
    int num_grad, pad3;
    // appended after the fields above so none of them moves: a Uniform / Gamma / GaussianMixture slot
    DistConstsT<GLABC_MAX_DIM> lq, gq;   // Local_Proposal; Global_Proposal (GlobalMCMC) or Importance_Proposal
};

// kernel parameter of the user-model evaluation kernel glabc_k_eval_user (user_model.cu): one row per thread,
// op = glabc_user_op (include/glabc.h)
struct UserEval {
    long long n;              // rows
    int op, pad;
    unsigned row_lo, row_hi;  // SIMULATE: Philox chain id of row 0 (row r draws from row_base + r)
    unsigned key0, key1;      // SIMULATE: the seed
    const float* in;          // theta [n][D] (SIMULATE, PRIOR) or y [n][YD] (DISCREPANCY, LOG_KERNEL)
    float* out;               // y [n][YD] (SIMULATE) or [n]
    float kern_c, kern_m;     // LOG_KERNEL: as UserRun
    float params[GLABC_USER_MAX_PARAMS];
};

}  // namespace glabc
