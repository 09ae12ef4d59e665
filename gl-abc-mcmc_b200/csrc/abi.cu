// The C-ABI of include/glabc.h: context, plugin binding, argument validation, the device and
// host-buffer sampler entry points.  No torch, no C++ types across the boundary.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <initializer_list>
#include <new>
#include <immintrin.h>

#include <atomic>
#include <chrono>
#include <cstdlib>
#include <string>
#include <thread>
#include <vector>

#include "launch.cuh"
#include "flow.cuh"
#include "flow_param_layout.h"
#include "step_aglmcmc.cuh"
#include "step_generic.cuh"
#include "step_mala.cuh"
#include "user_model.cuh"

using namespace glabc;

// A grow-only scratch buffer of the context, in device memory or (Pinned) in page-locked host memory.  reserve() keeps no
// contents: it frees the old buffer and allocates the larger one, and leaves the buffer empty (cap 0) when that fails.
template <class T, bool Pinned = false>
struct Scratch {
    T* p = nullptr;
    size_t cap = 0;
    Scratch() = default;
    Scratch(const Scratch&) = delete;
    Scratch& operator=(const Scratch&) = delete;
    ~Scratch() { release(); }
    cudaError_t reserve(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        release();
        const cudaError_t e = Pinned ? cudaHostAlloc(&p, n * sizeof(T), cudaHostAllocDefault) : cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        else p = nullptr;
        return e;
    }
    void release()
    {
        if (p) (void)(Pinned ? cudaFreeHost(p) : cudaFree(p));
        p = nullptr;
        cap = 0;
    }
};

struct glabc_ctx {
    int device = 0;
    int sm_count = 0, clock_khz = 0, cc = 0;
    std::string err;
    glabc_model_t model{};
    glabc_model_t model_pod{};   // as glabc_model_set bound it: a DiagGaussian prior set later changes `model` only
    bool has_model = false;
    glabc_dist_t dist[GLABC_SLOT_COUNT]{};
    bool has_dist[GLABC_SLOT_COUNT] = {false, false, false};
    glabc_dist_t prior{};     // a Uniform / Gamma / GaussianMixture prior of the model (glabc_model_prior_set)
    bool has_prior = false;   // false: the DiagGaussian of `model` is the prior
    // scratch of the host-buffer entry points
    Scratch<float> d_state;       // theta | y | aux | stats
    Scratch<double> d_state64;    // GLMALA carried float64 state
    // AGLMCMC block / KDE workspace (one allocation), KDE sampling scratch of the public entry points
    void* ag_mem = nullptr;
    size_t ag_bytes = 0, ag_used = 0;
    AgWorkspace ag{};
    int ag_dim = 0;
    Scratch<double> kde_cdf;
    Scratch<double> rs_scratch;   // block prefixes of glabc_resample
    Scratch<float> kde_part;      // partial sums of the point-split log_prob
    // RealNVP flow weights (device copies owned by the context)
    float* flow_mem = nullptr;
    size_t flow_floats = 0;
    FlowDev flow{};
    bool has_flow = false;
    int flow_blocks = 0;
    int32_t flow_precision = GLABC_FLOW_PRECISE;   // the mode that meets north_star's 1e-5 on log-densities is the default
    // training state of the flow (glabc_flow_train_init): Adam moments, gradient, per-CTA partial gradients, forward scratch
    float* tr_mem = nullptr;       // m | v | grad | loss
    float* tr_partial = nullptr;
    int tr_slices = 0;
    Scratch<float> tr_fwd;         // z [n][2] | log q [n]
    int64_t tr_step = 0;
    float tr_lr = 5e-4f, tr_beta1 = 0.9f, tr_beta2 = 0.999f, tr_eps = 1e-8f, tr_wd = 1e-5f;
    bool tr_ready = false;
    Scratch<float> d_trace[2];
    cudaStream_t s_compute = nullptr, s_copy = nullptr;
    // host entry, event transport (run_global_host_hybrid): device state + event buffer of the event-encoded chains, pinned staging
    cudaStream_t s_ev = nullptr;
    cudaEvent_t ev_group[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    Scratch<float> d_ev;
    Scratch<float, true> h_ev;
    cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
};

static int fail(glabc_ctx* ctx, int status, const char* fmt, ...)
{
    if (ctx) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        ctx->err = buf;
    }
    return status;
}

#define CUDA_TRY(ctx, expr)                                                                         \
    do {                                                                                            \
        cudaError_t e_ = (expr);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail((ctx), GLABC_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_));   \
    } while (0)

extern "C" {

int glabc_version(void) { return GLABC_ABI_VERSION; }

const char* glabc_status_string(int status)
{
    switch (status) {
    case GLABC_OK: return "ok";
    case GLABC_ERR_INVALID: return "invalid argument";
    case GLABC_ERR_UNSUPPORTED: return "model family / distribution / dimension not fused";
    case GLABC_ERR_CUDA: return "CUDA runtime error";
    case GLABC_ERR_NO_DEVICE: return "no usable CUDA device";
    default: return "unknown status";
    }
}

int glabc_ctx_create(int device, glabc_ctx** out)
{
    if (!out) return GLABC_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        (void)cudaGetLastError();
        return GLABC_ERR_NO_DEVICE;
    }
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) return GLABC_ERR_NO_DEVICE;
    if (device >= n) return GLABC_ERR_INVALID;
    glabc_ctx* ctx = new (std::nothrow) glabc_ctx();
    if (!ctx) return GLABC_ERR_INVALID;
    ctx->device = device;
    int major = 0, minor = 0;
    if (cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
        cudaDeviceGetAttribute(&ctx->clock_khz, cudaDevAttrClockRate, device) != cudaSuccess ||
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess ||
        cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device) != cudaSuccess) {
        delete ctx;
        return GLABC_ERR_CUDA;
    }
    ctx->cc = major * 10 + minor;
    *out = ctx;
    return GLABC_OK;
}

int glabc_ctx_destroy(glabc_ctx* ctx)
{
    if (!ctx) return GLABC_OK;
    cudaSetDevice(ctx->device);
    if (ctx->ag_mem) cudaFree(ctx->ag_mem);
    if (ctx->flow_mem) cudaFree(ctx->flow_mem);
    if (ctx->tr_mem) cudaFree(ctx->tr_mem);
    if (ctx->tr_partial) cudaFree(ctx->tr_partial);
    for (int b = 0; b < 2; ++b) {
        if (ctx->ev_done[b]) cudaEventDestroy(ctx->ev_done[b]);
        if (ctx->ev_free[b]) cudaEventDestroy(ctx->ev_free[b]);
    }
    if (ctx->s_ev) cudaStreamDestroy(ctx->s_ev);
    for (auto& e : ctx->ev_group)
        if (e) cudaEventDestroy(e);
    if (ctx->s_compute) cudaStreamDestroy(ctx->s_compute);
    if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
    delete ctx;   // the Scratch members free their buffers (the device is current)
    return GLABC_OK;
}

const char* glabc_last_error(const glabc_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int glabc_device_info(const glabc_ctx* ctx, int32_t* sm_count, int32_t* clock_khz, int32_t* cc)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (sm_count) *sm_count = ctx->sm_count;
    if (clock_khz) *clock_khz = ctx->clock_khz;
    if (cc) *cc = ctx->cc;
    return GLABC_OK;
}

int glabc_model_set(glabc_ctx* ctx, const glabc_model_t* model, size_t nbytes)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!model || nbytes != sizeof(glabc_model_t))
        return fail(ctx, GLABC_ERR_INVALID, "glabc_model_set: struct size %zu, expected %zu (ABI mismatch)", nbytes,
                    sizeof(glabc_model_t));
    if (model->family != GLABC_MODEL_ABS_NORMAL && model->family != GLABC_MODEL_ID_NORMAL)
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "model family %d is not fused", model->family);
    if (model->theta_dim < 1 || model->theta_dim > 4 || model->y_dim != model->theta_dim)
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "theta_dim=%d y_dim=%d: fused kernels exist for theta_dim == y_dim in 1..4",
                    model->theta_dim, model->y_dim);
    if (!(model->eps_scale > 0.0f)) return fail(ctx, GLABC_ERR_INVALID, "epsilon must be positive");
    for (int i = 0; i < model->theta_dim; ++i)
        if (!(model->prior_scale[i] > 0.0f)) return fail(ctx, GLABC_ERR_INVALID, "prior scale must be positive");
    ctx->model = ctx->model_pod = *model;
    ctx->has_model = true;
    ctx->has_prior = false;
    return GLABC_OK;
}

}  // extern "C"

// the checks of a glabc_dist_t shared by glabc_dist_set and glabc_model_prior_set
static int check_dist(glabc_ctx* ctx, const char* who, const glabc_dist_t* dist, size_t nbytes)
{
    if (!dist || nbytes != sizeof(glabc_dist_t))
        return fail(ctx, GLABC_ERR_INVALID, "%s: struct size %zu, expected %zu (ABI mismatch)", who, nbytes, sizeof(glabc_dist_t));
    if (dist->dim < 1 || dist->dim > GLABC_MAX_DIM) return fail(ctx, GLABC_ERR_UNSUPPORTED, "%s: dim %d outside 1..%d", who, dist->dim, GLABC_MAX_DIM);
    switch (dist->kind) {
    case GLABC_DIST_DIAG_GAUSSIAN:
        for (int i = 0; i < dist->dim; ++i)
            if (!(dist->c[i] > 0.0f)) return fail(ctx, GLABC_ERR_INVALID, "proposal scale must be positive");
        break;
    case GLABC_DIST_UNIFORM:
        for (int i = 0; i < dist->dim; ++i)
            if (!(dist->b[i] > dist->a[i])) return fail(ctx, GLABC_ERR_INVALID, "Uniform needs high > low");
        break;
    case GLABC_DIST_GAMMA:
        for (int i = 0; i < dist->dim; ++i)
            if (!(dist->a[i] > 0.0f) || !(dist->b[i] > 0.0f)) return fail(ctx, GLABC_ERR_INVALID, "Gamma needs shape, rate > 0");
        break;
    case GLABC_DIST_GAUSSIAN_MIXTURE:
        if (dist->n_modes < 1 || dist->n_modes > GLABC_MAX_MODES) return fail(ctx, GLABC_ERR_INVALID, "GaussianMixture: 1..%d modes", GLABC_MAX_MODES);
        for (int m = 0; m < dist->n_modes; ++m)
            for (int i = 0; i < dist->dim; ++i)
                if (!(dist->mix_scale[m][i] > 0.0f)) return fail(ctx, GLABC_ERR_INVALID, "GaussianMixture scale must be positive");
        break;
    default:
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "unknown distribution kind %d", dist->kind);
    }
    return GLABC_OK;
}

// The built-in kernels take distributions of dim <= kGenMaxDim (DistConsts); only the user-model kernels take wider ones
static int check_builtin_dim(glabc_ctx* ctx, const char* who, const glabc_dist_t& dist)
{
    if (dist.dim > kGenMaxDim)
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "%s: a distribution of dim %d; the built-in kernels take dim 1..%d (user models up to %d)", who,
                    dist.dim, kGenMaxDim, GLABC_MAX_DIM);
    return GLABC_OK;
}

extern "C" {

int glabc_dist_set(glabc_ctx* ctx, int slot, const glabc_dist_t* dist, size_t nbytes)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (slot < 0 || slot >= GLABC_SLOT_COUNT) return fail(ctx, GLABC_ERR_INVALID, "bad proposal slot %d", slot);
    const int st = check_dist(ctx, "glabc_dist_set", dist, nbytes);
    if (st) return st;
    ctx->dist[slot] = *dist;
    ctx->has_dist[slot] = true;
    return GLABC_OK;
}

int glabc_model_prior_set(glabc_ctx* ctx, const glabc_dist_t* prior, size_t nbytes)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_model) return fail(ctx, GLABC_ERR_INVALID, "glabc_model_prior_set: no model bound: call glabc_model_set first");
    glabc_model_t& m = ctx->model;
    if (!prior) {   // back to the DiagGaussian of the glabc_model_set POD
        m = ctx->model_pod;
        ctx->has_prior = false;
        return GLABC_OK;
    }
    if (nbytes == sizeof(glabc_dist_t) && check_builtin_dim(ctx, "glabc_model_prior_set", *prior)) return GLABC_ERR_UNSUPPORTED;
    if (nbytes == sizeof(glabc_dist_t) && prior->dim != m.theta_dim)
        return fail(ctx, GLABC_ERR_INVALID, "glabc_model_prior_set: prior dim %d does not match theta_dim %d", prior->dim, m.theta_dim);
    const int st = check_dist(ctx, "glabc_model_prior_set", prior, nbytes);
    if (st) return st;
    if (prior->kind == GLABC_DIST_DIAG_GAUSSIAN) {   // the tuned kernels take it from the model POD, as if given there
        for (int i = 0; i < m.theta_dim; ++i) {
            m.prior_loc[i] = prior->a[i];
            m.prior_log_scale[i] = prior->b[i];
            m.prior_scale[i] = prior->c[i];
        }
        ctx->has_prior = false;
        return GLABC_OK;
    }
    ctx->prior = *prior;
    ctx->has_prior = true;
    return GLABC_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// lowering of the PODs to kernel constants
// ---------------------------------------------------------------------------------------------
static float half_log_2pi(int d) { return static_cast<float>(-0.5 * d * std::log(2.0 * M_PI)); }

static GaussConsts make_gauss(const float* loc, const float* log_scale, const float* scale, int d)
{
    GaussConsts g{};
    double sum_ls = 0.0;
    for (int i = 0; i < d; ++i) {
        g.loc[i] = loc[i];
        g.log_scale[i] = log_scale[i];
        g.scale[i] = scale[i];
        g.inv_scale[i] = 1.0f / scale[i];
        g.nloc_inv[i] = -loc[i] / scale[i];
        sum_ls += log_scale[i];
    }
    g.c = half_log_2pi(d);
    g.c_fast = static_cast<float>(static_cast<double>(g.c) - sum_ls);
    return g;
}

// glabc_dist_t -> constants of a kernel that takes distributions of dim <= MAXD (dist_device.cuh): DistConsts for the
// built-in kernels, DistConstsT<GLABC_MAX_DIM> for the user-model kernels
template <int MAXD = kGenMaxDim>
static DistConstsT<MAXD> make_dist(const glabc_dist_t& p)
{
    DistConstsT<MAXD> q{};
    q.kind = p.kind;
    q.dim = p.dim;
    q.n_modes = p.n_modes;
    q.half_log_2pi = half_log_2pi(p.dim);
    for (int i = 0; i < p.dim && i < MAXD; ++i) {
        q.a[i] = p.a[i];
        q.b[i] = p.b[i];
        q.c[i] = p.c[i];
        if (p.kind == GLABC_DIST_GAMMA)
            q.c[i] = static_cast<float>(static_cast<double>(p.a[i]) * std::log(static_cast<double>(p.b[i])) - std::lgamma(static_cast<double>(p.a[i])));
    }
    if (p.kind == GLABC_DIST_GAUSSIAN_MIXTURE) {
        double run = 0.0;
        for (int m = 0; m < p.n_modes; ++m) {
            double sls = 0.0;
            for (int i = 0; i < p.dim && i < MAXD; ++i) {
                q.mix_loc[m][i] = p.mix_loc[m][i];
                q.mix_scale[m][i] = p.mix_scale[m][i];
                q.mix_inv_scale[m][i] = 1.0f / p.mix_scale[m][i];
                sls += p.mix_log_scale[m][i];
            }
            q.mix_c[m] = static_cast<float>(-0.5 * p.dim * std::log(2.0 * M_PI) + static_cast<double>(p.mix_log_w[m]) - sls);
            run += p.mix_w[m];
            q.mix_cdf[m] = static_cast<float>(run);
        }
    }
    return q;
}

static bool all_gaussian(const glabc_ctx* ctx, std::initializer_list<int> slots)
{
    for (int s : slots)
        if (ctx->dist[s].kind != GLABC_DIST_DIAG_GAUSSIAN) return false;
    return true;
}

static ModelConsts make_model(const glabc_model_t& m)
{
    ModelConsts k{};
    k.family = m.family;
    for (int i = 0; i < m.y_dim; ++i) {
        k.y_obs[i] = m.y_obs[i];
        k.noise_loc[i] = m.noise_loc[i];
        k.noise_scale[i] = m.noise_scale[i];
    }
    k.eps_log_scale = m.eps_log_scale;
    k.eps_scale = m.eps_scale;
    k.c_kern = half_log_2pi(1);
    k.kern_fast_c = k.c_kern - m.eps_log_scale;
    k.kern_fast_m = static_cast<float>(-0.5 / (static_cast<double>(m.eps_scale) * m.eps_scale));
    k.prior = make_gauss(m.prior_loc, m.prior_log_scale, m.prior_scale, m.theta_dim);
    return k;
}

// the `prior` argument of the launchers: the bound Uniform / Gamma / GaussianMixture, or kind DiagGaussian for the model's own
static DistConsts make_prior(const glabc_ctx* ctx)
{
    if (ctx->has_prior) return make_dist(ctx->prior);
    DistConsts q{};
    q.kind = GLABC_DIST_DIAG_GAUSSIAN;
    return q;
}

// A Uniform / Gamma / GaussianMixture prior runs FAST arithmetic with the native RNG and records nothing: the STRICT / replay
// kernels and the tapes and dumps are fused for the model's DiagGaussian prior.  Checked before anything is launched.
static int check_prior_run(glabc_ctx* ctx, const char* who, const glabc_run_t* run, bool dumps)
{
    if (ctx->has_prior && (run->arith_mode == GLABC_ARITH_STRICT || run->rng_mode == GLABC_RNG_REPLAY || run->tape_dump || dumps))
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "%s with a Uniform / Gamma / GaussianMixture prior runs FAST arithmetic with the native RNG "
                                                "and writes no tape or parity dump", who);
    return GLABC_OK;
}

// native branch coin: U_b = k * 2^-16 (k < 2^16);  U_b < gf  <=>  k < ceil(gf * 2^16)  (cf. SURVEY.md B-15)
static uint32_t gf_threshold16(float gf)
{
    if (!(gf > 0.0f)) return 0u;
    if (gf >= 1.0f) return 1u << 16;
    return static_cast<uint32_t>(std::ceil(static_cast<double>(gf) * 65536.0));
}

static int make_run_params(glabc_ctx* ctx, const glabc_run_t* run, int dim, int tape_slots, RunParams* out, int* block,
                           bool events_ok = false)
{
    if (!run) return fail(ctx, GLABC_ERR_INVALID, "null run description");
    if (run->trace_layout == GLABC_TRACE_EVENTS && !events_ok)
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "GLABC_TRACE_EVENTS is written by run_global (DiagGaussian proposals) and run_isir only");
    if (run->n_chains < 0 || run->n_chains > INT32_MAX) return fail(ctx, GLABC_ERR_INVALID, "n_chains out of range");
    if (run->n_steps < 0 || run->step_base < 0 || run->step_base + run->n_steps >= 0xFFFFFFF0ll)
        return fail(ctx, GLABC_ERR_INVALID, "step_base + n_steps must stay below 2^32 (Philox block counter)");
    if (run->n_steps >= (1 << 24))
        return fail(ctx, GLABC_ERR_INVALID, "at most 16,777,215 transitions per launch (float32 step counters): chunk the run "
                                            "with step_base, the chain continues bit-identically");
    if (run->trace_layout < GLABC_TRACE_NONE || run->trace_layout > GLABC_TRACE_EVENTS)
        return fail(ctx, GLABC_ERR_INVALID, "bad trace_layout %d", run->trace_layout);
    if (run->n_chains == 0) {   // nothing to do: empty buffers may be null pointers
        RunParams r{};
        *out = r;
        *block = 64;
        return GLABC_OK;
    }
    if (!run->theta || !run->y) return fail(ctx, GLABC_ERR_INVALID, "theta / y state pointers are required");
    if (run->trace_layout == GLABC_TRACE_EVENTS) {
        if (!run->trace || run->trace_rows < 2) return fail(ctx, GLABC_ERR_INVALID, "GLABC_TRACE_EVENTS needs trace [chains][trace_rows >= 2][1 + d]");
        if (run->rng_mode != GLABC_RNG_NATIVE || run->tape_dump) return fail(ctx, GLABC_ERR_UNSUPPORTED, "GLABC_TRACE_EVENTS: native RNG, no tape dump");
        if (run->trace_chain_off < 0 || run->trace_chain_off + run->n_chains > run->trace_chains)
            return fail(ctx, GLABC_ERR_INVALID, "chains fall outside the event buffer");
    } else if (run->trace_layout != GLABC_TRACE_NONE) {
        if (!run->trace) return fail(ctx, GLABC_ERR_INVALID, "trace pointer required for this trace_layout");
        const int64_t lo = run->step_base + (run->write_row0 ? 0 : 1) - run->trace_row_base;
        const int64_t hi = run->step_base + run->n_steps - run->trace_row_base;
        if (run->n_steps + (run->write_row0 ? 1 : 0) > 0 && (lo < 0 || hi >= run->trace_rows))
            return fail(ctx, GLABC_ERR_INVALID, "trace rows [%lld, %lld] fall outside the %lld-row buffer",
                        (long long)lo, (long long)hi, (long long)run->trace_rows);
        if (run->trace_chain_off < 0 || run->trace_chain_off + run->n_chains > run->trace_chains)
            return fail(ctx, GLABC_ERR_INVALID, "chains [%lld, +%lld) fall outside the %lld-chain trace buffer",
                        (long long)run->trace_chain_off, (long long)run->n_chains, (long long)run->trace_chains);
    }
    if (run->rng_mode != GLABC_RNG_NATIVE && run->rng_mode != GLABC_RNG_REPLAY)
        return fail(ctx, GLABC_ERR_INVALID, "bad rng_mode %d", run->rng_mode);
    if (run->arith_mode != GLABC_ARITH_FAST && run->arith_mode != GLABC_ARITH_STRICT)
        return fail(ctx, GLABC_ERR_INVALID, "bad arith_mode %d", run->arith_mode);
    if (run->rng_mode == GLABC_RNG_REPLAY && !run->tape32)
        return fail(ctx, GLABC_ERR_INVALID, "replay mode needs tape32 [n_steps][%d][n_chains]", tape_slots);
    int b = run->block_threads == 0 ? 64 : run->block_threads;
    if (b < 32 || b > 256 || (b & 31)) return fail(ctx, GLABC_ERR_INVALID, "block_threads must be a multiple of 32 in [32, 256]");
    *block = b;

    RunParams r{};
    r.n_chains = static_cast<int32_t>(run->n_chains);
    r.first_step = static_cast<uint32_t>(run->step_base + 1);
    r.last_step = static_cast<uint32_t>(run->step_base + run->n_steps);
    r.chain_lo0 = static_cast<uint32_t>(static_cast<uint64_t>(run->chain_id_base));
    r.chain_hi0 = static_cast<uint32_t>(static_cast<uint64_t>(run->chain_id_base) >> 32);
    r.rk = expand_key(make_uint2(static_cast<uint32_t>(run->seed), static_cast<uint32_t>(run->seed >> 32)));
    r.gf = run->global_frequency;
    const uint32_t thr16 = gf_threshold16(run->global_frequency);
    r.gf_all_global = thr16 >= (1u << 16);
    r.gf_thr_hi = r.gf_all_global ? 0xFFFFFFFFu : (thr16 << 16);
    r.write_row0 = run->write_row0 && run->trace_layout != GLABC_TRACE_NONE;
    r.trace_rows = run->trace_rows;
    r.trace_chains = run->trace_chains;
    r.trace_chain_off = run->trace_chain_off;
    r.trace_row_base = run->trace_row_base;
    r.theta = run->theta;
    r.y = run->y;
    r.aux = run->aux;
    r.trace = run->trace;
    r.stats = run->stats;
    r.tape32 = run->tape32;
    r.tape64 = run->tape64;
    r.debug = run->debug;
    r.tape_dump = run->tape_dump;
    r.tape64_dump = run->tape64_dump;
    r.n_candidates = run->n_candidates;
    r.trace_layout = run->trace_layout;
    r.state64 = run->state64;
    r.tape_grad0 = run->tape_grad0;
    r.tape_grad0_dump = run->tape_grad0_dump;
    r.debug64 = run->debug64;
    (void)dim;
    *out = r;
    return GLABC_OK;
}

// ---------------------------------------------------------------------------------------------
// sampler dispatch (device buffers)
// ---------------------------------------------------------------------------------------------
enum SamplerKind { SAMPLER_GLOBAL = 0, SAMPLER_ISIR = 1, SAMPLER_MALA = 2, SAMPLER_AGLMCMC = 3 };

static int run_device(glabc_ctx* ctx, SamplerKind kind, const glabc_run_t* run)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_model) return fail(ctx, GLABC_ERR_INVALID, "no model bound: call glabc_model_set first");
    const int d = ctx->model.theta_dim;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    RunParams R;
    int block = 0;
    switch (kind) {
    case SAMPLER_GLOBAL: {
        if (!ctx->has_dist[GLABC_SLOT_LOCAL] || !ctx->has_dist[GLABC_SLOT_GLOBAL])
            return fail(ctx, GLABC_ERR_INVALID, "run_global needs the LOCAL and GLOBAL proposal slots bound");
        const glabc_dist_t& lp = ctx->dist[GLABC_SLOT_LOCAL];
        const glabc_dist_t& gp = ctx->dist[GLABC_SLOT_GLOBAL];
        if (lp.dim != d || gp.dim != d) return fail(ctx, GLABC_ERR_INVALID, "proposal dim does not match theta_dim %d", d);
        const bool tuned = all_gaussian(ctx, {GLABC_SLOT_LOCAL, GLABC_SLOT_GLOBAL}) && !ctx->has_prior;
        int st = make_run_params(ctx, run, d, GLABC_TAPE_GLOBAL_SLOTS(d, d), &R, &block, tuned);
        if (st || (st = check_prior_run(ctx, "run_global", run, false))) return st;
        if (R.n_chains == 0) return GLABC_OK;
        if (!tuned) {
            // Uniform / Gamma / GaussianMixture proposals: the general kernel (float32; replay takes the proposal draws
            // themselves: tape32 [steps][2 + d][C] = U_b, eps_sim, U_a and tape64 [steps][d][C] = the draw in float64)
            if (run->tape_dump) return fail(ctx, GLABC_ERR_UNSUPPORTED, "tape dump exists for DiagGaussian proposals only");
            if (run->rng_mode == GLABC_RNG_REPLAY && !run->tape64)
                return fail(ctx, GLABC_ERR_INVALID, "replay with non-Gaussian proposals needs tape64 [n_steps][%d][n_chains] (the proposal draws)", d);
            GenericConsts G{};
            G.model = make_model(ctx->model);
            G.lp = make_dist(lp);
            G.gp = make_dist(gp);
            CUDA_TRY(ctx, launch_global_generic(G, make_prior(ctx), d, R, run->trace_layout, block, run->rng_mode == GLABC_RNG_REPLAY,
                                                static_cast<cudaStream_t>(run->stream)));
            return GLABC_OK;
        }
        CUDA_TRY(ctx, launch_global_mcmc(make_model(ctx->model), make_gauss(lp.a, lp.b, lp.c, d), make_gauss(gp.a, gp.b, gp.c, d),
                                         d, R, run->arith_mode == GLABC_ARITH_STRICT, run->rng_mode == GLABC_RNG_REPLAY,
                                         run->trace_layout, block, static_cast<cudaStream_t>(run->stream)));
        return GLABC_OK;
    }
    case SAMPLER_ISIR: {
        if (!ctx->has_dist[GLABC_SLOT_LOCAL] || !ctx->has_dist[GLABC_SLOT_IMPORTANCE])
            return fail(ctx, GLABC_ERR_INVALID, "run_isir needs the LOCAL and IMPORTANCE proposal slots bound");
        const glabc_dist_t& lp = ctx->dist[GLABC_SLOT_LOCAL];
        const glabc_dist_t& ip = ctx->dist[GLABC_SLOT_IMPORTANCE];
        if (lp.dim != d || ip.dim != d) return fail(ctx, GLABC_ERR_INVALID, "proposal dim does not match theta_dim %d", d);
        const bool tuned = all_gaussian(ctx, {GLABC_SLOT_LOCAL, GLABC_SLOT_IMPORTANCE}) && !ctx->has_prior;
        if (!run) return fail(ctx, GLABC_ERR_INVALID, "null run description");
        if (run->n_candidates < 1 || run->n_candidates > GLABC_MAX_K)
            return fail(ctx, GLABC_ERR_INVALID, "n_candidates (batch_size) must be in 1..%d", GLABC_MAX_K);
        if (!run->aux) return fail(ctx, GLABC_ERR_INVALID, "run_isir needs the aux state [C][%d] (log-weight, local flag)", GLABC_AUX_SLOTS);
        int st = make_run_params(ctx, run, d, GLABC_TAPE_ISIR_SLOTS(d, d, run->n_candidates), &R, &block, tuned);
        if (st || (st = check_prior_run(ctx, "run_isir", run, false))) return st;
        if (!tuned) {
            // Uniform / Gamma / GaussianMixture in the Local / Importance slots: the general kernel (replay takes the
            // proposal draws themselves: tape64 [steps][1 + K d][C] = resampling uniform, then the draws)
            if (run->tape_dump) return fail(ctx, GLABC_ERR_UNSUPPORTED, "tape dump exists for DiagGaussian proposals only");
            if (run->rng_mode == GLABC_RNG_REPLAY && !run->tape64)
                return fail(ctx, GLABC_ERR_INVALID, "replay of run_isir with non-Gaussian proposals needs tape64 [n_steps][1 + %d][n_chains]",
                            run->n_candidates * d);
            if (R.n_chains == 0) return GLABC_OK;
            IsirGenericConsts G{};
            G.model = make_model(ctx->model);
            G.lp = make_dist(lp);
            G.ip = make_dist(ip);
            CUDA_TRY(ctx, launch_isir_generic(G, make_prior(ctx), d, R, run->trace_layout, block, run->rng_mode == GLABC_RNG_REPLAY,
                                              static_cast<cudaStream_t>(run->stream)));
            return GLABC_OK;
        }
        if (run->rng_mode == GLABC_RNG_REPLAY && !run->tape64)
            return fail(ctx, GLABC_ERR_INVALID, "replay of run_isir needs tape64 (the float64 resampling uniforms)");
        if (R.n_chains == 0) return GLABC_OK;
        CUDA_TRY(ctx, launch_isir(make_model(ctx->model), make_gauss(lp.a, lp.b, lp.c, d), make_gauss(ip.a, ip.b, ip.c, d), d, R,
                                  run->arith_mode == GLABC_ARITH_STRICT, run->rng_mode == GLABC_RNG_REPLAY,
                                  run->trace_layout, block, static_cast<cudaStream_t>(run->stream)));
        return GLABC_OK;
    }
    case SAMPLER_MALA: {
        if (!ctx->has_dist[GLABC_SLOT_IMPORTANCE])
            return fail(ctx, GLABC_ERR_INVALID, "run_mala needs the IMPORTANCE proposal slot bound");
        const glabc_dist_t& ip = ctx->dist[GLABC_SLOT_IMPORTANCE];
        if (ip.dim != d) return fail(ctx, GLABC_ERR_INVALID, "proposal dim does not match theta_dim %d", d);
        if (!run) return fail(ctx, GLABC_ERR_INVALID, "null run description");
        const bool gip = !all_gaussian(ctx, {GLABC_SLOT_IMPORTANCE});
        if (gip && (run->arith_mode == GLABC_ARITH_STRICT || run->rng_mode == GLABC_RNG_REPLAY || run->tape_dump))
            return fail(ctx, GLABC_ERR_UNSUPPORTED, "run_mala with a non-Gaussian importance proposal runs FAST arithmetic with the native RNG "
                                                    "(the STRICT / replay / tape-dump kernel is fused for a DiagGaussian importance proposal)");
        if (run->n_candidates < 1 || run->n_candidates > GLABC_MAX_K)
            return fail(ctx, GLABC_ERR_INVALID, "n_candidates (batch_size) must be in 1..%d", GLABC_MAX_K);
        if (run->num_grad < 2 || run->num_grad > GLABC_MAX_NUM_GRAD)
            return fail(ctx, GLABC_ERR_INVALID, "num_grad must be in 2..%d (the variance is unbiased, GLMALA.py:88)", GLABC_MAX_NUM_GRAD);
        if (!(run->tau > 0.0f)) return fail(ctx, GLABC_ERR_INVALID, "tau must be positive");
        if (!run->aux || !run->state64)
            return fail(ctx, GLABC_ERR_INVALID, "run_mala needs aux [C][%d] and state64 [C][%d]", GLABC_AUX_SLOTS, GLABC_STATE64_SLOTS);
        int st = make_run_params(ctx, run, d, GLABC_TAPE_MALA_SLOTS(d, d, run->n_candidates, run->num_grad), &R, &block);
        if (st || (st = check_prior_run(ctx, "run_mala", run, false))) return st;
        if (run->rng_mode == GLABC_RNG_REPLAY && (!run->tape64 || !run->tape_grad0))
            return fail(ctx, GLABC_ERR_INVALID, "replay of run_mala needs tape64 and tape_grad0");
        if (run->tape_dump && !run->tape_grad0_dump)
            return fail(ctx, GLABC_ERR_INVALID, "tape_dump of run_mala also needs tape_grad0_dump");
        if (R.n_chains == 0) return GLABC_OK;
        if (run->block_threads == 0) block = 128;  // 4 chains (warps) per block
        MalaConsts K{};
        K.model = make_model(ctx->model);
        if (gip) {
            K.ip_generic = 1;
            K.ipg = make_dist(ip);
        } else {
            K.ip = make_gauss(ip.a, ip.b, ip.c, d);
        }
        const float zeros[GLABC_MAX_DIM] = {0}, ones[GLABC_MAX_DIM] = {1, 1, 1, 1, 1, 1, 1, 1};
        K.unit = make_gauss(zeros, zeros, ones, d);
        const double eps = ctx->model.epsilon > 0.0 ? ctx->model.epsilon : static_cast<double>(ctx->model.eps_scale);
        K.eps2 = eps * eps;
        K.tau = run->tau64 != 0.0 ? run->tau64 : static_cast<double>(run->tau);
        K.tau_f = run->tau;
        K.num_grad = run->num_grad;
        CUDA_TRY(ctx, launch_mala(K, make_prior(ctx), d, R, run->arith_mode == GLABC_ARITH_STRICT, run->rng_mode == GLABC_RNG_REPLAY, block,
                                  static_cast<cudaStream_t>(run->stream)));
        return GLABC_OK;
    }
    }
    return fail(ctx, GLABC_ERR_INVALID, "unknown sampler");
}

// ---------------------------------------------------------------------------------------------
// host-buffer entry points: the argument check, the chain state on the device, the time-chunk transport
// ---------------------------------------------------------------------------------------------
// Checks a host-buffer run before anything is allocated or launched, so that a bad argument leaves the caller's buffers
// untouched.  With n_chains == 0 there is nothing to do: the run passes before any pointer is looked at.
static int check_host_run(glabc_ctx* ctx, const glabc_run_t* run)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_model) return fail(ctx, GLABC_ERR_INVALID, "no model bound: call glabc_model_set first");
    if (!run) return fail(ctx, GLABC_ERR_INVALID, "null run description");
    if (run->rng_mode != GLABC_RNG_NATIVE) return fail(ctx, GLABC_ERR_INVALID, "host entry points run the native RNG only");
    if (int st = check_prior_run(ctx, "a host entry point", run, false)) return st;
    // GLABC_TRACE_EVENTS is a device-buffer layout (glabc.h): the scratch is sized for dense rows, an event writer would run
    // past it.  The event TRANSPORT of the host entries is chosen internally (run_global_host_hybrid), never by the caller.
    if (run->trace_layout != GLABC_TRACE_NONE && run->trace_layout != GLABC_TRACE_TIME_MAJOR &&
        run->trace_layout != GLABC_TRACE_CHAIN_MAJOR)
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "host entry points deliver GLABC_TRACE_NONE / TIME_MAJOR / CHAIN_MAJOR traces "
                                                "(trace_layout %d is a device-buffer layout)", run->trace_layout);
    if (run->n_chains <= 0 || run->n_steps < 0) return run->n_chains == 0 ? GLABC_OK : fail(ctx, GLABC_ERR_INVALID, "bad sizes");
    if (!run->theta || !run->y) return fail(ctx, GLABC_ERR_INVALID, "theta / y state pointers are required");
    if (run->trace_layout == GLABC_TRACE_NONE) return GLABC_OK;
    if (!run->trace) return fail(ctx, GLABC_ERR_INVALID, "trace pointer required for this trace_layout");
    const int64_t lo = run->step_base + (run->write_row0 ? 0 : 1) - run->trace_row_base;   // first and last host row written
    const int64_t hi = run->step_base + run->n_steps - run->trace_row_base;
    if (lo <= hi && (lo < 0 || hi >= run->trace_rows)) return fail(ctx, GLABC_ERR_INVALID, "trace rows fall outside the host buffer");
    if (run->trace_chain_off < 0 || run->trace_chain_off + run->n_chains > run->trace_chains)
        return fail(ctx, GLABC_ERR_INVALID, "chains fall outside the host trace buffer");
    return GLABC_OK;
}

// The per-chain state of a host-buffer run: theta [C][d], y [C][y_dim], aux [C][GLABC_AUX_SLOTS], stats [C][ns] and
// state64 [C][GLABC_STATE64_SLOTS].  aux, stats and state64 are null when the run carries none.
struct ChainState {
    float *theta, *y, *aux, *stats;
    double* state64;
};

static ChainState host_state(const glabc_run_t* run) { return {run->theta, run->y, run->aux, run->stats, run->state64}; }

// the state from chain c0 on
static ChainState chains_at(const glabc_ctx* ctx, const ChainState& s, int64_t c0)
{
    const int d = ctx->model.theta_dim;
    auto at = [c0](auto* p, int64_t width) { return p ? p + c0 * width : p; };
    return {at(s.theta, d), at(s.y, ctx->model.y_dim), at(s.aux, GLABC_AUX_SLOTS), at(s.stats, GLABC_NSTATS(d)),
            at(s.state64, GLABC_STATE64_SLOTS)};
}

// floats of the device state of n chains of the run (state64 apart)
static size_t state_floats(const glabc_ctx* ctx, const glabc_run_t* run, int64_t n)
{
    const int d = ctx->model.theta_dim;
    return size_t(n) * (d + ctx->model.y_dim + (run->aux ? GLABC_AUX_SLOTS : 0) + (run->stats ? GLABC_NSTATS(d) : 0));
}

// the state of n chains of the run laid out in `f` as theta | y | aux | stats, and state64 in `f64`
static ChainState carve_state(const glabc_ctx* ctx, const glabc_run_t* run, int64_t n, float* f, double* f64)
{
    ChainState s{};
    s.theta = f;
    s.y = s.theta + n * ctx->model.theta_dim;
    float* next = s.y + n * ctx->model.y_dim;
    if (run->aux) {
        s.aux = next;
        next += n * GLABC_AUX_SLOTS;
    }
    if (run->stats) s.stats = next;
    if (run->state64) s.state64 = f64;
    return s;
}

// Copies the state of chains [c0, c0 + n) between the run's host buffers and their device copy `dev` on stream s, in the
// direction `dir` (cudaMemcpyHostToDevice or cudaMemcpyDeviceToHost): the arrays `dev` has.  Returns the first error.
static cudaError_t stage_state(const glabc_ctx* ctx, const glabc_run_t* run, int64_t c0, int64_t n, const ChainState& dev,
                               cudaMemcpyKind dir, cudaStream_t s)
{
    const int d = ctx->model.theta_dim;
    const ChainState host = chains_at(ctx, host_state(run), c0);
    cudaError_t e = cudaSuccess;
    auto copy = [&](void* hp, void* dp, size_t chain_bytes) {
        if (!dp || e != cudaSuccess) return;
        const size_t bytes = size_t(n) * chain_bytes;
        e = dir == cudaMemcpyHostToDevice ? cudaMemcpyAsync(dp, hp, bytes, dir, s) : cudaMemcpyAsync(hp, dp, bytes, dir, s);
    };
    copy(host.theta, dev.theta, d * sizeof(float));
    copy(host.y, dev.y, ctx->model.y_dim * sizeof(float));
    copy(host.aux, dev.aux, GLABC_AUX_SLOTS * sizeof(float));
    copy(host.stats, dev.stats, GLABC_NSTATS(d) * sizeof(float));
    copy(host.state64, dev.state64, GLABC_STATE64_SLOTS * sizeof(double));
    return e;
}

// The run of chains [c0, c0 + n) of a host run, `s` being their state, on stream `stream`; every dump, tape and debug pointer
// is null.  For a launch the caller points the trace at its device buffer.
static glabc_run_t chain_slice(const glabc_run_t* run, int64_t c0, int64_t n, const ChainState& s, cudaStream_t stream)
{
    glabc_run_t r = *run;
    r.n_chains = n;
    r.chain_id_base = run->chain_id_base + c0;
    r.theta = s.theta;
    r.y = s.y;
    r.aux = s.aux;
    r.stats = s.stats;
    r.state64 = s.state64;
    r.stream = stream;
    r.tape32 = r.tape_grad0 = nullptr;
    r.tape64 = nullptr;
    r.debug = r.tape_dump = r.tape_grad0_dump = nullptr;
    r.debug64 = r.tape64_dump = nullptr;
    return r;
}

// streams and events of the dense transports, the device state of n chains of the run and two trace buffers
static int ensure_host_scratch(glabc_ctx* ctx, const glabc_run_t* run, int64_t n, size_t trace_floats, ChainState* dev)
{
    if (!ctx->s_compute) {
        CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_compute, cudaStreamNonBlocking));
        CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_done[b], cudaEventDisableTiming));
            CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_free[b], cudaEventDisableTiming));
        }
    }
    CUDA_TRY(ctx, ctx->d_state.reserve(state_floats(ctx, run, n)));
    CUDA_TRY(ctx, ctx->d_state64.reserve(run->state64 ? size_t(n) * GLABC_STATE64_SLOTS : 0));
    for (auto& t : ctx->d_trace) CUDA_TRY(ctx, t.reserve(trace_floats));
    *dev = carve_state(ctx, run, n, ctx->d_state.p, ctx->d_state64.p);
    return GLABC_OK;
}

// Time-chunk transport: H2D state, kernels in time chunks, D2H of each chunk's trace rows on a second stream overlapped with
// the next chunk's kernel, D2H state + stats.
static int run_host(glabc_ctx* ctx, SamplerKind kind, const glabc_run_t* run, int64_t chunk_steps, const glabc_aglmcmc_t* ag = nullptr)
{
    const int d = ctx->model.theta_dim;
    const int64_t C = run->n_chains;
    const bool traced = run->trace_layout != GLABC_TRACE_NONE;

    int64_t chunk = chunk_steps > 0 ? chunk_steps : (int64_t(64) << 20) / (C * d * int64_t(sizeof(float)));
    chunk = ((chunk + 31) / 32) * 32;
    if (chunk < 32) chunk = 32;
    if (chunk > run->n_steps) chunk = run->n_steps > 0 ? run->n_steps : 1;
    const int64_t buf_rows = chunk + 1;  // +1: the first chunk may carry row 0

    ChainState state;
    int st = ensure_host_scratch(ctx, run, C, traced ? size_t(buf_rows) * C * d : 0, &state);
    if (st) return st;
    cudaStream_t sc = ctx->s_compute, sx = ctx->s_copy;
    CUDA_TRY(ctx, stage_state(ctx, run, 0, C, state, cudaMemcpyHostToDevice, sc));

    int64_t done = 0;
    int b = 0;
    bool used[2] = {false, false};
    bool first_chunk = true;
    do {
        const int64_t n = std::min<int64_t>(chunk, run->n_steps - done);
        glabc_run_t dev = chain_slice(run, 0, C, state, sc);
        dev.n_steps = n;
        dev.step_base = run->step_base + done;
        dev.write_row0 = first_chunk && run->write_row0;
        const int64_t row_lo = dev.step_base + (dev.write_row0 ? 0 : 1);  // first absolute row this chunk writes
        const int64_t n_rows = n + (dev.write_row0 ? 1 : 0);
        if (traced) {
            if (used[b]) CUDA_TRY(ctx, cudaStreamWaitEvent(sc, ctx->ev_free[b], 0));
            dev.trace = ctx->d_trace[b].p;
            dev.trace_rows = buf_rows;
            dev.trace_chains = C;
            dev.trace_chain_off = 0;
            dev.trace_row_base = row_lo;
        }
        if (kind == SAMPLER_AGLMCMC) {   // the first chunk starts the run (initial block), the others continue from the workspace
            glabc_aglmcmc_t a = *ag;
            a.init = first_chunk ? ag->init : 0;
            a.init_p = a.init_s = a.ad_noise = a.ad_sim = nullptr;
            a.ad_idx = nullptr;
            a.ad_rec = a.ad_blk = a.init_w = nullptr;
            a.tape_rounds = a.dump_rounds = 0;
            st = glabc_run_aglmcmc(ctx, &dev, &a);
        } else {
            st = run_device(ctx, kind, &dev);
        }
        if (st) return st;
        if (traced && n_rows > 0) {
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_done[b], sc));
            CUDA_TRY(ctx, cudaStreamWaitEvent(sx, ctx->ev_done[b], 0));
            const int64_t host_row = row_lo - run->trace_row_base;
            if (run->trace_layout == GLABC_TRACE_TIME_MAJOR) {
                float* dst = run->trace + (host_row * run->trace_chains + run->trace_chain_off) * d;
                CUDA_TRY(ctx, cudaMemcpy2DAsync(dst, size_t(run->trace_chains) * d * sizeof(float), ctx->d_trace[b].p,
                                                size_t(C) * d * sizeof(float), size_t(C) * d * sizeof(float), size_t(n_rows),
                                                cudaMemcpyDeviceToHost, sx));
            } else {
                float* dst = run->trace + (run->trace_chain_off * run->trace_rows + host_row) * d;
                CUDA_TRY(ctx, cudaMemcpy2DAsync(dst, size_t(run->trace_rows) * d * sizeof(float), ctx->d_trace[b].p,
                                                size_t(buf_rows) * d * sizeof(float), size_t(n_rows) * d * sizeof(float), size_t(C),
                                                cudaMemcpyDeviceToHost, sx));
            }
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_free[b], sx));
            used[b] = true;
            b ^= 1;
        }
        done += n;
        first_chunk = false;
    } while (done < run->n_steps);

    CUDA_TRY(ctx, stage_state(ctx, run, 0, C, state, cudaMemcpyDeviceToHost, sc));
    CUDA_TRY(ctx, cudaStreamSynchronize(sc));
    CUDA_TRY(ctx, cudaStreamSynchronize(sx));
    return GLABC_OK;
}


// ---------------------------------------------------------------------------------------------
// AGLMCMC: workspace + entry point
// ---------------------------------------------------------------------------------------------
static int ensure_ag_workspace(glabc_ctx* ctx, int64_t C, int32_t B, int d, bool keep)
{
    if (keep) {
        if (!ctx->ag_mem || ctx->ag.C != C || ctx->ag.B != B || ctx->ag_dim != d)
            return fail(ctx, GLABC_ERR_INVALID, "glabc_run_aglmcmc: init = 0 but the context holds no workspace for %lld chains x block %d "
                                                "(start the run with init = 1)", (long long)C, B);
        return GLABC_OK;
    }
    const size_t cb = size_t(C) * size_t(B);
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~size_t(255); return o; };
    const size_t o_bt = take(cb * d * 4), o_bx = take(cb * d * 4), o_bw = take(cb * 4), o_bl = take(cb * 4), o_bd = take(cb * 4);
    const size_t o_kx = take(cb * d * 4), o_kw = take(cb * 4), o_kn = take(cb * 4), o_kl = take(cb * 4), o_kb = take(size_t(C) * d * 4);
    const size_t o_smp = take(cb * 4 * d * 4), o_cdf = take(cb * 8);
    const size_t o_i0 = take(size_t(C) * 4), o_i1 = take(size_t(C) * 4), o_i2 = take(size_t(C) * 4), o_i3 = take(size_t(C) * 4),
                 o_i4 = take(size_t(C) * 4), o_i5 = take(size_t(C) * 4), o_f0 = take(size_t(C) * 4), o_f1 = take(size_t(C) * 4);
    if (off > ctx->ag_bytes) {
        if (ctx->ag_mem) cudaFree(ctx->ag_mem);
        ctx->ag_mem = nullptr;
        ctx->ag_bytes = 0;
        CUDA_TRY(ctx, cudaMalloc(&ctx->ag_mem, off));
        ctx->ag_bytes = off;
    }
    ctx->ag_used = off;
    char* m = static_cast<char*>(ctx->ag_mem);
    AgWorkspace& W = ctx->ag;
    W.blk_theta = reinterpret_cast<float*>(m + o_bt); W.blk_x = reinterpret_cast<float*>(m + o_bx);
    W.blk_w = reinterpret_cast<float*>(m + o_bw); W.blk_lq = reinterpret_cast<float*>(m + o_bl);
    W.blk_dis = reinterpret_cast<float*>(m + o_bd);
    W.kde_X = reinterpret_cast<float*>(m + o_kx); W.kde_w = reinterpret_cast<float*>(m + o_kw);
    W.kde_wn = reinterpret_cast<float*>(m + o_kn); W.kde_lw = reinterpret_cast<float*>(m + o_kl);
    W.kde_bw = reinterpret_cast<float*>(m + o_kb); W.smp = reinterpret_cast<float*>(m + o_smp);
    W.cdf = reinterpret_cast<double*>(m + o_cdf);
    W.kde_n = reinterpret_cast<int32_t*>(m + o_i0); W.kk = reinterpret_cast<int32_t*>(m + o_i1);
    W.n_adapt = reinterpret_cast<int32_t*>(m + o_i2); W.pending = reinterpret_cast<int32_t*>(m + o_i3);
    W.lq_valid = reinterpret_cast<int32_t*>(m + o_i4); W.next_step = reinterpret_cast<uint32_t*>(m + o_i5);
    W.hat_eps = reinterpret_cast<float*>(m + o_f0); W.lq_cur = reinterpret_cast<float*>(m + o_f1);
    W.C = C;
    W.B = B;
    ctx->ag_dim = d;
    return GLABC_OK;
}

extern "C" int glabc_run_aglmcmc(glabc_ctx* ctx, const glabc_run_t* run, const glabc_aglmcmc_t* ag)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_model) return fail(ctx, GLABC_ERR_INVALID, "no model bound: call glabc_model_set first");
    if (!run || !ag) return fail(ctx, GLABC_ERR_INVALID, "null run / aglmcmc description");
    if (!ctx->has_dist[GLABC_SLOT_LOCAL] || !ctx->has_dist[GLABC_SLOT_IMPORTANCE])
        return fail(ctx, GLABC_ERR_INVALID, "run_aglmcmc needs the LOCAL and IMPORTANCE (Initial_ISIR_prop) proposal slots bound");
    const int d = ctx->model.theta_dim;
    const glabc_dist_t& lp = ctx->dist[GLABC_SLOT_LOCAL];
    const glabc_dist_t& ip = ctx->dist[GLABC_SLOT_IMPORTANCE];
    if (lp.dim != d || ip.dim != d) return fail(ctx, GLABC_ERR_INVALID, "proposal dim does not match theta_dim %d", d);
    if (!all_gaussian(ctx, {GLABC_SLOT_LOCAL}))
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "run_aglmcmc is fused for a DiagGaussian Local_Proposal");
    const bool gip = !all_gaussian(ctx, {GLABC_SLOT_IMPORTANCE});
    if (gip && (run->arith_mode == GLABC_ARITH_STRICT || run->rng_mode == GLABC_RNG_REPLAY || ag->ad_rec || ag->ad_blk || ag->init_w))
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "run_aglmcmc with a non-Gaussian Initial_ISIR_prop runs FAST arithmetic with the native RNG "
                                                "(the STRICT / replay / recording kernels are fused for a DiagGaussian Initial_ISIR_prop)");
    if (run->n_candidates < 1 || run->n_candidates > GLABC_MAX_K)
        return fail(ctx, GLABC_ERR_INVALID, "n_candidates (batch_size) must be in 1..%d", GLABC_MAX_K);
    if (ag->step_size < 1 || int64_t(ag->step_size) * run->n_candidates > GLABC_AG_MAX_BLOCK)
        return fail(ctx, GLABC_ERR_INVALID, "batch_size * step_size must be in 1..%d", GLABC_AG_MAX_BLOCK);
    if (ag->kde_rule != GLABC_BW_SILVERMAN && ag->kde_rule != GLABC_BW_SCOTT) return fail(ctx, GLABC_ERR_INVALID, "bad kde_rule");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    RunParams R;
    int block = 0;
    int st = make_run_params(ctx, run, d, GLABC_TAPE_GLOBAL_SLOTS(d, d), &R, &block);
    if (st || (st = check_prior_run(ctx, "run_aglmcmc", run, ag->ad_rec || ag->ad_blk || ag->init_w))) return st;
    if (run->block_threads == 0) block = 128;
    if (block > 128) return fail(ctx, GLABC_ERR_INVALID, "run_aglmcmc: block_threads at most 128");
    const bool replay = run->rng_mode == GLABC_RNG_REPLAY;
    if (replay && (!run->tape64 || !ag->ad_idx || !ag->ad_noise || !ag->ad_sim || ag->tape_rounds < 1 ||
                   (ag->init && (!ag->init_p || !ag->init_s))))
        return fail(ctx, GLABC_ERR_INVALID, "replay of run_aglmcmc needs tape64, init_p/init_s and the adaptation tapes");
    if (R.n_chains == 0) return GLABC_OK;
    const int32_t B = ag->step_size * run->n_candidates;
    st = ensure_ag_workspace(ctx, R.n_chains, B, d, !ag->init);
    if (st) return st;
    AgConsts K{};
    K.model = make_model(ctx->model);
    K.lp = make_gauss(lp.a, lp.b, lp.c, d);
    if (gip) {
        K.ip_generic = 1;
        K.ipg = make_dist(ip);
    } else {
        K.ip = make_gauss(ip.a, ip.b, ip.c, d);
    }
    K.S = ag->step_size;
    K.alpha = ag->alpha;
    K.hat_eps_T = ag->hat_eps_T;
    K.log_prior_floor = static_cast<float>(std::log(1e-10));
    AgTapes T{ag->init_p, ag->init_s, ag->ad_noise, ag->ad_sim, ag->ad_idx, ag->ad_rec, ag->ad_blk, ag->init_w, ag->tape_rounds,
              ag->dump_rounds};
    CUDA_TRY(ctx, launch_aglmcmc(K, make_prior(ctx), ctx->ag, T, R, d, ag->init, ag->kde_rule, run->arith_mode == GLABC_ARITH_STRICT, replay,
                                 run->trace_layout, block, static_cast<cudaStream_t>(run->stream)));
    return GLABC_OK;
}

/* the workspace of glabc_run_aglmcmc (every chain's candidate block, per-chain KDE, counters, eps-hat) as an opaque blob */
extern "C" int glabc_aglmcmc_state(glabc_ctx* ctx, void* blob, int64_t* bytes, int64_t n_chains, int32_t block, int32_t restore, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_model) return fail(ctx, GLABC_ERR_INVALID, "no model bound: call glabc_model_set first");
    if (!bytes) return fail(ctx, GLABC_ERR_INVALID, "glabc_aglmcmc_state: null size pointer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int d = ctx->model.theta_dim;
    if (!restore) {
        if (!ctx->ag_mem || ctx->ag_used == 0) return fail(ctx, GLABC_ERR_INVALID, "glabc_aglmcmc_state: the context holds no AGLMCMC workspace");
        if (!blob) { *bytes = static_cast<int64_t>(ctx->ag_used); return GLABC_OK; }     // size query
        if (*bytes < static_cast<int64_t>(ctx->ag_used)) return fail(ctx, GLABC_ERR_INVALID, "glabc_aglmcmc_state: blob too small");
        CUDA_TRY(ctx, cudaMemcpyAsync(blob, ctx->ag_mem, ctx->ag_used, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
        *bytes = static_cast<int64_t>(ctx->ag_used);
        return GLABC_OK;
    }
    if (!blob || n_chains < 1 || block < 1 || block > GLABC_AG_MAX_BLOCK) return fail(ctx, GLABC_ERR_INVALID, "glabc_aglmcmc_state: bad blob / sizes");
    int st = ensure_ag_workspace(ctx, n_chains, block, d, false);
    if (st) return st;
    if (*bytes != static_cast<int64_t>(ctx->ag_used))
        return fail(ctx, GLABC_ERR_INVALID, "glabc_aglmcmc_state: blob of %lld bytes, a workspace of %lld chains x block %d takes %zu",
                    (long long)*bytes, (long long)n_chains, block, ctx->ag_used);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ag_mem, blob, ctx->ag_used, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

// ---------------------------------------------------------------------------------------------
// KernelDensity entry points
// ---------------------------------------------------------------------------------------------
static int check_kde(glabc_ctx* ctx, const char* who, const void* X, int64_t sets, int64_t cap, int32_t dim)
{
    if (!X) return fail(ctx, GLABC_ERR_INVALID, "%s: null X", who);
    if (sets < 0 || cap < 1 || cap > INT32_MAX) return fail(ctx, GLABC_ERR_INVALID, "%s: bad sets / cap", who);
    if (dim < 1 || dim > 4) return fail(ctx, GLABC_ERR_UNSUPPORTED, "%s: dim %d outside 1..4", who, dim);
    return GLABC_OK;
}

extern "C" int glabc_kde_fit(glabc_ctx* ctx, const float* X, const float* w, const int32_t* n, int64_t sets, int64_t cap,
                             int32_t dim, int32_t rule, float* weights_out, float* bw_out, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    int st = check_kde(ctx, "glabc_kde_fit", X, sets, cap, dim);
    if (st) return st;
    if (!weights_out || !bw_out) return fail(ctx, GLABC_ERR_INVALID, "glabc_kde_fit: null output");
    if (rule != GLABC_BW_SILVERMAN && rule != GLABC_BW_SCOTT) return fail(ctx, GLABC_ERR_INVALID, "glabc_kde_fit: bad rule %d", rule);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, launch_kde_fit(X, w, n, nullptr, sets, cap, dim, rule, weights_out, nullptr, bw_out, static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

extern "C" int glabc_kde_log_prob(glabc_ctx* ctx, const float* X, const float* weights, const float* bw, const int32_t* n,
                                  int64_t sets, int64_t cap, int32_t dim, const float* x, int64_t m, float* out, int32_t arith,
                                  void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    int st = check_kde(ctx, "glabc_kde_log_prob", X, sets, cap, dim);
    if (st) return st;
    if (!weights || !bw || !x || !out || m < 0) return fail(ctx, GLABC_ERR_INVALID, "glabc_kde_log_prob: null pointer / bad m");
    if (arith != GLABC_ARITH_FAST && arith != GLABC_ARITH_STRICT) return fail(ctx, GLABC_ERR_INVALID, "bad arith_mode %d", arith);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    KdeSets S{X, weights, bw, n, nullptr, sets, cap};
    const int ksplit = arith == GLABC_ARITH_STRICT ? 1 : kde_logprob_split(sets, m, cap);
    if (ksplit > 1) CUDA_TRY(ctx, ctx->kde_part.reserve(size_t(ksplit) * size_t(sets) * size_t(m)));
    // (a non-null scratch pointer tells the launcher the point split is available, even when this call needs ksplit = 1)
    CUDA_TRY(ctx, launch_kde_logprob(S, nullptr, dim, x, m, out, arith == GLABC_ARITH_STRICT, static_cast<cudaStream_t>(stream), ksplit,
                                     ksplit > 1 ? ctx->kde_part.p : reinterpret_cast<float*>(out)));
    return GLABC_OK;
}

extern "C" int glabc_kde_sample(glabc_ctx* ctx, const float* X, const float* weights, const float* bw, const int32_t* n,
                                int64_t sets, int64_t cap, int32_t dim, int64_t m, uint64_t seed, const int32_t* idx_tape,
                                const float* noise_tape, float* out, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    int st = check_kde(ctx, "glabc_kde_sample", X, sets, cap, dim);
    if (st) return st;
    if (!weights || !bw || !out || m < 0) return fail(ctx, GLABC_ERR_INVALID, "glabc_kde_sample: null pointer / bad m");
    if ((idx_tape == nullptr) != (noise_tape == nullptr))
        return fail(ctx, GLABC_ERR_INVALID, "glabc_kde_sample: idx_tape and noise_tape go together");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t cs = static_cast<cudaStream_t>(stream);
    KdeSets S{X, weights, bw, n, nullptr, sets, cap};
    if (!idx_tape) {
        CUDA_TRY(ctx, ctx->kde_cdf.reserve(size_t(sets) * size_t(cap)));
        CUDA_TRY(ctx, launch_kde_cdf(weights, n, nullptr, sets, cap, ctx->kde_cdf.p, cs));
    }
    const RoundKeys rk = expand_key(make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
    CUDA_TRY(ctx, launch_kde_sample(S, dim, ctx->kde_cdf.p, m, rk, 0, nullptr, idx_tape, noise_tape, m, m * dim, 1, 0, 0, 0, out, cs));
    return GLABC_OK;
}


// ---------------------------------------------------------------------------------------------
// RealNVP flow (GLMCMC-NFs importance proposal)
// ---------------------------------------------------------------------------------------------
extern "C" int glabc_flow_set(glabc_ctx* ctx, const glabc_flow_t* f, size_t nbytes, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!f || nbytes != sizeof(glabc_flow_t))
        return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_set: struct size %zu, expected %zu (ABI mismatch)", nbytes, sizeof(glabc_flow_t));
    if (f->hidden != kFlowHidden || f->dim != 2)
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "the fused flow is MLP([1,128,128,2]) couplings on a 2-d theta (GLMCMC_NFs.py:56)");
    if (f->n_blocks < 1 || f->n_blocks > 1024) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_set: n_blocks out of range");
    if (!f->w1 || !f->b1 || !f->w2 || !f->b2 || !f->w3 || !f->b3) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_set: null weights");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t cs = static_cast<cudaStream_t>(stream);
    const size_t L = size_t(f->n_blocks), H = kFlowHidden;
    const FlowParamLayout P(f->n_blocks);
    // [packed W2: FP16 hi then FP16 lo, L*H*H floats in all][per-block operand blobs of the pipelined kernel][the flat FP32
    // parameter vector, FlowParamLayout]
    const size_t need = L * H * H + L * (kFlowAuxBytes / 4) + size_t(P.total);
    if (need > ctx->flow_floats) {
        if (ctx->flow_mem) cudaFree(ctx->flow_mem);
        ctx->flow_mem = nullptr;
        ctx->flow_floats = 0;
        CUDA_TRY(ctx, cudaMalloc(&ctx->flow_mem, need * sizeof(float)));
        ctx->flow_floats = need;
    }
    if (ctx->flow_blocks != f->n_blocks) ctx->tr_ready = false;   // moments of another architecture
    ctx->flow_blocks = f->n_blocks;
    float* w2p = ctx->flow_mem;                   // first: 16-byte (in fact 256-byte) aligned for cp.async.bulk
    float* w2p_lo = w2p + L * H * H / 2;          // the FP16 remainder W2 - FP16(W2) (PRECISE mode, training)
    uint8_t* aux = reinterpret_cast<uint8_t*>(ctx->flow_mem + L * H * H);
    float* par = ctx->flow_mem + L * H * H + L * (kFlowAuxBytes / 4);
    CUDA_TRY(ctx, cudaMemcpyAsync(par + P.w1, f->w1, L * H * 4, cudaMemcpyDeviceToDevice, cs));
    CUDA_TRY(ctx, cudaMemcpyAsync(par + P.b1, f->b1, L * H * 4, cudaMemcpyDeviceToDevice, cs));
    CUDA_TRY(ctx, cudaMemcpyAsync(par + P.w2, f->w2, L * H * H * 4, cudaMemcpyDeviceToDevice, cs));
    CUDA_TRY(ctx, cudaMemcpyAsync(par + P.b2, f->b2, L * H * 4, cudaMemcpyDeviceToDevice, cs));
    CUDA_TRY(ctx, cudaMemcpyAsync(par + P.w3, f->w3, L * 2 * H * 4, cudaMemcpyDeviceToDevice, cs));
    CUDA_TRY(ctx, cudaMemcpyAsync(par + P.b3, f->b3, L * 2 * 4, cudaMemcpyDeviceToDevice, cs));
    const float base[4] = {f->base_loc[0], f->base_loc[1], f->base_log_scale[0], f->base_log_scale[1]};
    CUDA_TRY(ctx, cudaMemcpyAsync(par + P.loc, base, sizeof(base), cudaMemcpyHostToDevice, cs));
    CUDA_TRY(ctx, cudaStreamSynchronize(cs));     // `base` is a stack array
    CUDA_TRY(ctx, launch_flow_pack(par + P.w2, w2p, w2p_lo, f->n_blocks, cs));
    CUDA_TRY(ctx, launch_flow_pack_aux(par + P.w1, par + P.b1, par + P.b2, par + P.w3, par + P.b3, aux, f->n_blocks, cs));
    FlowDev d{};
    d.aux = aux;
    d.w1 = par + P.w1; d.b1 = par + P.b1; d.w2p = w2p; d.w2p_lo = w2p_lo; d.b2 = par + P.b2; d.w3 = par + P.w3; d.b3 = par + P.b3;
    for (int i = 0; i < 2; ++i) {
        d.base_loc[i] = f->base_loc[i];
        d.base_log_scale[i] = f->base_log_scale[i];
    }
    d.n_blocks = f->n_blocks;
    ctx->flow = d;
    ctx->has_flow = true;
    return GLABC_OK;
}

static int run_flow(glabc_ctx* ctx, bool sample, const float* in, int64_t n, float* theta, float* log_q, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_flow) return fail(ctx, GLABC_ERR_INVALID, "no flow bound: call glabc_flow_set first");
    if (ctx->cc < 100) return fail(ctx, GLABC_ERR_UNSUPPORTED, "the flow kernels need tcgen05 tensor cores (sm_100a); this device is sm_%d", ctx->cc);
    if (!in || !log_q || (sample && !theta) || n < 0) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_%s: null pointer / bad n", sample ? "sample" : "log_prob");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, launch_flow(ctx->flow, sample, ctx->flow_precision == GLABC_FLOW_PRECISE, in, n, theta, log_q, ctx->sm_count,
                              static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

extern "C" int glabc_flow_precision(glabc_ctx* ctx, int32_t mode)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (mode != GLABC_FLOW_FAST && mode != GLABC_FLOW_PRECISE) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_precision: bad mode %d", mode);
    ctx->flow_precision = mode;
    return GLABC_OK;
}

// ---- training step (GLMCMC_NFs.py:63,112-124) ----
static float* flow_params(glabc_ctx* ctx)
{
    return ctx->flow_mem + size_t(ctx->flow_blocks) * kFlowHidden * kFlowHidden + size_t(ctx->flow_blocks) * (kFlowAuxBytes / 4);
}

extern "C" int64_t glabc_flow_param_count(int32_t n_blocks) { return n_blocks < 1 ? 0 : FlowParamLayout(n_blocks).total; }

extern "C" int glabc_flow_train_init(glabc_ctx* ctx, float lr, float beta1, float beta2, float eps, float weight_decay)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_flow) return fail(ctx, GLABC_ERR_INVALID, "no flow bound: call glabc_flow_set first");
    if (!(lr > 0.0f) || !(beta1 >= 0.0f && beta1 < 1.0f) || !(beta2 >= 0.0f && beta2 < 1.0f) || !(eps > 0.0f) || !(weight_decay >= 0.0f))
        return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_train_init: bad Adam hyper-parameters");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int64_t total = FlowParamLayout(ctx->flow_blocks).total;
    if (ctx->tr_mem) cudaFree(ctx->tr_mem);
    if (ctx->tr_partial) cudaFree(ctx->tr_partial);
    ctx->tr_mem = ctx->tr_partial = nullptr;
    ctx->tr_ready = false;
    CUDA_TRY(ctx, cudaMalloc(&ctx->tr_mem, (3 * size_t(total) + 4) * sizeof(float)));
    CUDA_TRY(ctx, cudaMemset(ctx->tr_mem, 0, (3 * size_t(total) + 4) * sizeof(float)));
    ctx->tr_slices = ctx->sm_count > 0 ? ctx->sm_count : 1;
    CUDA_TRY(ctx, cudaMalloc(&ctx->tr_partial, size_t(ctx->tr_slices) * size_t((total + 3) & ~int64_t(3)) * sizeof(float)));
    ctx->tr_lr = lr; ctx->tr_beta1 = beta1; ctx->tr_beta2 = beta2; ctx->tr_eps = eps; ctx->tr_wd = weight_decay;
    ctx->tr_step = 0;
    ctx->tr_ready = true;
    return GLABC_OK;
}

extern "C" int glabc_flow_grad(glabc_ctx* ctx, const float* x, int64_t n, float* grad, float* loss, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_flow || !ctx->tr_ready) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_grad: call glabc_flow_set and glabc_flow_train_init first");
    if (ctx->cc < 100) return fail(ctx, GLABC_ERR_UNSUPPORTED, "the flow kernels need tcgen05 tensor cores (sm_100a); this device is sm_%d", ctx->cc);
    if (!x || n < 1) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_grad: null samples / n < 1");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t cs = static_cast<cudaStream_t>(stream);
    const int64_t total = FlowParamLayout(ctx->flow_blocks).total;
    CUDA_TRY(ctx, ctx->tr_fwd.reserve(size_t(n) * 3));
    float* z = ctx->tr_fwd.p;
    float* lq = ctx->tr_fwd.p + 2 * n;
    float* g = grad ? grad : ctx->tr_mem + 2 * total;
    float* ls = loss ? loss : ctx->tr_mem + 3 * total;
    // forward: log q(x) and the latent z = f^-1(x), split-precision mode whatever the inference mode is
    CUDA_TRY(ctx, launch_flow(ctx->flow, false, true, x, n, z, lq, ctx->sm_count, cs));
    CUDA_TRY(ctx, launch_flow_loss(lq, n, ls, cs));
    const int64_t chunks = (n + flow_train_chunk_samples() - 1) / flow_train_chunk_samples();
    const int slices = static_cast<int>(chunks < ctx->tr_slices ? chunks : ctx->tr_slices);
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->tr_partial, 0, size_t(slices) * size_t((total + 3) & ~int64_t(3)) * sizeof(float), cs));
    CUDA_TRY(ctx, launch_flow_bwd(ctx->flow, z, n, ctx->tr_partial, slices, cs));
    CUDA_TRY(ctx, launch_flow_grad_reduce(ctx->tr_partial, slices, total, n, g, cs));
    return GLABC_OK;
}

extern "C" int glabc_flow_adam_step(glabc_ctx* ctx, const float* grad, const float* loss, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_flow || !ctx->tr_ready) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_adam_step: call glabc_flow_set and glabc_flow_train_init first");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t cs = static_cast<cudaStream_t>(stream);
    const FlowParamLayout P(ctx->flow_blocks);
    const float* g = grad ? grad : ctx->tr_mem + 2 * P.total;
    const float* ls = loss ? loss : ctx->tr_mem + 3 * P.total;
    float host_loss = 0.0f;
    CUDA_TRY(ctx, cudaMemcpyAsync(&host_loss, ls, sizeof(float), cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(ctx, cudaStreamSynchronize(cs));
    if (!std::isfinite(host_loss)) return GLABC_OK;   // GLMCMC_NFs.py:120-121: no backward, and Adam leaves gradient-less parameters alone
    ctx->tr_step += 1;
    float* par = flow_params(ctx);
    CUDA_TRY(ctx, launch_flow_adam(par, ctx->tr_mem, ctx->tr_mem + P.total, g, P.total, ls, ctx->tr_lr, ctx->tr_beta1, ctx->tr_beta2,
                                   ctx->tr_eps, ctx->tr_wd, ctx->tr_step, cs));
    // the kernels read W2 packed and the base parameters from the launch descriptor: refresh both
    const size_t LHH = size_t(ctx->flow_blocks) * kFlowHidden * kFlowHidden;
    CUDA_TRY(ctx, launch_flow_pack(par + P.w2, ctx->flow_mem, ctx->flow_mem + LHH / 2, ctx->flow_blocks, cs));
    CUDA_TRY(ctx, launch_flow_pack_aux(par + P.w1, par + P.b1, par + P.b2, par + P.w3, par + P.b3,
                                       reinterpret_cast<uint8_t*>(ctx->flow_mem + LHH), ctx->flow_blocks, cs));
    float base[4];
    CUDA_TRY(ctx, cudaMemcpyAsync(base, par + P.loc, sizeof(base), cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(ctx, cudaStreamSynchronize(cs));
    ctx->flow.base_loc[0] = base[0]; ctx->flow.base_loc[1] = base[1];
    ctx->flow.base_log_scale[0] = base[2]; ctx->flow.base_log_scale[1] = base[3];
    return GLABC_OK;
}

extern "C" int glabc_flow_train_step(glabc_ctx* ctx, const float* x, int64_t n, float* loss, void* stream)
{
    int st = glabc_flow_grad(ctx, x, n, nullptr, loss, stream);
    if (st) return st;
    return glabc_flow_adam_step(ctx, nullptr, loss, stream);
}

extern "C" int glabc_flow_get(glabc_ctx* ctx, float* params, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_flow) return fail(ctx, GLABC_ERR_INVALID, "no flow bound");
    if (!params) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_get: null pointer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpyAsync(params, flow_params(ctx), size_t(FlowParamLayout(ctx->flow_blocks).total) * sizeof(float), cudaMemcpyDeviceToDevice,
                                  static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

/* Adam moments and step count, for checkpoints: state[2 * P] = m | v (device); *step in / out */
extern "C" int glabc_flow_train_state(glabc_ctx* ctx, float* state, int64_t* step, int32_t restore, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_flow || !ctx->tr_ready) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_train_state: no training state");
    if (!state || !step) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_train_state: null pointer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t bytes = 2 * size_t(FlowParamLayout(ctx->flow_blocks).total) * sizeof(float);
    if (restore) {
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->tr_mem, state, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
        ctx->tr_step = *step;
    } else {
        CUDA_TRY(ctx, cudaMemcpyAsync(state, ctx->tr_mem, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
        *step = ctx->tr_step;
    }
    return GLABC_OK;
}

extern "C" int glabc_flow_sample(glabc_ctx* ctx, const float* eps, int64_t n, float* theta, float* log_q, void* stream)
{
    if (ctx && !eps) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_sample: null eps (glabc_flow_sample_native draws them in the kernel)");
    return run_flow(ctx, true, eps, n, theta, log_q, stream);
}

extern "C" int glabc_flow_sample_native(glabc_ctx* ctx, uint64_t seed, int64_t n, float* theta, float* log_q, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!theta || !log_q || n < 0) return fail(ctx, GLABC_ERR_INVALID, "glabc_flow_sample_native: null pointer / bad n");
    if (!ctx->has_flow) return fail(ctx, GLABC_ERR_INVALID, "no flow bound: call glabc_flow_set first");
    if (ctx->cc < 100) return fail(ctx, GLABC_ERR_UNSUPPORTED, "the flow kernels need tcgen05 tensor cores (sm_100a); this device is sm_%d", ctx->cc);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    FlowDev W = ctx->flow;
    W.seed_lo = static_cast<uint32_t>(seed);
    W.seed_hi = static_cast<uint32_t>(seed >> 32);
    CUDA_TRY(ctx, launch_flow(W, true, ctx->flow_precision == GLABC_FLOW_PRECISE, nullptr, n, theta, log_q, ctx->sm_count,
                              static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

extern "C" int glabc_flow_log_prob(glabc_ctx* ctx, const float* theta, int64_t n, float* log_q, void* stream)
{
    return run_flow(ctx, false, theta, n, nullptr, log_q, stream);
}


// ---------------------------------------------------------------------------------------------
// block iSIR with an external importance proposal (GLMCMC-NFs)
// ---------------------------------------------------------------------------------------------
// the block description of glabc_run_block_isir / glabc_block_weights and their user-model twins
static int check_block(glabc_ctx* ctx, const char* who, const glabc_run_t* run, const glabc_block_isir_t* b)
{
    if (run->n_candidates < 1 || run->n_candidates > GLABC_MAX_K) return fail(ctx, GLABC_ERR_INVALID, "n_candidates must be in 1..%d", GLABC_MAX_K);
    if (b->step_size < 1 || int64_t(b->step_size) * run->n_candidates != b->block || b->block > GLABC_AG_MAX_BLOCK)
        return fail(ctx, GLABC_ERR_INVALID, "%s: block must equal batch_size * step_size and be at most %d", who, GLABC_AG_MAX_BLOCK);
    if (!b->blk_theta || !b->blk_x || !b->blk_w || !b->blk_lq || !b->kk || !b->pending || !b->next_step || !b->lq_cur || !b->lq_valid)
        return fail(ctx, GLABC_ERR_INVALID, "%s: null block / state buffer", who);
    return GLABC_OK;
}

static int block_isir_setup(glabc_ctx* ctx, const char* who, const glabc_run_t* run, const glabc_block_isir_t* b, bool need_local,
                            AgConsts* K, AgWorkspace* W, RunParams* R, int* block)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctx->has_model) return fail(ctx, GLABC_ERR_INVALID, "no model bound: call glabc_model_set first");
    if (!run || !b) return fail(ctx, GLABC_ERR_INVALID, "%s: null run / block description", who);
    if (need_local && !ctx->has_dist[GLABC_SLOT_LOCAL]) return fail(ctx, GLABC_ERR_INVALID, "%s needs the LOCAL proposal slot bound", who);
    const int d = ctx->model.theta_dim;
    if (int st = check_block(ctx, who, run, b)) return st;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    int st = make_run_params(ctx, run, d, GLABC_TAPE_GLOBAL_SLOTS(d, d), R, block);
    if (st) return st;
    if (run->rng_mode != GLABC_RNG_NATIVE) return fail(ctx, GLABC_ERR_UNSUPPORTED, "%s runs the native RNG only", who);
    if ((st = check_prior_run(ctx, who, run, false))) return st;
    if (run->block_threads == 0) *block = 128;
    if (*block > 128) return fail(ctx, GLABC_ERR_INVALID, "%s: block_threads at most 128", who);
    *K = AgConsts{};
    K->model = make_model(ctx->model);
    if (need_local) {
        const glabc_dist_t& lp = ctx->dist[GLABC_SLOT_LOCAL];
        if (lp.dim != d) return fail(ctx, GLABC_ERR_INVALID, "proposal dim does not match theta_dim %d", d);
        if (lp.kind != GLABC_DIST_DIAG_GAUSSIAN) return fail(ctx, GLABC_ERR_UNSUPPORTED, "%s is fused for a DiagGaussian Local_Proposal", who);
        K->lp = make_gauss(lp.a, lp.b, lp.c, d);
        K->ip = K->lp;  // unused: the importance proposal is external
    }
    K->S = b->step_size;
    *W = AgWorkspace{};
    W->blk_theta = b->blk_theta; W->blk_x = b->blk_x; W->blk_w = b->blk_w; W->blk_lq = b->blk_lq;
    W->kk = b->kk; W->pending = b->pending; W->next_step = b->next_step; W->lq_cur = b->lq_cur; W->lq_valid = b->lq_valid;
    W->C = R->n_chains;
    W->B = b->block;
    return GLABC_OK;
}

extern "C" int glabc_run_block_isir(glabc_ctx* ctx, const glabc_run_t* run, const glabc_block_isir_t* b)
{
    AgConsts K;
    AgWorkspace W;
    RunParams R;
    int block = 0;
    int st = block_isir_setup(ctx, "glabc_run_block_isir", run, b, true, &K, &W, &R, &block);
    if (st) return st;
    if (R.n_chains == 0) return GLABC_OK;
    CUDA_TRY(ctx, launch_block_isir(K, make_prior(ctx), W, R, ctx->model.theta_dim, run->arith_mode == GLABC_ARITH_STRICT, run->trace_layout, block,
                                    static_cast<cudaStream_t>(run->stream)));
    return GLABC_OK;
}

extern "C" int glabc_block_weights(glabc_ctx* ctx, const glabc_run_t* run, const glabc_block_isir_t* b, uint32_t round)
{
    AgConsts K;
    AgWorkspace W;
    RunParams R;
    int block = 0;
    int st = block_isir_setup(ctx, "glabc_block_weights", run, b, false, &K, &W, &R, &block);
    if (st) return st;
    if (R.n_chains == 0) return GLABC_OK;
    CUDA_TRY(ctx, launch_block_weights(K, make_prior(ctx), W, R, ctx->model.theta_dim, round, static_cast<cudaStream_t>(run->stream)));
    return GLABC_OK;
}


// ---------------------------------------------------------------------------------------------
// device-side forward() / log_prob() of a bound proposal distribution
// ---------------------------------------------------------------------------------------------
extern "C" int glabc_dist_log_prob(glabc_ctx* ctx, int slot, const float* z, int64_t n, float* log_p, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (slot < 0 || slot >= GLABC_SLOT_COUNT || !ctx->has_dist[slot]) return fail(ctx, GLABC_ERR_INVALID, "glabc_dist_log_prob: slot %d is not bound", slot);
    if (check_builtin_dim(ctx, "glabc_dist_log_prob", ctx->dist[slot])) return GLABC_ERR_UNSUPPORTED;
    if (!z || !log_p || n < 0) return fail(ctx, GLABC_ERR_INVALID, "glabc_dist_log_prob: null pointer / bad n");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const RoundKeys rk = expand_key(make_uint2(0u, 0u));
    CUDA_TRY(ctx, launch_dist_eval(make_dist(ctx->dist[slot]), ctx->dist[slot].dim, rk, n, z, nullptr, log_p, static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

extern "C" int glabc_dist_sample(glabc_ctx* ctx, int slot, int64_t n, uint64_t seed, float* z, float* log_p, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (slot < 0 || slot >= GLABC_SLOT_COUNT || !ctx->has_dist[slot]) return fail(ctx, GLABC_ERR_INVALID, "glabc_dist_sample: slot %d is not bound", slot);
    if (check_builtin_dim(ctx, "glabc_dist_sample", ctx->dist[slot])) return GLABC_ERR_UNSUPPORTED;
    if (!z || n < 0) return fail(ctx, GLABC_ERR_INVALID, "glabc_dist_sample: null pointer / bad n");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const RoundKeys rk = expand_key(make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
    CUDA_TRY(ctx, launch_dist_eval(make_dist(ctx->dist[slot]), ctx->dist[slot].dim, rk, n, nullptr, z, log_p, static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

// ---------------------------------------------------------------------------------------------
// GlobalMCMC with a user-supplied model compiled at run time (user_model.cu)
// ---------------------------------------------------------------------------------------------
static bool valid_dist_kind(int kind) { return kind >= GLABC_DIST_DIAG_GAUSSIAN && kind <= GLABC_DIST_GAUSSIAN_MIXTURE; }

extern "C" int glabc_user_model_check_proposals(const glabc_user_model_t* um, int32_t local_kind, int32_t far_kind, int32_t cc, char* log,
                                                size_t log_cap)
{
    if (log && log_cap) log[0] = '\0';
    if (!um || !um->source) return GLABC_ERR_INVALID;
    if (um->theta_dim < 1 || um->theta_dim > GLABC_MAX_DIM || um->y_dim < 1 || um->y_dim > 2 * GLABC_MAX_DIM || um->n_noise < 0 ||
        um->n_noise > GLABC_USER_MAX_NOISE || um->n_datasets < 0 || !valid_dist_kind(local_kind) || !valid_dist_kind(far_kind))
        return GLABC_ERR_INVALID;
    std::string err;
    const int st = user_model_check(cc, *um, local_kind, far_kind, err);
    if (log && log_cap) {
        strncpy(log, err.c_str(), log_cap - 1);
        log[log_cap - 1] = '\0';
    }
    return st;
}

extern "C" int glabc_user_model_check(const glabc_user_model_t* um, int32_t cc, char* log, size_t log_cap)
{
    return glabc_user_model_check_proposals(um, GLABC_DIST_DIAG_GAUSSIAN, GLABC_DIST_DIAG_GAUSSIAN, cc, log, log_cap);
}

// the checks of a user model every entry that launches one of its kernels makes first
static int check_user_model(glabc_ctx* ctx, const glabc_user_model_t* um, const char* who)
{
    if (!um || !um->source) return fail(ctx, GLABC_ERR_INVALID, "%s: null model / source", who);
    if (um->theta_dim < 1 || um->theta_dim > GLABC_MAX_DIM || um->y_dim < 1 || um->y_dim > 2 * GLABC_MAX_DIM)
        return fail(ctx, GLABC_ERR_INVALID, "user model: theta_dim in 1..%d, y_dim in 1..%d", GLABC_MAX_DIM, 2 * GLABC_MAX_DIM);
    if (um->n_noise < 0 || um->n_noise > GLABC_USER_MAX_NOISE || um->n_params < 0 || um->n_params > GLABC_USER_MAX_PARAMS)
        return fail(ctx, GLABC_ERR_INVALID, "user model: n_noise in 0..%d, n_params in 0..%d", GLABC_USER_MAX_NOISE, GLABC_USER_MAX_PARAMS);
    if (!(um->epsilon > 0.0)) return fail(ctx, GLABC_ERR_INVALID, "user model: epsilon must be positive");
    if (um->n_datasets < 0) return fail(ctx, GLABC_ERR_INVALID, "user model: n_datasets must be >= 0");
    if (um->n_datasets == 0) {
        if (um->dataset_params || um->chains_per_dataset != 0)
            return fail(ctx, GLABC_ERR_INVALID, "user model: dataset_params / chains_per_dataset given without n_datasets");
        return GLABC_OK;
    }
    if (!um->dataset_params) return fail(ctx, GLABC_ERR_INVALID, "batched user model: dataset_params is NULL with n_datasets %lld",
                                         static_cast<long long>(um->n_datasets));
    if (um->chains_per_dataset < 1) return fail(ctx, GLABC_ERR_INVALID, "batched user model: chains_per_dataset must be >= 1");
    if (um->chains_per_dataset > INT64_MAX / um->n_datasets)
        return fail(ctx, GLABC_ERR_INVALID, "batched user model: n_datasets * chains_per_dataset overflows int64");
    return GLABC_OK;
}

// a batched model's rows (chains or evaluation rows) first .. first + n - 1 must name datasets of its table
static int check_dataset_rows(glabc_ctx* ctx, const glabc_user_model_t* um, uint64_t first, int64_t n, const char* who)
{
    if (um->n_datasets == 0 || n <= 0) return GLABC_OK;
    const uint64_t total = static_cast<uint64_t>(um->n_datasets) * static_cast<uint64_t>(um->chains_per_dataset);
    if (first >= total || static_cast<uint64_t>(n) > total - first)
        return fail(ctx, GLABC_ERR_INVALID, "%s: ids %llu .. %llu reach beyond n_datasets x chains_per_dataset = %llu", who,
                    static_cast<unsigned long long>(first), static_cast<unsigned long long>(first + n - 1),
                    static_cast<unsigned long long>(total));
    return GLABC_OK;
}

// the batched-model fields of UserRun / UserEval (read by the kernels compiled with -DGLABC_BATCHED only)
template <class P>
static void set_dataset_table(const glabc_user_model_t& um, P* p)
{
    p->ds_params = um.dataset_params;
    p->ds_m = um.chains_per_dataset;
    p->ds_np = um.n_params;
}

// log K(dis) = kern_c + kern_m * dis^2, the Gaussian ABC kernel of width epsilon (Mixture.py:38-53)
static void user_kernel_consts(const glabc_user_model_t& um, float* kern_c, float* kern_m)
{
    const float eps = static_cast<float>(um.epsilon);
    *kern_c = static_cast<float>(-0.5 * std::log(2.0 * M_PI)) - std::log(eps);
    *kern_m = -0.5f / (eps * eps);
}

static int run_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_user_model_t* um, int kind)
{
    const bool isir = kind >= 1, mala = kind == 2;   // 0 GlobalMCMC, 1 GLMCMC (iSIR), 2 GLMALA
    if (!ctx) return GLABC_ERR_INVALID;
    if (int st = check_user_model(ctx, um, "glabc_run_*_user")) return st;
    if (run) {   // a batched model's chain ids (a negative chain_id_base reads as one beyond any table)
        if (int st = check_dataset_rows(ctx, um, static_cast<uint64_t>(run->chain_id_base), run->n_chains, "glabc_run_*_user")) return st;
    }
    const int d = um->theta_dim;
    const int far_slot = isir ? GLABC_SLOT_IMPORTANCE : GLABC_SLOT_GLOBAL;   // the state-independent proposal of the sampler
    for (int slot : {mala ? far_slot : static_cast<int>(GLABC_SLOT_LOCAL), far_slot}) {
        if (!ctx->has_dist[slot])
            return fail(ctx, GLABC_ERR_INVALID, "%s needs the %s%s proposal slot(s) bound", mala ? "glabc_run_mala_user" : isir ? "glabc_run_isir_user" : "glabc_run_global_user",
                        mala ? "" : "LOCAL and ", isir ? "IMPORTANCE" : "GLOBAL");
        if (ctx->dist[slot].dim != d) return fail(ctx, GLABC_ERR_INVALID, "proposal dim does not match the user model's theta_dim %d", d);
    }
    if (isir) {
        if (!run) return fail(ctx, GLABC_ERR_INVALID, "null run description");
        if (run->n_candidates < 1 || run->n_candidates > GLABC_MAX_K)
            return fail(ctx, GLABC_ERR_INVALID, "n_candidates (batch_size) must be in 1..%d", GLABC_MAX_K);
        if (!run->aux) return fail(ctx, GLABC_ERR_INVALID, "glabc_run_isir_user needs the aux state [C][%d] (log-weight, local flag)", GLABC_AUX_SLOTS);
    }
    if (mala) {
        if (d > GLABC_AUX_SLOTS - 3) return fail(ctx, GLABC_ERR_UNSUPPORTED, "glabc_run_mala_user: theta_dim at most %d (the cached gradient lives in the aux slots)", GLABC_AUX_SLOTS - 3);
        if (run->num_grad < 2 || run->num_grad > GLABC_MAX_NUM_GRAD) return fail(ctx, GLABC_ERR_INVALID, "num_grad must be in 2..%d", GLABC_MAX_NUM_GRAD);
        if (!(run->tau > 0.0f)) return fail(ctx, GLABC_ERR_INVALID, "tau must be positive");
    }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    RunParams R;
    int block = 0;
    int st = make_run_params(ctx, run, d, 0, &R, &block);
    if (st) return st;
    if (run->rng_mode != GLABC_RNG_NATIVE) return fail(ctx, GLABC_ERR_UNSUPPORTED, "the user-model kernels run the native RNG only");
    CUDA_TRY(ctx, cudaFree(nullptr));   // make sure the primary context exists and is current for the driver calls
    void* fn = nullptr;
    std::string err;
    const glabc_dist_t& lp = ctx->dist[mala ? far_slot : GLABC_SLOT_LOCAL];   // GLMALA has no Local_Proposal
    const glabc_dist_t& gp = ctx->dist[far_slot];
    // the kinds are compiled in; GLMALA reads only the IMPORTANCE slot, so its module takes the Gaussian local path
    const int lp_kind = mala ? GLABC_DIST_DIAG_GAUSSIAN : lp.kind;
    st = user_model_compile(ctx->device, ctx->cc, *um, lp_kind, gp.kind, kind, &fn, err);
    if (st) return fail(ctx, st, "%s", err.c_str());
    UserRun U{};
    U.n_chains = R.n_chains;
    U.first_step = R.first_step;
    U.last_step = R.last_step;
    U.chain_lo0 = R.chain_lo0;
    U.chain_hi0 = R.chain_hi0;
    U.key0 = static_cast<uint32_t>(run->seed);
    U.key1 = static_cast<uint32_t>(run->seed >> 32);
    const double gf = static_cast<double>(run->global_frequency);
    U.gf_all_global = gf >= 1.0;
    U.gf_thr = gf <= 0.0 ? 0u : (gf >= 1.0 ? 0xFFFFFFFFu : static_cast<uint32_t>(gf * 4294967296.0));
    U.write_row0 = R.write_row0;
    U.trace_layout = run->trace_layout;
    U.trace_rows = R.trace_rows;
    U.trace_chains = R.trace_chains;
    U.trace_chain_off = R.trace_chain_off;
    U.trace_row_base = R.trace_row_base;
    U.theta = R.theta;
    U.y = R.y;
    U.trace = R.trace;
    U.stats = R.stats;
    if (mala) {
        U.tau = run->tau;
        U.eps2 = static_cast<float>(um->epsilon * um->epsilon);
        U.num_grad = run->num_grad;
    }
    U.aux = isir ? run->aux : nullptr;
    U.n_candidates = isir ? run->n_candidates : 0;
    for (int k = 0; k < d; ++k) {   // glabc_dist_t DiagGaussian: a = loc, b = log_scale, c = exp(log_scale) in float32
        if (lp.kind == GLABC_DIST_DIAG_GAUSSIAN) {
            U.lp_loc[k] = lp.a[k];
            U.lp_scale[k] = lp.c[k];
        }
        if (gp.kind == GLABC_DIST_DIAG_GAUSSIAN) {
            U.gp_loc[k] = gp.a[k];
            U.gp_scale[k] = gp.c[k];
            U.gp_inv_scale[k] = 1.0f / gp.c[k];
        }
    }
    U.lq = make_dist<GLABC_MAX_DIM>(lp);   // read by the kernels compiled for a Uniform / Gamma / GaussianMixture slot
    U.gq = make_dist<GLABC_MAX_DIM>(gp);
    user_kernel_consts(*um, &U.kern_c, &U.kern_m);
    for (int k = 0; k < um->n_params; ++k) U.params[k] = um->params[k];
    set_dataset_table(*um, &U);
    st = user_model_launch(fn, U, mala ? 64 : (block > 128 ? 128 : block), static_cast<cudaStream_t>(run->stream), err);
    if (st) return fail(ctx, st, "%s", err.c_str());
    return GLABC_OK;
}

extern "C" int glabc_run_global_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_user_model_t* um) { return run_user(ctx, run, um, 0); }
extern "C" int glabc_run_isir_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_user_model_t* um) { return run_user(ctx, run, um, 1); }
extern "C" int glabc_run_mala_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_user_model_t* um) { return run_user(ctx, run, um, 2); }

// glabc_k_block_isir_user (weights = false) / glabc_k_block_weights_user: the block-iSIR step and the block weights of
// glabc_run_block_isir / glabc_block_weights for a user model
static int run_block_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_block_isir_t* b, uint32_t round,
                          const glabc_user_model_t* um, bool weights)
{
    const char* who = weights ? "glabc_block_weights_user" : "glabc_run_block_isir_user";
    if (!ctx) return GLABC_ERR_INVALID;
    if (int st = check_user_model(ctx, um, who)) return st;
    if (um->n_datasets > 0)   // a block-iSIR proposal is trained on, or pooled over, all chains: meaningless across datasets
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "%s: a batched user model (n_datasets > 0) is not supported", who);
    if (!run || !b) return fail(ctx, GLABC_ERR_INVALID, "%s: null run / block description", who);
    const int d = um->theta_dim;
    if (!ctx->has_dist[GLABC_SLOT_LOCAL]) return fail(ctx, GLABC_ERR_INVALID, "%s needs the LOCAL proposal slot bound", who);
    const glabc_dist_t& lp = ctx->dist[GLABC_SLOT_LOCAL];
    if (lp.dim != d) return fail(ctx, GLABC_ERR_INVALID, "proposal dim does not match the user model's theta_dim %d", d);
    if (int st = check_block(ctx, who, run, b)) return st;
    if (run->arith_mode == GLABC_ARITH_STRICT || run->rng_mode == GLABC_RNG_REPLAY)
        return fail(ctx, GLABC_ERR_UNSUPPORTED, "%s: the user-model kernels run FAST arithmetic with the native RNG only", who);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    RunParams R;
    int block = 0;
    int st = make_run_params(ctx, run, d, 0, &R, &block);
    if (st) return st;
    if (R.n_chains == 0) return GLABC_OK;
    CUDA_TRY(ctx, cudaFree(nullptr));   // the primary context, current for the driver calls
    void* fn = nullptr;
    std::string err;
    st = user_model_block_fn(ctx->device, ctx->cc, *um, lp.kind, weights, &fn, err);
    if (st) return fail(ctx, st, "%s", err.c_str());
    UserBlockRun U{};
    U.n_chains = R.n_chains;
    U.block = b->block;
    U.step_size = b->step_size;
    U.n_candidates = run->n_candidates;
    U.first_step = R.first_step;
    U.last_step = R.last_step;
    U.chain_lo0 = R.chain_lo0;
    U.chain_hi0 = R.chain_hi0;
    U.key0 = static_cast<uint32_t>(run->seed);
    U.key1 = static_cast<uint32_t>(run->seed >> 32);
    const double gf = static_cast<double>(run->global_frequency);
    U.gf_all_global = gf >= 1.0;
    U.gf_thr = gf <= 0.0 ? 0u : (gf >= 1.0 ? 0xFFFFFFFFu : static_cast<uint32_t>(gf * 4294967296.0));
    U.round = round;
    U.write_row0 = R.write_row0;
    U.trace_layout = run->trace_layout;
    U.trace_rows = R.trace_rows;
    U.trace_chains = R.trace_chains;
    U.trace_chain_off = R.trace_chain_off;
    U.trace_row_base = R.trace_row_base;
    U.theta = R.theta;
    U.y = R.y;
    U.trace = R.trace;
    U.stats = R.stats;
    U.blk_theta = b->blk_theta;
    U.blk_x = b->blk_x;
    U.blk_w = b->blk_w;
    U.blk_lq = b->blk_lq;
    U.kk = b->kk;
    U.pending = b->pending;
    U.next_step = b->next_step;
    U.lq_cur = b->lq_cur;
    U.lq_valid = b->lq_valid;
    if (lp.kind == GLABC_DIST_DIAG_GAUSSIAN)
        for (int k = 0; k < d; ++k) {
            U.lp_loc[k] = lp.a[k];
            U.lp_scale[k] = lp.c[k];
        }
    U.lq = make_dist<GLABC_MAX_DIM>(lp);
    user_kernel_consts(*um, &U.kern_c, &U.kern_m);
    for (int k = 0; k < um->n_params; ++k) U.params[k] = um->params[k];
    st = user_model_block_launch(fn, U, weights, static_cast<cudaStream_t>(run->stream), err);
    if (st) return fail(ctx, st, "%s", err.c_str());
    return GLABC_OK;
}

extern "C" int glabc_run_block_isir_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_block_isir_t* blk, const glabc_user_model_t* model)
{
    return run_block_user(ctx, run, blk, 0u, model, false);
}

extern "C" int glabc_block_weights_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_block_isir_t* blk, uint32_t round,
                                        const glabc_user_model_t* model)
{
    return run_block_user(ctx, run, blk, round, model, true);
}

// glabc_k_eval_user on n rows; the caller has checked ctx, the model, n and the buffers
static int eval_user(glabc_ctx* ctx, const glabc_user_model_t* um, int op, const float* in, int64_t n, uint64_t seed,
                     uint64_t row_base, float* out, void* stream)
{
    if (n == 0) return GLABC_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaFree(nullptr));   // the primary context, current for the driver calls
    void* fn = nullptr;
    std::string err;
    int st = user_model_eval_fn(ctx->device, ctx->cc, *um, &fn, err);
    if (st) return fail(ctx, st, "%s", err.c_str());
    UserEval E{};
    E.n = n;
    E.op = op;
    E.row_lo = static_cast<uint32_t>(row_base);
    E.row_hi = static_cast<uint32_t>(row_base >> 32);
    E.key0 = static_cast<uint32_t>(seed);
    E.key1 = static_cast<uint32_t>(seed >> 32);
    E.in = in;
    E.out = out;
    user_kernel_consts(*um, &E.kern_c, &E.kern_m);
    for (int k = 0; k < um->n_params; ++k) E.params[k] = um->params[k];
    set_dataset_table(*um, &E);
    st = user_model_eval_launch(fn, E, ctx->sm_count, static_cast<cudaStream_t>(stream), err);
    if (st) return fail(ctx, st, "%s", err.c_str());
    return GLABC_OK;
}

extern "C" int glabc_user_simulate(glabc_ctx* ctx, const glabc_user_model_t* um, const float* theta, int64_t n, uint64_t seed,
                                   uint64_t row_base, float* y, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (int st = check_user_model(ctx, um, "glabc_user_simulate")) return st;
    if (n < 0 || (n > 0 && (!theta || !y))) return fail(ctx, GLABC_ERR_INVALID, "glabc_user_simulate: null buffer / n < 0");
    if (int st = check_dataset_rows(ctx, um, row_base, n, "glabc_user_simulate")) return st;
    return eval_user(ctx, um, GLABC_USER_SIMULATE, theta, n, seed, row_base, y, stream);
}

extern "C" int glabc_user_evaluate(glabc_ctx* ctx, const glabc_user_model_t* um, int32_t op, const float* x, int64_t n, float* out,
                                   void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (int st = check_user_model(ctx, um, "glabc_user_evaluate")) return st;
    if (op != GLABC_USER_PRIOR && op != GLABC_USER_DISCREPANCY && op != GLABC_USER_LOG_KERNEL)
        return fail(ctx, GLABC_ERR_INVALID, "glabc_user_evaluate: unknown op %d", op);
    if (n < 0 || (n > 0 && (!x || !out))) return fail(ctx, GLABC_ERR_INVALID, "glabc_user_evaluate: null buffer / n < 0");
    if (int st = check_dataset_rows(ctx, um, 0, n, "glabc_user_evaluate")) return st;
    return eval_user(ctx, um, op, x, n, 0, 0, out, stream);
}


// ---------------------------------------------------------------------------------------------
// Host entry of GlobalMCMC with a chain-major host trace: part of the chains travels as EVENTS.
// A chain is piecewise constant (the README workload moves on 1.2 % of its steps), so its dense float32 trace is 98 %
// repetition and the 5.2 GB device -> host copy of 65,536 x 1e4 rows is what bounds the call (PCIe, ~55 GB/s).  Here the
// last `f` of the chains are run with GLABC_TRACE_EVENTS, their moves (a few hundred KB per thousand chains) are copied
// back, and the host cores expand them into the caller's dense buffer WHILE the DMA engine brings the other chains' dense
// rows over PCIe (dense_chain_groups below).  The caller's buffer ends up bit-identical to the all-dense path.
// A chain with more moves than the event capacity makes the event part fall back to the dense path.
// Environment: GLABC_HOST_EVENTS=0 disables the event transport; GLABC_HOST_EVENT_FRACTION sets the share of the chains that
// travels as events (default 1 with AVX-512 stores, else 0.6); GLABC_HOST_TIMING prints the phase times to stderr.  The
// expansion takes the host's cores, split between the ranks of a node by LOCAL_WORLD_SIZE.
// ---------------------------------------------------------------------------------------------
// Run-length expansion of one chain into the caller's dense rows.  With AVX-512 and a row size that divides a cache line
// (d in {1, 2, 4}) the whole chain is written as FULL 64-byte lines with non-temporal stores — a line that straddles a move
// is assembled in a register first — so no line is read for ownership: 137 GB/s on the 16 host cores of the B200 box against
// 65 GB/s for ordinary stores (profiles/micro/host_fill.cu; narrower NT stores are slower than ordinary ones).
__attribute__((target("avx512f"))) static void expand_chain_nt512(const float* ev, uint32_t m, int d, int64_t row_base, int64_t row_end,
                                                                  float* out)
{
    const int per_line = 16 / d;
    alignas(64) float buf[16], pat[16];
    int lv = 0;                       // floats of the current (aligned) line already assembled in buf
    float* dst = nullptr;             // next float to write
    bool aligned = false;
    for (uint32_t k = 1; k <= m; ++k) {
        const float* e = ev + static_cast<int64_t>(k) * (1 + d);
        uint32_t r0, r1;
        memcpy(&r0, e, sizeof(r0));
        if (k < m) memcpy(&r1, e + (1 + d), sizeof(r1));
        else r1 = static_cast<uint32_t>(row_end + 1);
        int64_t n = static_cast<int64_t>(r1) - r0;
        const float* row = e + 1;
        if (k == 1) dst = out + (static_cast<int64_t>(r0) - row_base) * d;
        while (!aligned && n > 0) {   // head of the chain: whole rows up to the first cache-line boundary
            if ((reinterpret_cast<uintptr_t>(dst) & 63u) == 0) {
                aligned = true;
                break;
            }
            for (int i = 0; i < d; ++i) dst[i] = row[i];
            dst += d;
            --n;
        }
        if (n == 0) continue;
        if (lv > 0) {                 // finish the line a previous run left open
            while (lv < 16 && n > 0) {
                for (int i = 0; i < d; ++i) buf[lv + i] = row[i];
                lv += d;
                --n;
            }
            if (lv == 16) {
                _mm512_stream_ps(dst, _mm512_load_ps(buf));
                dst += 16;
                lv = 0;
            }
        }
        if (n >= per_line) {
            for (int i = 0; i < 16; ++i) pat[i] = row[i % d];
            const __m512 v = _mm512_load_ps(pat);
            const int64_t lines = n / per_line;
            for (int64_t l = 0; l < lines; ++l) _mm512_stream_ps(dst + l * 16, v);
            dst += lines * 16;
            n -= lines * per_line;
        }
        for (; n > 0; --n) {          // open the next line
            for (int i = 0; i < d; ++i) buf[lv + i] = row[i];
            lv += d;
        }
    }
    for (int i = 0; i < lv; ++i) dst[i] = buf[i];   // tail of the chain
}

static void fill_rows_plain(float* dst, int64_t n, const float* row, int d)
{
    if (d == 2) {
        float2* p = reinterpret_cast<float2*>(dst);
        const float2 v = make_float2(row[0], row[1]);
        for (int64_t i = 0; i < n; ++i) p[i] = v;
    } else {
        for (int64_t i = 0; i < n; ++i)
            for (int k = 0; k < d; ++k) dst[i * d + k] = row[k];
    }
}

static void expand_chain(const float* ev, int64_t cap, int d, int64_t row_base, int64_t row_end, float* out, bool nt512)
{
    uint32_t m;
    memcpy(&m, ev, sizeof(m));
    if (m > cap - 1) m = static_cast<uint32_t>(cap - 1);
    if (nt512) {
        expand_chain_nt512(ev, m, d, row_base, row_end, out);
        return;
    }
    for (uint32_t k = 1; k <= m; ++k) {
        const float* e = ev + static_cast<int64_t>(k) * (1 + d);
        uint32_t r0, r1;
        memcpy(&r0, e, sizeof(r0));
        if (k < m) memcpy(&r1, e + (1 + d), sizeof(r1));
        else r1 = static_cast<uint32_t>(row_end + 1);
        fill_rows_plain(out + (static_cast<int64_t>(r0) - row_base) * d, static_cast<int64_t>(r1) - r0, e + 1, d);
    }
}

// Expands chains [c0, c1) of an event buffer [chains][cap][1 + d] into the chain-major rows of `trace` [chains][trace_rows][d]
// on n_threads host threads, the chains dealt round-robin.
static void expand_parallel(const float* events, int64_t c0, int64_t c1, int64_t cap, int d, int64_t row_base, int64_t row_end,
                            float* trace, int64_t trace_rows, int n_threads, bool nt512)
{
    std::vector<std::thread> workers;
    for (int t = 0; t < n_threads; ++t)
        workers.emplace_back([=]() {
            for (int64_t c = c0 + t; c < c1; c += n_threads)
                expand_chain(events + c * cap * (1 + d), cap, d, row_base, row_end, trace + c * trace_rows * d, nt512);
            _mm_sfence();   // the non-temporal stores are globally visible before the thread is joined
        });
    for (auto& w : workers) w.join();
}

// Dense transport for a chain-major host trace: the chains are run in GROUPS over all their steps, and each group's
// [chains][rows][d] block — contiguous on both sides — goes back in one full-rate copy while the next group's kernel runs
// (time chunks of a chain-major trace would be 2-D copies of ~1 KB segments, which the DMA engine moves at half the rate).
static int dense_chain_groups(glabc_ctx* ctx, SamplerKind kind, const glabc_run_t* run, int64_t Cd)
{
    const int d = ctx->model.theta_dim;
    const int64_t n_rows = run->n_steps + (run->write_row0 ? 1 : 0);
    const int64_t row_lo = run->step_base + (run->write_row0 ? 0 : 1);
    int64_t Cg = (int64_t(320) << 20) / (n_rows * d * int64_t(sizeof(float))) / 32 * 32;
    if (Cg < 32) Cg = 32;
    if (Cg > Cd) Cg = Cd;
    ChainState state;
    int st = ensure_host_scratch(ctx, run, Cd, size_t(Cg) * n_rows * d, &state);
    if (st) return st;
    cudaStream_t sc = ctx->s_compute, sx = ctx->s_copy;
    CUDA_TRY(ctx, stage_state(ctx, run, 0, Cd, state, cudaMemcpyHostToDevice, sc));
    bool used[2] = {false, false};
    int b = 0;
    for (int64_t g0 = 0; g0 < Cd; g0 += Cg) {
        const int64_t n = std::min<int64_t>(Cg, Cd - g0);
        glabc_run_t dev = chain_slice(run, g0, n, chains_at(ctx, state, g0), sc);
        dev.trace = ctx->d_trace[b].p;
        dev.trace_rows = n_rows;
        dev.trace_chains = n;
        dev.trace_chain_off = 0;
        dev.trace_row_base = row_lo;
        if (used[b]) CUDA_TRY(ctx, cudaStreamWaitEvent(sc, ctx->ev_free[b], 0));
        st = run_device(ctx, kind, &dev);
        if (st) return st;
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_done[b], sc));
        CUDA_TRY(ctx, cudaStreamWaitEvent(sx, ctx->ev_done[b], 0));
        float* dst = run->trace + ((run->trace_chain_off + g0) * run->trace_rows + (row_lo - run->trace_row_base)) * d;
        CUDA_TRY(ctx, cudaMemcpy2DAsync(dst, size_t(run->trace_rows) * d * sizeof(float), ctx->d_trace[b].p, size_t(n_rows) * d * sizeof(float),
                                        size_t(n_rows) * d * sizeof(float), size_t(n), cudaMemcpyDeviceToHost, sx));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_free[b], sx));
        used[b] = true;
        b ^= 1;
    }
    CUDA_TRY(ctx, stage_state(ctx, run, 0, Cd, state, cudaMemcpyDeviceToHost, sc));
    CUDA_TRY(ctx, cudaStreamSynchronize(sc));
    CUDA_TRY(ctx, cudaStreamSynchronize(sx));
    return GLABC_OK;
}

// The dense transport of GlobalMCMC / GLMCMC: a chain-major trace with the default chunking (chunk_steps == 0) travels chain
// group by chain group, anything else in time chunks.
static int run_host_dense(glabc_ctx* ctx, SamplerKind kind, const glabc_run_t* run, int64_t chunk_steps)
{
    if (run->trace_layout == GLABC_TRACE_CHAIN_MAJOR && chunk_steps == 0 && run->n_steps > 0)
        return dense_chain_groups(ctx, kind, run, run->n_chains);
    return run_host(ctx, kind, run, chunk_steps);
}

static int run_global_host_hybrid(glabc_ctx* ctx, SamplerKind kind, const glabc_run_t* run, int64_t chunk_steps, bool* handled)
{
    *handled = false;
    const char* off = getenv("GLABC_HOST_EVENTS");
    if (off && off[0] == '0') return GLABC_OK;
    if (run->trace_layout != GLABC_TRACE_CHAIN_MAJOR || run->n_steps < 512 || run->n_chains < 256) return GLABC_OK;
    const int far_slot = kind == SAMPLER_ISIR ? GLABC_SLOT_IMPORTANCE : GLABC_SLOT_GLOBAL;
    // the event writer lives in the tuned kernels only: Gaussian proposals and the model's DiagGaussian prior
    if (!ctx->has_dist[GLABC_SLOT_LOCAL] || !ctx->has_dist[far_slot] || !all_gaussian(ctx, {GLABC_SLOT_LOCAL, far_slot}) || ctx->has_prior)
        return GLABC_OK;
    if (kind == SAMPLER_ISIR && !run->aux) return GLABC_OK;
    const int d = ctx->model.theta_dim, yd = ctx->model.y_dim, ns = GLABC_NSTATS(d);
    const bool nt512 = (d == 1 || d == 2 || d == 4) && __builtin_cpu_supports("avx512f");
    // with full-line non-temporal stores the expansion alone runs at the host's DRAM write rate, which a concurrent dense DMA
    // would only share; with ordinary stores (65 GB/s) the PCIe copy of part of the chains adds bandwidth
    double frac = nt512 ? 1.0 : 0.6;
    if (const char* f = getenv("GLABC_HOST_EVENT_FRACTION")) frac = atof(f);
    if (!(frac > 0.0)) return GLABC_OK;
    if (frac > 1.0) frac = 1.0;
    const int64_t C = run->n_chains;
    int64_t Ce = static_cast<int64_t>(C * frac) / 32 * 32;
    if (Ce <= 0) return GLABC_OK;
    const int64_t Cd = C - Ce;
    const int64_t row_end = run->step_base + run->n_steps;
    *handled = true;
    if (!ctx->s_ev) {
        CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_ev, cudaStreamNonBlocking));
        for (auto& e : ctx->ev_group) CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    int64_t cap = run->n_steps / 32;
    if (cap < 64) cap = 64;
    if (cap > run->n_steps + 2) cap = run->n_steps + 2;
    const size_t n_state = state_floats(ctx, run, Ce), n_events = size_t(Ce) * size_t(cap) * (1 + d);
    CUDA_TRY(ctx, ctx->d_ev.reserve(n_state + n_events));
    CUDA_TRY(ctx, ctx->h_ev.reserve(n_state + n_events));
    const ChainState state = carve_state(ctx, run, Ce, ctx->d_ev.p, nullptr);   // the event chains' state, then their events
    float* d_events = ctx->d_ev.p + n_state;
    float* h_state = ctx->h_ev.p;                 // final state of the event chains, committed once no chain overflowed
    float* h_events = ctx->h_ev.p + n_state;
    cudaStream_t se = ctx->s_ev;
    CUDA_TRY(ctx, stage_state(ctx, run, Cd, Ce, state, cudaMemcpyHostToDevice, se));
    // the event chains in up to 8 groups: the kernel of group g + 1 and the copy of group g's events overlap the expansion of
    // group g - 1 on the host cores
    // (a group's kernel is latency-bound — a chain's steps are sequential — so it takes about as long as a full launch's warp:
    // many small groups are free for the 2 ms GlobalMCMC kernel, while the 24 ms iSIR kernel is cut in three at most)
    int n_groups = static_cast<int>(Ce / 8192);
    const int max_groups = kind == SAMPLER_ISIR ? 3 : 8;
    if (n_groups < 1) n_groups = 1;
    if (n_groups > max_groups) n_groups = max_groups;
    const int64_t per_group = ((Ce + n_groups - 1) / n_groups + 31) / 32 * 32;
    int st = GLABC_OK;
    for (int g = 0; g < n_groups; ++g) {
        const int64_t g0 = g * per_group, gn = std::min<int64_t>(per_group, Ce - g0);
        if (gn <= 0) {
            n_groups = g;
            break;
        }
        glabc_run_t dev = chain_slice(run, Cd + g0, gn, chains_at(ctx, state, g0), se);
        dev.trace = d_events + g0 * cap * (1 + d);
        dev.trace_layout = GLABC_TRACE_EVENTS;
        dev.trace_rows = cap;
        dev.trace_chains = gn;
        dev.trace_chain_off = 0;
        dev.trace_row_base = 0;
        st = run_device(ctx, kind, &dev);
        if (st) return st;
        CUDA_TRY(ctx, cudaMemcpyAsync(h_events + g0 * cap * (1 + d), d_events + g0 * cap * (1 + d), size_t(gn) * cap * (1 + d) * sizeof(float),
                                      cudaMemcpyDeviceToHost, se));
        if (g == n_groups - 1) CUDA_TRY(ctx, cudaMemcpyAsync(h_state, ctx->d_ev.p, n_state * sizeof(float), cudaMemcpyDeviceToHost, se));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_group[g], se));
    }

    // the host cores expand the events while the dense part (below) streams over PCIe
    std::atomic<int> overflow{0};
    // one process per GPU shares the host's cores: LOCAL_WORLD_SIZE (torchrun) divides them between the ranks
    int n_threads = static_cast<int>(std::thread::hardware_concurrency());
    if (const char* lws = getenv("LOCAL_WORLD_SIZE")) {
        const int r = atoi(lws);
        if (r > 1) n_threads = (n_threads + r - 1) / r;
    }
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 64) n_threads = 64;
    const int device = ctx->device;
    cudaEvent_t evg[8];
    for (int g = 0; g < 8; ++g) evg[g] = ctx->ev_group[g];
    const int64_t trace_rows = run->trace_rows, row_base = run->trace_row_base;
    float* ev_trace = run->trace + (run->trace_chain_off + Cd) * trace_rows * d;   // row 0 of the first event chain
    const bool timing = getenv("GLABC_HOST_TIMING") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    auto ms_since = [t_start]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count(); };
    std::thread expander([=, &overflow]() {
        cudaSetDevice(device);
        double t_first = 0.0;
        for (int g = 0; g < n_groups; ++g) {
            if (cudaEventSynchronize(evg[g]) != cudaSuccess) {
                overflow.store(2);
                return;
            }
            if (g == 0) t_first = ms_since();
            const int64_t g0 = g * per_group, g1 = std::min<int64_t>(g0 + per_group, Ce);
            for (int64_t j = g0; j < g1; ++j) {   // a chain with more moves than the capacity: the event part is redone densely
                uint32_t m;
                memcpy(&m, h_events + j * cap * (1 + d), sizeof(m));
                if (m > static_cast<uint32_t>(cap - 1)) {
                    overflow.store(1);
                    return;
                }
            }
            expand_parallel(h_events, g0, g1, cap, d, row_base, row_end, ev_trace, trace_rows, n_threads, nt512);
        }
        if (timing) fprintf(stderr, "[glabc host] first events at %.1f ms, all expanded at %.1f ms (%lld chains, %d groups, %d threads, nt512 %d)\n",
                            t_first, ms_since(), static_cast<long long>(Ce), n_groups, n_threads, static_cast<int>(nt512));
    });

    if (Cd > 0) st = dense_chain_groups(ctx, kind, run, Cd);   // the dense part: chains [0, Cd), group by group over PCIe
    if (timing) fprintf(stderr, "[glabc host] dense part (%lld chains) done at %.1f ms\n", static_cast<long long>(Cd), ms_since());
    expander.join();
    if (timing) fprintf(stderr, "[glabc host] joined at %.1f ms\n", ms_since());
    if (st) return st;
    if (overflow.load() == 2) return fail(ctx, GLABC_ERR_CUDA, "event transport: waiting for the event copy failed");
    if (overflow.load() == 1) {   // redo the event chains densely from their (untouched) initial host state
        glabc_run_t redo = chain_slice(run, Cd, Ce, chains_at(ctx, host_state(run), Cd), nullptr);
        redo.trace_chain_off = run->trace_chain_off + Cd;
        return run_host_dense(ctx, kind, &redo, chunk_steps);
    }
    const ChainState staged = carve_state(ctx, run, Ce, h_state, nullptr);
    memcpy(run->theta + Cd * d, staged.theta, size_t(Ce) * d * sizeof(float));
    memcpy(run->y + Cd * yd, staged.y, size_t(Ce) * yd * sizeof(float));
    if (staged.aux) memcpy(run->aux + Cd * GLABC_AUX_SLOTS, staged.aux, size_t(Ce) * GLABC_AUX_SLOTS * sizeof(float));
    if (staged.stats) memcpy(run->stats + Cd * ns, staged.stats, size_t(Ce) * ns * sizeof(float));
    return GLABC_OK;
}

// The host-buffer entry points: the argument check, then for GlobalMCMC / GLMCMC the event transport where it applies and
// the dense transport otherwise; GLMALA and AGLMCMC travel in time chunks.
static int run_host_entry(glabc_ctx* ctx, SamplerKind kind, const glabc_run_t* run, int64_t chunk_steps, const glabc_aglmcmc_t* ag = nullptr)
{
    int st = check_host_run(ctx, run);
    if (st || run->n_chains == 0) return st;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (kind == SAMPLER_MALA || kind == SAMPLER_AGLMCMC) return run_host(ctx, kind, run, chunk_steps, ag);
    bool handled = false;
    st = run_global_host_hybrid(ctx, kind, run, chunk_steps, &handled);
    if (handled || st) return st;
    return run_host_dense(ctx, kind, run, chunk_steps);
}

extern "C" {

int glabc_run_global(glabc_ctx* ctx, const glabc_run_t* run) { return run_device(ctx, SAMPLER_GLOBAL, run); }

int glabc_run_global_host(glabc_ctx* ctx, const glabc_run_t* run, int64_t chunk_steps)
{
    return run_host_entry(ctx, SAMPLER_GLOBAL, run, chunk_steps);
}

int glabc_run_isir(glabc_ctx* ctx, const glabc_run_t* run) { return run_device(ctx, SAMPLER_ISIR, run); }

int glabc_run_isir_host(glabc_ctx* ctx, const glabc_run_t* run, int64_t chunk_steps)
{
    return run_host_entry(ctx, SAMPLER_ISIR, run, chunk_steps);
}

int glabc_run_mala(glabc_ctx* ctx, const glabc_run_t* run) { return run_device(ctx, SAMPLER_MALA, run); }

int glabc_run_mala_host(glabc_ctx* ctx, const glabc_run_t* run, int64_t chunk_steps)
{
    return run_host_entry(ctx, SAMPLER_MALA, run, chunk_steps);
}

int glabc_run_aglmcmc_host(glabc_ctx* ctx, const glabc_run_t* run, const glabc_aglmcmc_t* ag, int64_t chunk_steps)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ag) return fail(ctx, GLABC_ERR_INVALID, "null aglmcmc description");
    return run_host_entry(ctx, SAMPLER_AGLMCMC, run, chunk_steps, ag);
}

int glabc_resample(glabc_ctx* ctx, const float* W, int64_t n, int64_t N, float u0, int64_t* idx, uint64_t* count, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (n < 0 || N < 0 || (n > 0 && !W) || (N > 0 && !idx) || !count) return fail(ctx, GLABC_ERR_INVALID, "glabc_resample: bad sizes / null pointer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, ctx->rs_scratch.reserve(static_cast<size_t>((n + 4095) / 4096) + 1));
    CUDA_TRY(ctx, launch_resample(W, n, N, u0, idx, reinterpret_cast<unsigned long long*>(count), ctx->rs_scratch.p,
                                  static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

int glabc_esjd(glabc_ctx* ctx, const float* trace, int32_t layout, int64_t rows, int64_t chains, int32_t dim, float* out,
               void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!trace || !out) return fail(ctx, GLABC_ERR_INVALID, "glabc_esjd: null pointer");
    if (layout != GLABC_TRACE_TIME_MAJOR && layout != GLABC_TRACE_CHAIN_MAJOR)
        return fail(ctx, GLABC_ERR_INVALID, "glabc_esjd: bad layout %d", layout);
    if (rows < 2) return fail(ctx, GLABC_ERR_INVALID, "glabc_esjd: needs at least 2 rows");
    if (dim < 1 || dim > 3) return fail(ctx, GLABC_ERR_UNSUPPORTED, "glabc_esjd: dim %d outside 1..3", dim);
    if (chains <= 0) return GLABC_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, launch_esjd(trace, layout, rows, chains, dim, out, static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

int glabc_expand_events(const float* events, int64_t chains, int64_t cap, int32_t dim, int64_t row_base, int64_t row_end, float* trace,
                        int64_t trace_rows, int32_t n_threads)
{
    if (!events || !trace || chains < 0 || cap < 2 || dim < 1 || dim > GLABC_MAX_DIM || row_end < row_base || row_end - row_base >= trace_rows)
        return GLABC_ERR_INVALID;
    for (int64_t c = 0; c < chains; ++c) {   // validate before writing anything: counts within capacity, rows ascending and in range
        const float* ev = events + c * cap * (1 + dim);
        uint32_t m;
        memcpy(&m, ev, sizeof(m));
        if (m > static_cast<uint32_t>(cap - 1)) return GLABC_ERR_INVALID;
        int64_t prev = row_base - 1;
        for (uint32_t k = 1; k <= m; ++k) {
            uint32_t r;
            memcpy(&r, ev + static_cast<int64_t>(k) * (1 + dim), sizeof(r));
            if (static_cast<int64_t>(r) <= prev || static_cast<int64_t>(r) > row_end) return GLABC_ERR_INVALID;
            prev = r;
        }
    }
    const bool nt512 = (dim == 1 || dim == 2 || dim == 4) && __builtin_cpu_supports("avx512f");
    int nt = n_threads > 0 ? n_threads : static_cast<int>(std::thread::hardware_concurrency());
    if (nt < 1) nt = 1;
    if (nt > 64) nt = 64;
    if (nt > chains) nt = chains > 0 ? static_cast<int>(chains) : 1;
    expand_parallel(events, 0, chains, cap, dim, row_base, row_end, trace, trace_rows, nt, nt512);
    return GLABC_OK;
}

int glabc_summarize(glabc_ctx* ctx, const float* stats, int64_t chains, int32_t dim, double* out, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!out || (chains > 0 && !stats)) return fail(ctx, GLABC_ERR_INVALID, "glabc_summarize: null pointer");
    if (dim < 1 || dim > 4) return fail(ctx, GLABC_ERR_UNSUPPORTED, "glabc_summarize: dim %d outside 1..4", dim);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, launch_summarize(stats, chains, dim, out, static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

int glabc_philox_kat(glabc_ctx* ctx, const uint32_t* ctr, const uint32_t* key, int64_t n, uint32_t* out, void* stream)
{
    if (!ctx) return GLABC_ERR_INVALID;
    if (!ctr || !key || !out) return fail(ctx, GLABC_ERR_INVALID, "glabc_philox_kat: null pointer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, launch_philox_kat(ctr, key, n, out, static_cast<cudaStream_t>(stream)));
    return GLABC_OK;
}

}  // extern "C"
