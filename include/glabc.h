/*
 * glabc.h — C-ABI of the B200-native GL-ABC-MCMC sampler inner loop.
 *
 * The reference (caofff/GL-ABC-MCMC, `glabcmcmc` 1.0.1) is pure Python and has no FFI; its operator
 * boundary for this path is the set of duck-typed Python calls the sampler loops make
 * (SURVEY.md §8(b)).  This header is the boundary a maintainer would bind instead (ctypes stub in
 * INTEGRATION.md).  Every entry point names the reference loop it replaces.
 *
 * Conventions
 *   - plain pointers + sizes, no C++/torch types; every function returns a glabc_status (0 = OK);
 *     glabc_last_error(ctx) gives the message of the last failure on that context.
 *   - `*_dev` pointers are CUDA device pointers on the context's device; `*_host` are host pointers
 *     (pinned memory makes the copies asynchronous, pageable memory works too).
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).  Device entry
 *     points only enqueue work; host entry points return when the result is in the host buffers.
 *   - no hidden global state: one context per (thread, device); a context is not thread-safe and it is
 *     single-stream: its scratch buffers (KDE partial sums, resample scans, the host entry points' staging,
 *     the flow's packed operands and training state) are reused by consecutive calls without cross-stream
 *     ordering — issue the calls of one context on ONE stream (or order the streams with events yourself).
 *   - the per-chain statistics (`stats`) are float32 running sums: exact counters up to 2^24 steps per
 *     chain, and moments meant for diagnostics over <= ~1e6 steps; accumulate longer runs on the host in
 *     float64 from per-launch (or per-checkpoint) stats buffers.
 *   - all floating-point parameters are float32 values the host evaluated the way the reference
 *     does (e.g. scale = exp(log_scale) in float32, distribution.py:170), so device code never has to
 *     re-derive a constant with a different libm.
 */
#ifndef GLABC_H
#define GLABC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GLABC_ABI_VERSION 1
#define GLABC_MAX_DIM 8      /* theta_dim and y_dim of a fused model family               */
#define GLABC_MAX_MODES 8    /* GaussianMixture components                                  */
#define GLABC_MAX_K 16       /* iSIR candidates per global move (reference `batch_size`)    */

typedef enum {
    GLABC_OK = 0,
    GLABC_ERR_INVALID = 1,       /* bad argument (message says which)                       */
    GLABC_ERR_UNSUPPORTED = 2,   /* model family / distribution kind / dim not fused        */
    GLABC_ERR_CUDA = 3,          /* a CUDA runtime call failed                              */
    GLABC_ERR_NO_DEVICE = 4      /* no usable CUDA device — there is no CPU fallback        */
} glabc_status;

/* ---- ABC model plugin (reference: examples/Mixture.py:5-53, README.md:66-104) -------------- */
typedef enum {
    /* y = |theta| + noise_loc + noise_scale * eps   (Mixture.py:19-23), y_dim == theta_dim    */
    GLABC_MODEL_ABS_NORMAL = 1,
    /* y = theta + noise_loc + noise_scale * eps     (Gaussian location model)                 */
    GLABC_MODEL_ID_NORMAL = 2
} glabc_model_family;

typedef struct {
    int32_t family;                        /* glabc_model_family                                */
    int32_t theta_dim;
    int32_t y_dim;
    int32_t reserved;
    float y_obs[GLABC_MAX_DIM];            /* Mixture.py:9                                      */
    float noise_loc[GLABC_MAX_DIM];        /* Mixture.py:19 (0)                                 */
    float noise_scale[GLABC_MAX_DIM];      /* exp(log(sqrt(0.05))) in float32, Mixture.py:19    */
    float prior_loc[GLABC_MAX_DIM];        /* Mixture.py:30                                     */
    float prior_log_scale[GLABC_MAX_DIM];
    float prior_scale[GLABC_MAX_DIM];      /* exp(prior_log_scale) in float32                   */
    float eps_log_scale;                   /* log(epsilon) in float32, Mixture.py:43            */
    float eps_scale;                       /* exp(log(epsilon)) in float32 (0.05 -> 0.049999997)*/
    double epsilon;                        /* the Python float `ABCset.epsilon` itself (GLMALA.py:90
                                              uses epsilon**2 in float64)                       */
} glabc_model_t;

/* ---- proposal / prior distributions (reference: distribution.py:50,90,143,206) ------------- */
typedef enum {
    GLABC_DIST_NONE = 0,
    GLABC_DIST_DIAG_GAUSSIAN = 1,          /* distribution.py:143-181                           */
    GLABC_DIST_UNIFORM = 2,                /* distribution.py:50-86                             */
    GLABC_DIST_GAMMA = 3,                  /* distribution.py:90-137                            */
    GLABC_DIST_GAUSSIAN_MIXTURE = 4        /* distribution.py:206-293                           */
} glabc_dist_kind;

typedef struct {
    int32_t kind;                          /* glabc_dist_kind                                   */
    int32_t dim;
    int32_t n_modes;                       /* GaussianMixture only                              */
    int32_t reserved;
    /* DiagGaussian: a = loc, b = log_scale, c = exp(log_scale).
       Uniform:      a = low, b = high,      c[0] = log_prob_val (distribution.py:71).
       Gamma:        a = shape, b = rate.                                                       */
    float a[GLABC_MAX_DIM];
    float b[GLABC_MAX_DIM];
    float c[GLABC_MAX_DIM];
    /* GaussianMixture: loc / log_scale / scale per mode, log of the soft-maxed weights.        */
    float mix_loc[GLABC_MAX_MODES][GLABC_MAX_DIM];
    float mix_log_scale[GLABC_MAX_MODES][GLABC_MAX_DIM];
    float mix_scale[GLABC_MAX_MODES][GLABC_MAX_DIM];
    float mix_log_w[GLABC_MAX_MODES];
    float mix_w[GLABC_MAX_MODES];
} glabc_dist_t;

typedef enum { GLABC_SLOT_LOCAL = 0, GLABC_SLOT_GLOBAL = 1, GLABC_SLOT_IMPORTANCE = 2,
               GLABC_SLOT_COUNT = 3 } glabc_slot;

/* ---- run description -------------------------------------------------------------------- */
typedef enum {
    GLABC_RNG_NATIVE = 0,   /* per-thread Philox4x32-10, counter = (global chain id, step, slot)  */
    GLABC_RNG_REPLAY = 1    /* consume a tape of the reference's own draws (parity mode)          */
} glabc_rng_mode;

typedef enum {
    GLABC_ARITH_FAST = 0,   /* FMA contraction, reciprocal multiplies, MUFU approximations        */
    GLABC_ARITH_STRICT = 1  /* the reference's float32 operation order, IEEE div/sqrt, no FMA     */
} glabc_arith_mode;

typedef enum {
    GLABC_TRACE_NONE = 0,        /* statistics only                                               */
    GLABC_TRACE_TIME_MAJOR = 1,  /* trace[row][chain][d]                                          */
    GLABC_TRACE_CHAIN_MAJOR = 2, /* trace[chain][row][d] — out[c] is a reference-shaped chain,
                                    rows staged through shared memory (GlobalMCMC.py:34,98)       */
    GLABC_TRACE_EVENTS = 3       /* run_global / device buffers only: the chain as its MOVES.  trace[chain][trace_rows][1 + d]:
                                    entry 0 = {number of moves (uint32 bits), -}, entry k >= 1 = {row index (uint32 bits),
                                    theta[d]} of the k-th row whose theta differs from the previous row's (the first row
                                    written always counts).  A chain is piecewise constant — the README workload moves on
                                    1.2 % of its steps — so this is the trace losslessly run-length encoded; moves beyond
                                    trace_rows - 1 are counted but not stored.  The host-buffer entry point uses it to bring
                                    part of the chains back as events and expands them with the host cores.              */
} glabc_trace_layout;

/* Per-chain statistics accumulated in-kernel (replaces the reference's unused `num_acc`,
 * GlobalMCMC.py:33,50,65, and feeds esjd(), ESJD.py:17-24, without re-reading the trace).       */
#define GLABC_STAT_STEPS 0          /* transitions performed                                      */
#define GLABC_STAT_GLOBAL_STEPS 1   /* of which took the global branch                            */
#define GLABC_STAT_ACC_LOCAL 2      /* accepted local moves                                       */
#define GLABC_STAT_ACC_GLOBAL 3     /* accepted / switched global moves                           */
#define GLABC_STAT_SUM 4            /* + i            : sum_t theta_i          (i < d)            */
/*                     4 + d + i          : sum_t theta_i^2                                       */
/*                     4 + 2d + tri(i,j)  : sum_t delta_i delta_j, i <= j (row-major upper tri)   */
#define GLABC_NSTATS(d) (4 + 2 * (d) + ((d) * ((d) + 1)) / 2)

#define GLABC_AUX_SLOTS 8
#define GLABC_AUX_LOGW 0            /* iSIR: cached log-weight of the current state               */
#define GLABC_AUX_LOCAL 1           /* iSIR: 1.0 if a local move was accepted since (init 1.0);
                                       GLMALA never sets it again after the first global move
                                       (GLMALA.py:152-157 vs :195-199), reproduced                */
#define GLABC_AUX_WIDE 2            /* GLMALA: theta / y are float64 tensors (a local move was accepted:
                                       GLMALA.py:43 adds a float64 gradient, SURVEY.md B-5)       */
#define GLABC_AUX_LW_WIDE 3         /* GLMALA: the cached log-weight (hence the iSIR weights) is float64 */
#define GLABC_AUX_HAVE_GRAD 4       /* GLMALA: grad_logABC_Theta_old is not None (GLMALA.py:183)  */

/* GLMALA carried float64 state, state64[C][GLABC_STATE64_SLOTS]                                  */
#define GLABC_STATE64_SLOTS 16
#define GLABC_S64_THETA 0           /* + i, i < d  (used when AUX_WIDE)                           */
#define GLABC_S64_Y 4               /* + i                                                        */
#define GLABC_S64_GRAD 8            /* + i: grad_logABC_Theta_old                                 */
#define GLABC_S64_LOGW 12           /* cached log-weight                                          */

/* Common fields of every sampler launch.  One launch advances `n_chains` independent chains by
 * `n_steps` transitions (loop iterations i = step_base+1 .. step_base+n_steps of the reference's
 * `for i in range(1, num_ite)`), so a run can be cut into time chunks or resumed.                */
typedef struct {
    int64_t n_chains;         /* chains in this launch (this rank's shard)                        */
    int64_t n_steps;          /* transitions to perform                                           */
    int64_t step_base;        /* transitions already performed (0 for a fresh chain)              */
    int64_t chain_id_base;    /* global id of chain 0 of this shard: Philox streams are keyed by
                                 the global id, so traces do not depend on the GPU count          */
    uint64_t seed;
    float global_frequency;   /* compared in float32, strict <  (SURVEY.md B-15)                  */
    int32_t rng_mode;         /* glabc_rng_mode                                                   */
    int32_t arith_mode;       /* glabc_arith_mode                                                 */
    int32_t trace_layout;     /* glabc_trace_layout                                               */
    int32_t write_row0;       /* also store the incoming state as trace row `step_base`           */
    int32_t block_threads;    /* 0 = library default                                              */
    int32_t n_candidates;     /* iSIR K = reference `batch_size` (run_isir / run_mala only)       */
    int32_t num_grad;         /* GLMALA gradient sample count (run_mala only)                     */
    float tau;                /* GLMALA step size (run_mala only)                                 */
    int64_t trace_rows;       /* rows of the full trace buffer (num_ite); row index = step index  */
    int64_t trace_chains;     /* chains of the full trace buffer (>= n_chains)                    */
    int64_t trace_chain_off;  /* first chain of this launch inside the trace buffer               */
    int64_t trace_row_base;   /* step index stored in row 0 of the trace buffer (0 unless the buffer
                                 holds a time chunk of a longer run)                               */
    /* state, updated in place: theta[C][d], y[C][y_dim] (float32)                                */
    float* theta;
    float* y;
    float* aux;               /* [C][GLABC_AUX_SLOTS] sampler-specific carried state (iSIR: cached
                                 log-weight + `local` flag, GLMCMC.py:51-55,60-65), or NULL       */
    float* trace;             /* NULL iff GLABC_TRACE_NONE                                        */
    float* stats;             /* [n_chains][GLABC_NSTATS(d)], accumulated (+=); may be NULL       */
    /* replay mode only */
    const float* tape32;      /* [n_steps][tape_slots][n_chains] float32 draws                    */
    const double* tape64;     /* [n_steps][n_chains] float64 draws (np.random.uniform), or NULL   */
    float* debug;             /* [n_steps][GLABC_DEBUG_SLOTS][n_chains] per-step quantities/NULL  */
    /* native mode only */
    float* tape_dump;         /* [n_steps][tape_slots][n_chains]: the draws the kernel used, in tape
                                 layout, so a replay (or the CPU oracle) can re-run the same chain */
    double* tape64_dump;      /* [n_steps][n_chains]: the float64 resampling uniforms used (iSIR)   */
    /* GLMALA (run_mala) only */
    double* state64;          /* [C][GLABC_STATE64_SLOTS] carried float64 state, updated in place  */
    const float* tape_grad0;  /* replay: [d*num_grad*y_dim][n_chains] draws of the first gradient
                                 (grad_logABC_Theta_old is None, GLMALA.py:183-184)                */
    float* tape_grad0_dump;   /* native: the same, written by the kernel                           */
    double* debug64;          /* [n_steps][GLABC_DEBUG64_SLOTS][n_chains] per-step quantities/NULL */
    double tau64;             /* the Python float `tau` (GLMALA.py:43 uses tau**2/2 in float64 while z*tau
                                 is a float32 product); 0 = use (double)tau                          */
    void* stream;
} glabc_run_t;

/* replay tape slots for run_global: U_b, eps_prop[d], eps_sim[y_dim], U_a  (SURVEY.md A.1)       */
#define GLABC_TAPE_GLOBAL_SLOTS(d, yd) (2 + (d) + (yd))
/* replay tape slots for run_isir: U_b, eps_prop[K][d], eps_sim[K][y_dim], U_a (local); the
 * float64 resampling uniform is in tape64                      (SURVEY.md A.2)                    */
#define GLABC_TAPE_ISIR_SLOTS(d, yd, K) (2 + (K) * ((d) + (yd)))
/* debug slots (float32; slot 0 holds an integer value):
 *   0 flags: bit0 global branch, bit1 state changed, bits 8.. iSIR resample index + 1 (0 = None)
 *   GlobalMCMC / local moves: 1 log prior(theta'), 2 log kernel(y'), 3 log_acc
 *   iSIR global move:         1 log-weight of the current state, 2 sum of the K+1 weights,
 *                             3 normalised weight of the current state, 4+j log-weight of
 *                             candidate j (j < K)                                                 */
#define GLABC_DEBUG_SLOTS (4 + GLABC_MAX_K)
/* replay tape slots for run_mala: the iSIR layout (a local step keeps z[d] in the first proposal slots,
 * eps_sim[y_dim] in the first simulator slots, U_a last) followed by the gradient normals
 * [d][num_grad][y_dim] of theta' (one copy: + and - share them, GLMALA.py:76-83)  (SURVEY.md A.3)  */
#define GLABC_TAPE_MALA_SLOTS(d, yd, K, num) (2 + (K) * ((d) + (yd)) + (d) * (num) * (yd))
/* run_mala debug64 slots (float64): 0 flags (bit0 global, bit1 state changed, bits 8.. resample index + 1,
 *   bit16 float64 weights); MALA local move: 1 log_acc, 2+i theta'[i], 6+i y'[i], 10+i grad'[i] (i < 4),
 *   14 log prior', 15 log kernel', 16 log q(theta|theta'), 17 log q(theta'|theta); the float64 statistics inside the
 *   gradient at theta' (GLMALA.py:86-89): 20+i mu_plus[i], 24+i mu_minus[i], 28+i Sigma_plus[i], 32+i Sigma_minus[i];
 *   iSIR global move: 1 log-weight of the current state, 2 sum of weights, 3 normalised weight of the
 *   current state, 4+j log-weight of candidate j                                                   */
#define GLABC_DEBUG64_SLOTS 36
#define GLABC_MAX_NUM_GRAD 4096

/* ---- AGLMCMC (AGLMCMC.py:44-288) -------------------------------------------------------------
 * Every chain owns a block of B = batch_size * step_size pre-generated importance candidates
 * (theta0, x0, w0, log q0, dis0; AGLMCMC.py:84-112); a global move runs iSIR against the next
 * batch_size of them (:127-162); after step_size global moves the chain adapts (:170-249): eps-hat
 * quantile update, weighted KernelDensity refit on the block, a new block sampled from the KDE.
 * The block / KDE workspace lives inside the context (sized n_chains * B).                          */
typedef enum { GLABC_BW_SILVERMAN = 0, GLABC_BW_SCOTT = 1 } glabc_bw_rule;

#define GLABC_AG_REC_SLOTS 8     /* per adaptation: 0 eps-hat, 1 KDE training points, 2+i bandwidth[i] (i < 4) */
#define GLABC_AG_MAX_BLOCK 4096  /* batch_size * step_size                                                    */

typedef struct {
    int32_t step_size;        /* adaptation period S in global moves (AGLMCMC.py:167)                  */
    int32_t init;             /* 1: start of a run — draw the initial block from the IMPORTANCE slot
                                 (AGLMCMC.py:84-119); 0: continue from the context's workspace          */
    float alpha;              /* AGLMCMC.py:186                                                         */
    float hat_eps_T;          /* AGLMCMC.py:174,196                                                     */
    int32_t kde_rule;         /* glabc_bw_rule; the reference uses 'silverman' (AGLMCMC.py:214)         */
    int32_t tape_rounds;      /* replay: adaptations the tapes hold per chain                           */
    /* replay tapes (the reference's draws), chain-minor like tape32 */
    const float* init_p;      /* [B*d][C]   normals of Initial_ISIR_prop.forward(B)   (AGLMCMC.py:84)  */
    const float* init_s;      /* [B*y][C]   simulator normals of the initial block     (:94)            */
    const int32_t* ad_idx;    /* [R][4B][C] torch.multinomial indices of KDE.sample    (:220)           */
    const float* ad_noise;    /* [R][4B*d][C] KDE.sample normals                                        */
    const float* ad_sim;      /* [R][B*y][C] simulator normals of the new block        (:232)           */
    /* optional dumps for parity tests (any rng mode) */
    float* ad_rec;            /* [R][GLABC_AG_REC_SLOTS][C]                                             */
    float* ad_blk;            /* [R][B][d + 3][C]: theta0[d], log q0, w0, dis0 of the block after adaptation r */
    float* init_w;            /* [B][C] weights of the initial block                                    */
    int32_t dump_rounds;      /* R of ad_rec / ad_blk                                                   */
    int32_t reserved;
} glabc_aglmcmc_t;

/* ---- RealNVP importance proposal of GLMCMC-NFs (GLMCMC_NFs.py:51-61; normflows 1.7 pieces, SURVEY.md App. C) ----
 * n_blocks x [AffineCouplingBlock(MLP([1, hidden, hidden, 2])), Permute(2, 'swap')] over DiagGaussian(2).
 * Weight pointers are DEVICE pointers in torch's nn.Linear layout ([out][in]); glabc_flow_set copies them.   */
typedef struct {
    int32_t n_blocks;            /* 32, GLMCMC_NFs.py:51                                                   */
    int32_t hidden;              /* 128, GLMCMC_NFs.py:56                                                  */
    int32_t dim;                 /* 2                                                                      */
    int32_t reserved;
    const float* w1;             /* [n_blocks][hidden]          Linear(1, hidden).weight                    */
    const float* b1;             /* [n_blocks][hidden]                                                      */
    const float* w2;             /* [n_blocks][hidden][hidden]  Linear(hidden, hidden).weight               */
    const float* b2;             /* [n_blocks][hidden]                                                      */
    const float* w3;             /* [n_blocks][2][hidden]       Linear(hidden, 2).weight (row 0 shift, 1 log-scale) */
    const float* b3;             /* [n_blocks][2]                                                           */
    float base_loc[2];           /* nf.distributions.base.DiagGaussian(2).loc                               */
    float base_log_scale[2];
} glabc_flow_t;

/* ---- block iSIR with an external importance proposal (GLMCMC-NFs, GLMCMC_NFs.py:90-152) --------------------
 * Caller-owned DEVICE buffers: every chain's block of `block` = batch_size * step_size candidates and its counters. */
typedef struct {
    int32_t step_size;        /* S: global moves per block (GLMCMC_NFs.py:111)                              */
    int32_t block;            /* B = batch_size * step_size                                                 */
    float* blk_theta;         /* [C][B][d]  candidates from the proposal (NF_model.sample, :72,127)         */
    float* blk_x;             /* [C][B][y]  their simulations (:80,136)                                     */
    float* blk_w;             /* [C][B]     importance weights (:82-85)                                     */
    float* blk_lq;            /* [C][B]     proposal log-densities                                          */
    int32_t* kk;              /* [C] global moves done in the current block                                 */
    int32_t* pending;         /* [C] out: bit 0 = block consumed (kk == S), bit 1 = needs lq_cur refreshed  */
    uint32_t* next_step;      /* [C] loop index of the next iteration to perform (init step_base + 1)       */
    float* lq_cur;            /* [C] proposal log-density of the current state (NF_model.log_prob, :98)     */
    int32_t* lq_valid;        /* [C] lq_cur is up to date                                                   */
} glabc_block_isir_t;

/* ---- user-supplied model, compiled at run time (SURVEY.md 8(f) n1) ------------------------------------------
 * The plugin surface of the reference is duck-typed Python (`generate_samples / prior_log_prob / discrepancy`,
 * examples/Mixture.py:13-36, README.md:66-104).  A model outside the built-in family is given as CUDA C++ source
 * defining three device functions; the library compiles them (NVRTC, sm_100a) INTO the fused GlobalMCMC step kernel,
 * so the simulator, prior and discrepancy are inlined into the same single kernel as the proposal, the Gaussian ABC
 * kernel (Mixture.py:38-53) and the Metropolis-Hastings test:
 *
 *   __device__ void  glabc_user_simulate(const float* theta, const float* noise, const float* params, float* y);
 *       y[y_dim] <- one simulator draw at theta[theta_dim]; noise[n_noise] are independent N(0,1) draws
 *       (generate_samples, Mixture.py:13-26)
 *   __device__ float glabc_user_prior_log_prob(const float* theta, const float* params);      (Mixture.py:28-31)
 *   __device__ float glabc_user_discrepancy(const float* y, const float* params);             (Mixture.py:33-36)
 *
 * `params` (<= GLABC_USER_MAX_PARAMS floats) carries the model's constants (y_obs, noise scales, ...).            */
#define GLABC_USER_MAX_PARAMS 64
#define GLABC_USER_MAX_NOISE 32
typedef struct {
    int32_t theta_dim;        /* 1..GLABC_MAX_DIM                                                            */
    int32_t y_dim;            /* 1..2*GLABC_MAX_DIM                                                          */
    int32_t n_noise;          /* N(0,1) draws one simulator call consumes, 0..GLABC_USER_MAX_NOISE           */
    int32_t n_params;
    const char* source;       /* NUL-terminated CUDA C++ defining the three functions above                  */
    float params[GLABC_USER_MAX_PARAMS];
    double epsilon;           /* width of the Gaussian ABC kernel (Mixture.py:7,43)                          */
} glabc_user_model_t;

typedef struct glabc_ctx glabc_ctx;

#if defined(__GNUC__)
#define GLABC_API __attribute__((visibility("default")))
#else
#define GLABC_API
#endif

/* ---- lifecycle --------------------------------------------------------------------------- */
GLABC_API int glabc_version(void);
/* device < 0: use the current CUDA device. Fails with GLABC_ERR_NO_DEVICE when no GPU is present. */
GLABC_API int glabc_ctx_create(int device, glabc_ctx** out);
GLABC_API int glabc_ctx_destroy(glabc_ctx* ctx);
GLABC_API const char* glabc_last_error(const glabc_ctx* ctx);
GLABC_API const char* glabc_status_string(int status);
/* multiprocessor count, SM clock (kHz) and the library's default block size, for roofline math   */
GLABC_API int glabc_device_info(const glabc_ctx* ctx, int32_t* sm_count, int32_t* clock_khz, int32_t* cc);

/* ---- plugin binding ------------------------------------------------------------------------ */
/* replaces the `ABCset` argument of every sampler (GlobalMCMC.py:6, GLMCMC.py:24, ...)           */
GLABC_API int glabc_model_set(glabc_ctx* ctx, const glabc_model_t* model, size_t nbytes);
/* replaces Local_Proposal / Global_Proposal / Importance_Proposal (GlobalMCMC.py:6-7,
 * GLMCMC.py:24-25).  dim 1..GLABC_MAX_DIM: the built-in model family runs dim <= 4 (its theta_dim), a user model up to 8. */
GLABC_API int glabc_dist_set(glabc_ctx* ctx, int slot, const glabc_dist_t* dist, size_t nbytes);
/* Prior of the bound model (replaces the DiagGaussian in glabc_model_t's prior_* fields): any glabc_dist_t kind,
 * dim == theta_dim.  NULL restores the model's DiagGaussian.  glabc_model_set clears a bound prior.
 * A DiagGaussian is written into the model's prior_* fields (the same run as giving it in the model POD).  With a Uniform /
 * Gamma / GaussianMixture prior every sampler runs FAST arithmetic with the native RNG: GLABC_ARITH_STRICT, GLABC_RNG_REPLAY,
 * tape_dump and the AGLMCMC parity dumps are refused with GLABC_ERR_UNSUPPORTED.  Outside the prior's support the log prior
 * is -inf: from such a state the first proposal with a finite prior is accepted, a candidate with -inf is never selected.
 * GLABC_ERR_INVALID: no model bound, dim != theta_dim, invalid parameters (the checks of glabc_dist_set);
 * GLABC_ERR_UNSUPPORTED: dim > 4.                                                                                        */
GLABC_API int glabc_model_prior_set(glabc_ctx* ctx, const glabc_dist_t* prior, size_t nbytes);

/* device-side forward() / log_prob() of the distribution bound to `slot` (distribution.py:73-86, 106-137, 166-181,
 * 242-293): z[n][dim] -> log_p[n], and n fresh draws z[n][dim] (+ their log-densities, log_p may be NULL).
 * dim <= 4; a wider distribution (for a user model) is refused with GLABC_ERR_UNSUPPORTED.                            */
GLABC_API int glabc_dist_log_prob(glabc_ctx* ctx, int slot, const float* z, int64_t n, float* log_p, void* stream);
GLABC_API int glabc_dist_sample(glabc_ctx* ctx, int slot, int64_t n, uint64_t seed, float* z, float* log_p, void* stream);

/* ---- samplers: device buffers, asynchronous on `stream` ------------------------------------- */
/* GlobalMCMC loop body, GlobalMCMC.py:37-68 (local RW-MH / global independence-MH mixture).  DiagGaussian proposals
 * in both slots run the tuned kernel (replay + strict arithmetic available); any Uniform / Gamma / GaussianMixture
 * proposal selects the general kernel (float32).  Its replay mode takes the reference's proposal draws themselves:
 * tape32 [n_steps][2 + d][C] = U_b, eps_sim[d], U_a and tape64 [n_steps][d][C] = the draw in float64 (theta' of a global
 * move, the increment of a local one); debug slots 0..3 as for the tuned kernel.
 * A non-Gaussian model prior (glabc_model_prior_set) also selects the general kernel: FAST arithmetic, native RNG.    */
GLABC_API int glabc_run_global(glabc_ctx* ctx, const glabc_run_t* run);

/* GLMCMC loop body, GLMCMC.py:58-104, incl. weight_sampling GLMCMC.py:7-22: iSIR global move with
 * `n_candidates` fresh draws from the IMPORTANCE slot, local RW-MH from the LOCAL slot.  `aux` carries
 * the cached log-weight and the `local` flag (init {0, 1}, GLMCMC.py:49-55).
 * A Uniform / Gamma / GaussianMixture proposal in either slot selects the general kernel; it follows the reference's dtype
 * promotion (after a float64 draw is taken the weights are exponentiated in float64: aux slots GLABC_AUX_WIDE / _LW_WIDE).
 * Its replay mode takes the proposal draws themselves: tape32 [n_steps][2 + K y_dim][C] = U_b, eps_sim[K][y_dim] (a local
 * move: eps_sim[y_dim] first), U_a (last slot); tape64 [n_steps][1 + K d][C] = the float64 resampling uniform, then the draws
 * theta_j (a local move: the increment z in the first d); debug slots as for the tuned kernel, + bit 16 of slot 0 = float64
 * weights.  A non-Gaussian model prior (glabc_model_prior_set) also selects the general kernel: FAST, native RNG.       */
GLABC_API int glabc_run_isir(glabc_ctx* ctx, const glabc_run_t* run);

/* GLMALA loop body, GLMALA.py:150-200: the iSIR global move of run_isir (GLMALA.py:151-180) and a MALA
 * local move (Local_proposal_forward :25-44, log_proposal :97-116) whose drift is the finite-difference
 * synthetic-likelihood gradient numberical_gradient_logABC (:46-95) from 2*d*num_grad simulator draws with
 * common random numbers.  run->tau, run->num_grad, run->n_candidates; needs aux and state64.
 * A Uniform / Gamma / GaussianMixture Importance_Proposal runs in the throughput kernel (GLABC_ARITH_FAST, native RNG, no
 * tape dump; candidates drawn as in glabc_run_isir's general kernel); with GLABC_ARITH_STRICT / GLABC_RNG_REPLAY it is refused
 * with GLABC_ERR_UNSUPPORTED — the replay kernel is fused for a DiagGaussian importance proposal.  The same holds for a
 * non-Gaussian model prior (glabc_model_prior_set), whatever block_threads is.                                          */
GLABC_API int glabc_run_mala(glabc_ctx* ctx, const glabc_run_t* run);

/* AGLMCMC loop body, AGLMCMC.py:124-272.  LOCAL slot = Local_Proposal, IMPORTANCE slot = Initial_ISIR_prop;
 * run->n_candidates = batch_size.  Chains pause individually when they reach an adaptation; the call runs
 * step / adapt rounds until every chain has performed run->n_steps iterations.  Debug slots (float32, `debug`):
 * 0 flags as run_isir; global move: 1 proposal log-density of the current state, 2 its weight, 3 sum of the
 * K+1 weights; local move: as run_global.
 * A Uniform / Gamma / GaussianMixture Initial_ISIR_prop (the initial candidate block, AGLMCMC.py:84-112, and the weight
 * of the current state before the first adaptation, :137-149) is taken with GLABC_ARITH_FAST and the native RNG; STRICT /
 * replay / recording runs and a non-Gaussian Local_Proposal are refused with GLABC_ERR_UNSUPPORTED.  A non-Gaussian model
 * prior (glabc_model_prior_set) runs FAST with the native RNG as well; KDE draws with log prior <= log(1e-10) (outside a
 * Uniform box, say) never enter a block.                                                                                */
GLABC_API int glabc_run_aglmcmc(glabc_ctx* ctx, const glabc_run_t* run, const glabc_aglmcmc_t* ag);

/* GlobalMCMC loop body (GlobalMCMC.py:37-68) for a user-supplied model: LOCAL / GLOBAL slots hold proposals of any
 * glabc_dist_kind and of the model's theta_dim (1..GLABC_MAX_DIM); native RNG, FAST arithmetic; run->theta [C][theta_dim],
 * run->y [C][y_dim]; trace / stats as glabc_run_global.  The first call for a given source and pair of proposal kinds
 * compiles it (about a second); the module is cached for the life of the process.  A compile error is returned as
 * GLABC_ERR_INVALID with the NVRTC log in glabc_last_error.
 * Semantics of the proposals as glabc_run_global's general kernel: a local move is theta + z, z ~ Local_Proposal, with no
 * proposal term in the MH ratio (so an asymmetric Gamma local proposal gives the reference's biased chain); a global move
 * adds log q(theta) - log q(theta').  Two DiagGaussian slots run the fused Gaussian arithmetic; the simulator's noise is
 * drawn from the same random numbers whatever the proposal kinds.                                                     */
GLABC_API int glabc_run_global_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_user_model_t* model);
/* GLMCMC loop body (GLMCMC.py:58-104, weight_sampling :7-22) for a user-supplied model: LOCAL = Local_Proposal, IMPORTANCE =
 * Importance_Proposal (any glabc_dist_kind, as glabc_run_global_user), run->n_candidates = batch_size, run->aux as
 * glabc_run_isir.  The importance weights are exponentiated max-shifted (the reference's un-shifted float32 exp can underflow a
 * whole row to `None`; the shift removes that artefact and nothing else).  log-weight = log prior + log K - log q; a NaN
 * weight counts as 0, a -inf candidate is never selected, and a current state outside the importance proposal's support has
 * log-weight +inf: that global move selects nothing and the chain stays.                                                  */
GLABC_API int glabc_run_isir_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_user_model_t* model);
/* GLMALA (GLMALA.py:150-200) for a user model: IMPORTANCE slot (any glabc_dist_kind, its global move as
 * glabc_run_isir_user), run->n_candidates, run->tau, run->num_grad; aux [C][8] carries
 * the cached log-weight (slot 0), the `local` flag (1), "gradient cached" (2) and the cached gradient (3 ..): theta_dim <= 5.
 * A thread per chain; the finite-difference gradient's draws (GLMALA.py:46-95) are dealt over the warp.                    */
GLABC_API int glabc_run_mala_user(glabc_ctx* ctx, const glabc_run_t* run, const glabc_user_model_t* model);
/* Compile-only check of a user model for compute capability `cc` (100 = sm_100a): needs NVRTC but neither a GPU nor a
 * context.  The NVRTC log (or "" on success) is copied to log[log_cap].  Compiles the kernels for DiagGaussian proposals. */
GLABC_API int glabc_user_model_check(const glabc_user_model_t* model, int32_t cc, char* log, size_t log_cap);
/* The same for the proposal kinds (glabc_dist_kind) a run will bind: local_kind for the LOCAL slot, far_kind for the
 * GLOBAL (glabc_run_global_user) or IMPORTANCE (glabc_run_isir_user, glabc_run_mala_user) slot.  An unknown kind is
 * GLABC_ERR_INVALID.                                                                                                  */
GLABC_API int glabc_user_model_check_proposals(const glabc_user_model_t* model, int32_t local_kind, int32_t far_kind, int32_t cc,
                                               char* log, size_t log_cap);

/* The model's functions outside a run (generate_samples / prior_log_prob / discrepancy / calculate_log_kernel of the plugin
 * surface, Mixture.py:13-53), one row per thread in the kernel glabc_k_eval_user of the same NVRTC module as the step kernels:
 * a module already loaded for the model (any proposal kinds) serves them, otherwise the DiagGaussian one is compiled.
 * DEVICE buffers, asynchronous on `stream`.  n == 0 launches nothing; n < 0, a NULL buffer with n > 0, an invalid model or
 * (glabc_user_evaluate) an unknown op are GLABC_ERR_INVALID, refused before anything is launched.                          */
typedef enum {
    GLABC_USER_SIMULATE = 0,      /* theta[n][theta_dim] -> y[n][y_dim]: the entry glabc_user_simulate below           */
    GLABC_USER_PRIOR = 1,         /* x = theta[n][theta_dim] -> out[n] = glabc_user_prior_log_prob                     */
    GLABC_USER_DISCREPANCY = 2,   /* x = y[n][y_dim]         -> out[n] = glabc_user_discrepancy                         */
    GLABC_USER_LOG_KERNEL = 3     /* x = y[n][y_dim]         -> out[n] = log K(dis) = -0.5 log(2 pi) - log eps - dis^2 / (2 eps^2),
                                     evaluated as the step kernels' kernel term (model->epsilon)                            */
} glabc_user_op;
/* y[n][y_dim] = one simulator draw per row of theta[n][theta_dim].  Row r takes its n_noise N(0,1) draws from the Philox4x32-10
 * blocks with counter (row_base + r, step 0, slot 2 + b), b < ceil(n_noise / 4), key = seed, as Box-Muller pairs -- the
 * numbers a step kernel would draw for its simulator at step 0.  No run draws at step 0 (a launch draws at steps
 * step_base + 1 ..), so with row_base = run->chain_id_base and the run's seed, row c is a simulated initial y of chain c that
 * depends on the chain's global id only, not on the shard that runs it.                                                     */
GLABC_API int glabc_user_simulate(glabc_ctx* ctx, const glabc_user_model_t* model, const float* theta, int64_t n, uint64_t seed,
                                  uint64_t row_base, float* y, void* stream);
/* op = GLABC_USER_PRIOR, GLABC_USER_DISCREPANCY or GLABC_USER_LOG_KERNEL on the n rows of x, out[n] float32.                  */
GLABC_API int glabc_user_evaluate(glabc_ctx* ctx, const glabc_user_model_t* model, int32_t op, const float* x, int64_t n, float* out,
                                  void* stream);

/* ---- KernelDensity (kernel_density.py:4-177), batched over `sets` independent point sets ------------------
 * Set s holds n[s] points X[s][cap][dim] (n == NULL: every set holds `cap` points).                          */
/* fit, kernel_density.py:22-94: weights_out[s][j] = w / sum(w) (uniform when w == NULL),
 * bw_out[s][i] = h(n, dim, rule) * weighted unbiased std of coordinate i                                    */
GLABC_API int glabc_kde_fit(glabc_ctx* ctx, const float* X, const float* w, const int32_t* n, int64_t sets, int64_t cap,
                            int32_t dim, int32_t rule, float* weights_out, float* bw_out, void* stream);
/* log_prob, kernel_density.py:96-128: out[s][q] = logsumexp_j(log N(x[s][q]; X[s][j], diag(bw[s]^2)) + log(w[s][j] + 1e-10))
 * for m queries per set, x[s][m][dim].  arith: glabc_arith_mode.                                             */
GLABC_API int glabc_kde_log_prob(glabc_ctx* ctx, const float* X, const float* weights, const float* bw, const int32_t* n,
                                 int64_t sets, int64_t cap, int32_t dim, const float* x, int64_t m, float* out,
                                 int32_t arith, void* stream);
/* sample, kernel_density.py:130-156: out[s][q] = X[s][idx] + bw[s] * normal, idx ~ Categorical(weights[s]).
 * idx_tape / noise_tape ([s][m] / [s][m][dim], or NULL): replay the reference's torch.multinomial / randn draws. */
GLABC_API int glabc_kde_sample(glabc_ctx* ctx, const float* X, const float* weights, const float* bw, const int32_t* n,
                               int64_t sets, int64_t cap, int32_t dim, int64_t m, uint64_t seed, const int32_t* idx_tape,
                               const float* noise_tape, float* out, void* stream);

/* GLMCMC-NFs loop body, GLMCMC_NFs.py:90-152, ONE pass: every chain advances until it has done run->n_steps
 * iterations, consumed its block (pending bit 0: GLMCMC_NFs.py:111 — train / regenerate) or needs the proposal
 * log-density of a changed state (pending bit 1).  The caller refreshes lq_cur with glabc_flow_log_prob, refills the
 * block with glabc_flow_sample + glabc_block_weights, and calls again.  LOCAL slot = Local_Proposal.             */
GLABC_API int glabc_run_block_isir(glabc_ctx* ctx, const glabc_run_t* run, const glabc_block_isir_t* blk);
/* (a non-Gaussian model prior: FAST arithmetic only, as glabc_run_aglmcmc)                                               */
/* GLMCMC_NFs.py:73-85,129-140: blk_x = simulate(blk_theta), blk_w = exp(prior + log K - blk_lq), NaN -> 0;
 * `round` keys the simulator's Philox normals (run->seed, run->chain_id_base as usual)                           */
GLABC_API int glabc_block_weights(glabc_ctx* ctx, const glabc_run_t* run, const glabc_block_isir_t* blk, uint32_t round);

/* ---- RealNVP flow on the tensor cores (tcgen05 kind::f16, FP32 accumulate in TMEM) --------------------------
 * NormalizingFlow.sample(n) (GLMCMC_NFs.py:72,127): eps[n][2] standard normals in -> theta[n][2], log_q[n];
 * NormalizingFlow.log_prob(x) (GLMCMC_NFs.py:98): theta[n][2] -> log_q[n].  Device pointers.
 * Operand precision of the 128 x 128 hidden layer (glabc_flow_precision, per context):
 *   GLABC_FLOW_PRECISE (default)  FP16 hi + lo split of activations and weights, three MMAs, layers 1 / 3 in FP32: log q and
 *                                 log_prob agree with a float64 evaluation of the reference's float32 network within 1e-5
 *                                 relative (the tolerance north_star states for log-densities);
 *   GLABC_FLOW_FAST               single FP16 operands, one MMA (+ the output layer as a second small MMA): ~3x the samples/s,
 *                                 agreement ~1e-3.  sample() still returns the exact log-density of the map it applied.     */
#define GLABC_FLOW_FAST 0
#define GLABC_FLOW_PRECISE 1
GLABC_API int glabc_flow_precision(glabc_ctx* ctx, int32_t mode);
GLABC_API int glabc_flow_set(glabc_ctx* ctx, const glabc_flow_t* flow, size_t nbytes, void* stream);
GLABC_API int glabc_flow_sample(glabc_ctx* ctx, const float* eps, int64_t n, float* theta, float* log_q, void* stream);
/* the same with the base normals drawn inside the kernel (Philox4x32-10 keyed by `seed`, counter = sample index): no eps buffer */
GLABC_API int glabc_flow_sample_native(glabc_ctx* ctx, uint64_t seed, int64_t n, float* theta, float* log_q, void* stream);
GLABC_API int glabc_flow_log_prob(glabc_ctx* ctx, const float* theta, int64_t n, float* log_q, void* stream);

/* ---- the flow's training step (GLMCMC_NFs.py:63,112-124): loss = NF_model.forward_kld(x) = -mean log q(x), backward through
 * the coupling blocks, torch.optim.Adam(lr, weight_decay).  The context owns the FP32 master parameters (copied in by
 * glabc_flow_set) and the Adam moments.  Flat parameter / gradient layout, P = glabc_flow_param_count(n_blocks) floats:
 *   w1 [L][128] | b1 [L][128] | w2 [L][128][128] | b2 [L][128] | w3 [L][2][128] | b3 [L][2] | base loc [2] | base log_scale [2]
 *   glabc_flow_train_init   (re)starts training: zero moments, step count 0, Adam hyper-parameters (GLMCMC_NFs.py:63: lr 5e-4,
 *                           weight_decay 1e-5; betas 0.9 / 0.999 and eps 1e-8 are torch's defaults)
 *   glabc_flow_grad         x [n][2] (device) -> grad [P] (device; NULL: the context's buffer) = d loss / d parameters, and
 *                           loss [1] (device; NULL: the context's).  A multi-GPU caller all-reduces `grad` (mean) next.
 *   glabc_flow_adam_step    one Adam update of the master parameters from `grad` (NULL: the context's buffer), then the
 *                           kernels' packed weights are refreshed.  Nothing is updated when *loss is NaN / inf: the reference
 *                           skips backward() then (:120-121) and Adam.step() leaves gradient-less parameters untouched.
 *   glabc_flow_train_step   = glabc_flow_grad + glabc_flow_adam_step (single GPU)
 *   glabc_flow_get          the master parameters -> params [P] (device)
 *   glabc_flow_train_state  save (restore = 0) / load (1) the Adam moments state [2 P] = m | v (device) and *step: with
 *                           glabc_flow_get / glabc_flow_set this checkpoints a flow in training                            */
GLABC_API int64_t glabc_flow_param_count(int32_t n_blocks);
GLABC_API int glabc_flow_train_init(glabc_ctx* ctx, float lr, float beta1, float beta2, float eps, float weight_decay);
GLABC_API int glabc_flow_grad(glabc_ctx* ctx, const float* x, int64_t n, float* grad, float* loss, void* stream);
GLABC_API int glabc_flow_adam_step(glabc_ctx* ctx, const float* grad, const float* loss, void* stream);
GLABC_API int glabc_flow_train_step(glabc_ctx* ctx, const float* x, int64_t n, float* loss, void* stream);
GLABC_API int glabc_flow_get(glabc_ctx* ctx, float* params, void* stream);
GLABC_API int glabc_flow_train_state(glabc_ctx* ctx, float* state, int64_t* step, int32_t restore, void* stream);

/* ---- samplers: host buffers (the reference-facing call: H2D state, run, D2H trace + stats) --- */
/* `run->theta`, `y`, `aux`, `state64`, `trace`, `stats` are HOST pointers here; the trace is copied back in
 * `chunk_steps`-row chunks overlapped with the next chunk's kernel (0 = library default).        */
GLABC_API int glabc_run_global_host(glabc_ctx* ctx, const glabc_run_t* run, int64_t chunk_steps);
GLABC_API int glabc_run_isir_host(glabc_ctx* ctx, const glabc_run_t* run, int64_t chunk_steps);
GLABC_API int glabc_run_mala_host(glabc_ctx* ctx, const glabc_run_t* run, int64_t chunk_steps);
/* AGLMCMC.py:124-272 on host buffers: the chains' candidate blocks and KDEs stay in the context's workspace; the run is cut
 * into time chunks (ag->init applies to the first, the others continue) and each chunk's rows travel while the next one runs */
GLABC_API int glabc_run_aglmcmc_host(glabc_ctx* ctx, const glabc_run_t* run, const glabc_aglmcmc_t* ag, int64_t chunk_steps);
/* Checkpoint of glabc_run_aglmcmc's workspace (every chain's block of candidates, its KernelDensity, counters and eps-hat) as an
 * opaque device blob.  restore = 0: blob == NULL returns the size in *bytes, otherwise the workspace is copied out; restore = 1:
 * a workspace for n_chains x block (= batch_size * step_size) is set up from the blob, ready for glabc_run_aglmcmc with
 * ag->init = 0 and run->step_base = the iterations already done (bit-identical continuation).                          */
GLABC_API int glabc_aglmcmc_state(glabc_ctx* ctx, void* blob, int64_t* bytes, int64_t n_chains, int32_t block, int32_t restore,
                                  void* stream);

/* ---- diagnostics --------------------------------------------------------------------------- */
/* esjd(), ESJD.py:2-25, for every chain of a device trace: out[c] = det(D^T D/(N-1))^(1/d).
 * layout = glabc_trace_layout of `trace` ([rows][chains][d] or [chains][rows][d]).                */
GLABC_API int glabc_esjd(glabc_ctx* ctx, const float* trace, int32_t layout, int64_t rows, int64_t chains,
               int32_t dim, float* out, void* stream);

/* HOST-side expansion of a GLABC_TRACE_EVENTS buffer (already copied to host memory) into dense chain-major rows:
 * trace[c][r - row_base][dim] for r = first recorded row .. row_end, chain c's events at events[c][cap][1 + dim].  What the
 * host-buffer entry points do internally (full-line non-temporal stores with AVX-512, n_threads workers, 0 = all cores); a
 * caller that keeps GLABC_TRACE_EVENTS traces on the device can expand them later with this.  No GPU needed.
 * GLABC_ERR_INVALID (nothing written) if a count exceeds cap - 1 or rows are not ascending within [row_base, row_end].   */
GLABC_API int glabc_expand_events(const float* events, int64_t chains, int64_t cap, int32_t dim, int64_t row_base, int64_t row_end,
                                  float* trace, int64_t trace_rows, int32_t n_threads);

/* Additive summary of a shard's per-chain statistics (stats [chains][GLABC_NSTATS(dim)], as the samplers fill them) in one
 * launch: out[6 + 2 dim] float64 += {chains, steps, global steps, accepted local, accepted global, sum over chains of
 * esjd (ESJD.py:21-24 from the Gram accumulators), sum theta[dim], sum theta^2[dim]} — the vector the ranks all-reduce.
 * The caller zeroes `out`.                                                                                              */
GLABC_API int glabc_summarize(glabc_ctx* ctx, const float* stats, int64_t chains, int32_t dim, double* out, void* stream);

/* resample(W, N), GLMCMC_NFs.py:29-40 / AGLMCMC.py:30-41 — systematic resampling of the candidate block by its normalised
 * weights W[n] (device, float32) with the ONE uniform u0 = torch.rand(1) the reference draws: idx[i] (device, int64, i < N) =
 * the index emitted for u_i = (u0 + i) / N, or n when u_i lies at or beyond the last cumulative weight (the reference returns
 * fewer than N indices then; they are always the LAST ones, so idx[0 .. *count) is the reference's list); count (device).   */
GLABC_API int glabc_resample(glabc_ctx* ctx, const float* W, int64_t n, int64_t N, float u0, int64_t* idx, uint64_t* count,
                             void* stream);

/* raw Philox4x32-10 blocks for known-answer tests: out[n][4] = philox(ctr[n][4], key[n][2])       */
GLABC_API int glabc_philox_kat(glabc_ctx* ctx, const uint32_t* ctr, const uint32_t* key, int64_t n,
                     uint32_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GLABC_H */
