// K4-train — the flow's training step of GLMCMC-NFs (GLMCMC_NFs.py:112-124): loss = forward_kld(x) = -mean log q(x) over the
// resampled candidates, backward through the 32 coupling blocks, Adam(lr 5e-4, weight_decay 1e-5) (GLMCMC_NFs.py:63).
//
//   forward   k_flow_pipe_precise<false> (flow_pipe.cuh: log_prob, PRECISE) — log q(x) and the latent z = f^-1(x)
//   backward  k_flow_bwd (this file).  The flow is invertible, so nothing is stored: starting from z the sweep walks the blocks
//             in the order opposite to log_prob's (l = 0 .. L-1), RE-COMPUTES block l's MLP from the block's output, rebuilds the
//             block's input (z2 = z2' e^s + shift), and back-propagates.  Per tile of 128 samples and block, three GEMMs on the
//             tensor cores (tcgen05, M128 N128 K128, FP16 hi + lo split = three MMAs per K step, FP32 accumulate in TMEM):
//                 H2pre = H1 W2^T          A = H1  [sample][i]  K-major   B = W2 [j][i]  K-major
//                 dH1   = dH2 W2           A = dH2 [sample][j]  K-major   B = W2 [j][i]  read MN-major (K = j): the same bytes
//                 dW2  += dH2^T H1         A = dH2 read MN-major (M = j)  B = H1 read MN-major (N = i), K = sample; the
//                                          accumulator stays in TMEM across the CTA's tiles
//             (an operand stored [row][col] in the no-swizzle K-major core-matrix layout IS the MN-major layout of its
//             transpose with LBO and SBO exchanged, so H1 and dH2 are written to shared memory once each).
//             Layers 1 and 3 (K = 1, N = 2), the ReLU masks and the bias / vector gradients run on the CUDA cores; sums over
//             the samples go through a small shared-memory transpose in a fixed order, and every CTA adds into its OWN slice of
//             a partial-gradient buffer which k_flow_grad_reduce folds in CTA order: the step is deterministic.
//   update    k_flow_adam — torch.optim.Adam's arithmetic (weight decay folded into the gradient, bias-corrected moments).
// The backward sweep carries the adjoints unscaled (d loss / d log q = -1 per sample); the 1 / n of the mean is applied by the
// reduction.  FP16 operands are written saturating (an adjoint beyond 65504 clips instead of becoming inf).
#pragma once
#include "flow.cuh"
#include "flow_param_layout.h"

namespace glabc {

constexpr int kTrThreads = 128;                 // one thread per sample row = TMEM lane
constexpr int kTrTiles = 4;                     // tiles per chunk (512 samples share one fetch of W2)
constexpr int kTrOpBytes = kFlowHidden * kFlowHidden * 2;   // one 128 x 128 FP16 operand: 32 KB
constexpr int kTrScratchCols = 16;
// shared memory: W2 hi/lo | H1 hi/lo | X hi/lo (H2-derived: dH2) | vectors | state | scratch | small gradients | barriers
constexpr int kTrVecFloats = 5 * kFlowHidden + 8;                        // w1 b1 b2 w3[0] w3[1] b3
constexpr int kTrStateFloats = 4 * kTrTiles * kFlowTile;                 // z1 z2' g1 g2'
constexpr int kTrScratchFloats = kFlowTile * (kTrScratchCols + 1) + 2 * kFlowTile;   // [128][17] + dshift / ds per sample
constexpr int kTrGradFloats = 5 * kFlowHidden + 8;                       // dw1 db1 db2 dw3[0] dw3[1] db3
constexpr int kTrSmemBytes = 6 * kTrOpBytes + 4 * (kTrVecFloats + kTrStateFloats + kTrScratchFloats + kTrGradFloats) + 64;

// saturating FP16 hi / lo split of two floats, packed (lo element in bits 0..15)
__device__ __forceinline__ void split_pack(float a, float b, uint32_t& hi, uint32_t& lo)
{
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
    const float2 f = unpack_half2(hi);
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(b - f.y), "f"(a - f.x));
}

// the three MMAs of one split-precision GEMM: (A_hi + A_lo)(B_hi + B_lo) without the lo x lo term.
// a_step / b_step: byte advance of the operand per K = 16 step (256 for a K-major view, 4096 for an MN-major view)
__device__ __forceinline__ void gemm_split(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, bool a_mn, bool b_mn,
                                           uint32_t idesc, bool accumulate)
{
    const uint32_t a_step = a_mn ? 4096u : 256u, b_step = b_mn ? 4096u : 256u;
    const uint32_t a_lbo = a_mn ? 2048u : 128u, a_sbo = a_mn ? 128u : 2048u;
    const uint32_t b_lbo = b_mn ? 2048u : 128u, b_sbo = b_mn ? 128u : 2048u;
#pragma unroll 1
    for (int term = 0; term < 3; ++term) {
        const uint32_t a0 = term == 1 ? a_lo : a_hi, b0 = term == 2 ? b_lo : b_hi;
#pragma unroll
        for (int k = 0; k < kFlowHidden / 16; ++k)
            umma_f16_ss(tmem_d, umma_desc(a0 + k * a_step, a_lbo, a_sbo), umma_desc(b0 + k * b_step, b_lbo, b_sbo), idesc,
                        (accumulate || term > 0 || k > 0) ? 1u : 0u);
    }
}

// row r's 128 values -> FP16 hi / lo, 8 columns (one 16-byte core-matrix row) at a time
__device__ __forceinline__ void store_op8(uint8_t* hi_base, uint8_t* lo_base, int row, int col0, const float (&v)[8])
{
    uint4 h, l;
    split_pack(v[0], v[1], h.x, l.x);
    split_pack(v[2], v[3], h.y, l.y);
    split_pack(v[4], v[5], h.z, l.z);
    split_pack(v[6], v[7], h.w, l.w);
    const uint32_t off = (static_cast<uint32_t>(row) >> 3) * 2048u + (static_cast<uint32_t>(col0) >> 3) * 128u + (static_cast<uint32_t>(row) & 7u) * 16u;
    *reinterpret_cast<uint4*>(hi_base + off) = h;
    *reinterpret_cast<uint4*>(lo_base + off) = l;
}

// Column sums over the 128 sample rows, fixed order: thread (q = tid / 32, c = tid % 32) adds rows 32 q .. 32 q + 31 of column c,
// then thread c (< ncols) folds the four quarter sums.  scratch: [128][kTrScratchCols + 1] values, part: [4][kTrScratchCols].
// `weight` (per row, or nullptr) multiplies the value.  Call with ALL threads; the result lands in acc[col0 + c] (+=) by thread c.

__global__ void __launch_bounds__(kTrThreads, 1) k_flow_bwd(const __grid_constant__ FlowDev W, const float* __restrict__ z_final, int64_t n,
                                                             float* __restrict__ partial)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sW2h = smem;
    uint8_t* sW2l = smem + kTrOpBytes;
    uint8_t* sH1h = smem + 2 * kTrOpBytes;
    uint8_t* sH1l = smem + 3 * kTrOpBytes;
    uint8_t* sXh = smem + 4 * kTrOpBytes;
    uint8_t* sXl = smem + 5 * kTrOpBytes;
    float* sVec = reinterpret_cast<float*>(smem + 6 * kTrOpBytes);   // w1 | b1 | b2 | w3[0] | w3[1] | b3[2]
    float* sState = sVec + kTrVecFloats;                              // [4][tiles][128]: z1, z2', g1, g2'
    float* sScr = sState + kTrStateFloats;                            // [128][17]
    float* sDp = sScr + kFlowTile * (kTrScratchCols + 1);             // [2][128]: dshift, ds of the tile's samples
    float* sGrad = sDp + 2 * kFlowTile;                               // dw1 | db1 | db2 | dw3[0] | dw3[1] | db3[2] (+ base: 4)
    uint64_t* bars = reinterpret_cast<uint64_t*>(sGrad + kTrGradFloats);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = W.n_blocks;
    const FlowParamLayout P(L);
    float* mine = partial + static_cast<int64_t>(blockIdx.x) * ((P.total + 3) & ~int64_t(3));   // this CTA's slice (16-byte aligned)
    constexpr int TS = kTrTiles * kFlowTile;
    const uint32_t bar_w = smem_u32(&bars[0]), bar_m = smem_u32(&bars[1]);

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        mbar_init(bar_w, 1);
        mbar_init(bar_m, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_a = *tmem_slot;            // columns 0..127: H2pre, then dH1
    const uint32_t tmem_w = tmem_a + 128u;         // columns 128..255: dW2 of the current block, summed over the chunk's tiles
    const uint32_t trow = static_cast<uint32_t>(warp * 32) << 16;   // this warp's TMEM lanes
    constexpr uint32_t idesc = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);   // F32 accumulate, F16 x F16, N = M = 128
    uint32_t ph_w = 0, ph_m = 0;
    const float sig0 = expf(W.base_log_scale[0]), sig1 = expf(W.base_log_scale[1]);
    const int64_t n_chunks = (n + TS - 1) / TS;

    // column sums of sScr[128][ncols] (optionally each row times wrow[row]) into acc[0 .. ncols), fixed order
    auto colsum = [&](float* acc, const float* wrow, int ncols) {
        __syncthreads();   // sScr written
        // 128 threads = 4 row-quarters x 32: with ncols <= 16, threads c >= ncols idle in the first phase
        const int q = tid >> 5, c = lane;
        float s = 0.0f;
        if (c < ncols) {
#pragma unroll 8
            for (int r = 0; r < 32; ++r) {
                const int row = q * 32 + r;
                const float v = sScr[row * (kTrScratchCols + 1) + c];
                s += wrow != nullptr ? v * wrow[row] : v;
            }
        }
        // fold the four quarters in order through shuffles is not possible across warps: park them behind the tile
        __syncthreads();   // everyone has read sScr
        if (c < ncols) sScr[q * (kTrScratchCols + 1) + c] = s;
        __syncthreads();
        if (tid < ncols)
            acc[tid] += ((sScr[tid] + sScr[(kTrScratchCols + 1) + tid]) + sScr[2 * (kTrScratchCols + 1) + tid]) + sScr[3 * (kTrScratchCols + 1) + tid];
        __syncthreads();
    };

    for (int64_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        // ---- the chunk's latent states and the adjoints of the base density ----
        float bl0 = 0.0f, bl1 = 0.0f, bs0 = 0.0f, bs1 = 0.0f;   // this thread's share of d loc, d log_scale
        for (int t = 0; t < kTrTiles; ++t) {
            const int64_t idx = (chunk * kTrTiles + t) * kFlowTile + tid;
            float a = 0.0f, b = 0.0f, g0 = 0.0f, g1 = 0.0f;
            if (idx < n) {
                a = z_final[idx * 2];
                b = z_final[idx * 2 + 1];
                const float r0 = (a - W.base_loc[0]) / sig0, r1 = (b - W.base_loc[1]) / sig1;
                g0 = r0 / sig0;          // d(-log p) / dz = r / sigma
                g1 = r1 / sig1;
                bl0 -= g0;               // d(-log p) / d loc = -r / sigma
                bl1 -= g1;
                bs0 += 1.0f - r0 * r0;   // d(-log p) / d log_scale = 1 - r^2
                bs1 += 1.0f - r1 * r1;
            }
            sState[0 * TS + t * kFlowTile + tid] = a;
            sState[1 * TS + t * kFlowTile + tid] = b;
            sState[2 * TS + t * kFlowTile + tid] = g0;
            sState[3 * TS + t * kFlowTile + tid] = g1;
        }
        {   // base-density gradients of the chunk: four column sums over the 128 threads
            for (int i = tid; i < kTrGradFloats; i += kTrThreads) sGrad[i] = 0.0f;
            sScr[tid * (kTrScratchCols + 1) + 0] = bl0;
            sScr[tid * (kTrScratchCols + 1) + 1] = bl1;
            sScr[tid * (kTrScratchCols + 1) + 2] = bs0;
            sScr[tid * (kTrScratchCols + 1) + 3] = bs1;
            colsum(sGrad + 5 * kFlowHidden + 2, nullptr, 4);
            if (tid < 2) mine[P.loc + tid] += sGrad[5 * kFlowHidden + 2 + tid];
            else if (tid < 4) mine[P.log_scale + tid - 2] += sGrad[5 * kFlowHidden + 2 + tid];
        }
        int tiles = 0;
        for (int t = 0; t < kTrTiles; ++t)
            if ((chunk * kTrTiles + t) * kFlowTile < n) tiles = t + 1;

        for (int l = 0; l < L; ++l) {   // log_prob applied block L-1 first and block 0 last: the sweep undoes 0 first
            __syncthreads();
            if (tid == 0) {
                mbar_expect_tx(bar_w, 2 * kTrOpBytes);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    bulk_g2s(smem_u32(sW2h) + q * (kTrOpBytes / 4), reinterpret_cast<const uint8_t*>(W.w2p) + static_cast<int64_t>(l) * kTrOpBytes + q * (kTrOpBytes / 4),
                             kTrOpBytes / 4, bar_w);
                    bulk_g2s(smem_u32(sW2l) + q * (kTrOpBytes / 4), reinterpret_cast<const uint8_t*>(W.w2p_lo) + static_cast<int64_t>(l) * kTrOpBytes + q * (kTrOpBytes / 4),
                             kTrOpBytes / 4, bar_w);
                }
            }
            sVec[tid] = W.w1[l * kFlowHidden + tid];
            sVec[128 + tid] = W.b1[l * kFlowHidden + tid];
            sVec[256 + tid] = W.b2[l * kFlowHidden + tid];
            sVec[384 + tid] = W.w3[(l * 2) * kFlowHidden + tid];
            sVec[512 + tid] = W.w3[(l * 2 + 1) * kFlowHidden + tid];
            if (tid < 2) sVec[640 + tid] = W.b3[l * 2 + tid];
            for (int i = tid; i < kTrGradFloats; i += kTrThreads) sGrad[i] = 0.0f;
            __syncthreads();
            mbar_wait(bar_w, ph_w);
            ph_w ^= 1u;

            for (int t = 0; t < tiles; ++t) {
                const bool valid = (chunk * kTrTiles + t) * kFlowTile + tid < n;
                const float z1 = sState[0 * TS + t * kFlowTile + tid], z2o = sState[1 * TS + t * kFlowTile + tid];
                const float g1 = sState[2 * TS + t * kFlowTile + tid], g2o = sState[3 * TS + t * kFlowTile + tid];
                // ---- layer 1 (FP32) -> H1 operand ----
#pragma unroll 2
                for (int c = 0; c < kFlowHidden; c += 8) {
                    float h[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) h[j] = fmaxf(fmaf(sVec[c + j], z1, sVec[128 + c + j]), 0.0f);
                    store_op8(sH1h, sH1l, tid, c, h);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                tc_fence_before();
                __syncthreads();
                if (tid == 0) {   // H2pre = H1 W2^T
                    tc_fence_after();
                    gemm_split(tmem_a, smem_u32(sH1h), smem_u32(sH1l), smem_u32(sW2h), smem_u32(sW2l), false, false, idesc, false);
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_m) : "memory");
                }
                mbar_wait(bar_m, ph_m);
                ph_m ^= 1u;
                tc_fence_after();
                // ---- layer 3 (N = 2, FP32): shift, log-scale; the block's input; the adjoint of (shift, s) ----
                float p0 = 0.0f, p1 = 0.0f;
#pragma unroll 1
                for (int c = 0; c < kFlowHidden; c += 32) {
                    uint32_t v[32];
                    tmem_ld32(tmem_a + trow + c, v);
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float h2 = fmaxf(__uint_as_float(v[j]) + sVec[256 + c + j], 0.0f);
                        p0 = fmaf(h2, sVec[384 + c + j], p0);
                        p1 = fmaf(h2, sVec[512 + c + j], p1);
                    }
                }
                const float shift = p0 + sVec[640], s = p1 + sVec[641];
                const float es = expf(s), ems = expf(-s);
                const float z2 = fmaf(z2o, es, shift);                       // the block's input: z2' = (z2 - shift) e^-s
                const float dshift = valid ? -g2o * ems : 0.0f;
                const float ds = valid ? fmaf(-g2o, z2o, 1.0f) : 0.0f;       // dz2'/ds = -z2';  log q -= s and d loss / d log q = -1
                const float dz2 = g2o * ems;
                sDp[tid] = dshift;
                sDp[kFlowTile + tid] = ds;
                // db3: two column sums
                sScr[tid * (kTrScratchCols + 1) + 0] = dshift;
                sScr[tid * (kTrScratchCols + 1) + 1] = ds;
                colsum(sGrad + 5 * kFlowHidden, nullptr, 2);
                // ---- dH2 = (dshift w3[0] + ds w3[1]) [H2pre + b2 > 0] -> X operand; dW3 and db2 as column sums ----
#pragma unroll 1
                for (int c = 0; c < kFlowHidden; c += kTrScratchCols) {
                    uint32_t v[16];
                    tmem_ld16_async(tmem_a + trow + c, v);
                    tmem_ld_wait();
                    float h2[16], d2[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        h2[j] = fmaxf(__uint_as_float(v[j]) + sVec[256 + c + j], 0.0f);
                        d2[j] = h2[j] > 0.0f ? fmaf(dshift, sVec[384 + c + j], ds * sVec[512 + c + j]) : 0.0f;
                    }
                    {
                        float a8[8], b8[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) { a8[j] = d2[j]; b8[j] = d2[8 + j]; }
                        store_op8(sXh, sXl, tid, c, a8);
                        store_op8(sXh, sXl, tid, c + 8, b8);
                    }
#pragma unroll
                    for (int j = 0; j < 16; ++j) sScr[tid * (kTrScratchCols + 1) + j] = h2[j];
                    colsum(sGrad + 3 * kFlowHidden + c, sDp, kTrScratchCols);                 // dw3[0][j] += sum_s dshift[s] h2[s][j]
#pragma unroll
                    for (int j = 0; j < 16; ++j) sScr[tid * (kTrScratchCols + 1) + j] = h2[j];
                    colsum(sGrad + 4 * kFlowHidden + c, sDp + kFlowTile, kTrScratchCols);     // dw3[1][j] += sum_s ds[s] h2[s][j]
#pragma unroll
                    for (int j = 0; j < 16; ++j) sScr[tid * (kTrScratchCols + 1) + j] = d2[j];
                    colsum(sGrad + 2 * kFlowHidden + c, nullptr, kTrScratchCols);             // db2[j] += sum_s dh2[s][j]
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                tc_fence_before();
                __syncthreads();
                if (tid == 0) {
                    tc_fence_after();
                    // dH1 = dH2 W2 (B read MN-major: K = j) and dW2 += dH2^T H1 (both read MN-major: K = sample)
                    gemm_split(tmem_a, smem_u32(sXh), smem_u32(sXl), smem_u32(sW2h), smem_u32(sW2l), false, true, idesc | (1u << 16), false);
                    gemm_split(tmem_w, smem_u32(sXh), smem_u32(sXl), smem_u32(sH1h), smem_u32(sH1l), true, true, idesc | (1u << 15) | (1u << 16), t > 0);
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_m) : "memory");
                }
                mbar_wait(bar_m, ph_m);
                ph_m ^= 1u;
                tc_fence_after();
                // ---- dH1 masked by layer 1's ReLU: d z1, d w1, d b1 ----
                float dz1 = 0.0f;
#pragma unroll 1
                for (int c = 0; c < kFlowHidden; c += kTrScratchCols) {
                    uint32_t v[16];
                    tmem_ld16_async(tmem_a + trow + c, v);
                    tmem_ld_wait();
                    float d1[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const bool on = fmaf(sVec[c + j], z1, sVec[128 + c + j]) > 0.0f;
                        d1[j] = on ? __uint_as_float(v[j]) : 0.0f;
                        dz1 = fmaf(d1[j], sVec[c + j], dz1);
                    }
#pragma unroll
                    for (int j = 0; j < 16; ++j) sScr[tid * (kTrScratchCols + 1) + j] = d1[j];
                    colsum(sGrad + 1 * kFlowHidden + c, nullptr, kTrScratchCols);                             // db1
#pragma unroll
                    for (int j = 0; j < 16; ++j) sScr[tid * (kTrScratchCols + 1) + j] = d1[j];
                    colsum(sGrad + 0 * kFlowHidden + c, sState + 0 * TS + t * kFlowTile, kTrScratchCols);     // dw1 += sum_s dh1 z1
                }
                // ---- the block's inputs become the next block's outputs (Permute(swap) undone) ----
                sState[0 * TS + t * kFlowTile + tid] = z2;
                sState[1 * TS + t * kFlowTile + tid] = z1;
                sState[2 * TS + t * kFlowTile + tid] = dz2;
                sState[3 * TS + t * kFlowTile + tid] = g1 + dz1;
                tc_fence_before();
                __syncthreads();   // TMEM columns, operand buffers and sScr are free for the next tile
            }
            // ---- block l's gradients of this chunk into the CTA's slice ----
            if (tiles > 0) {
                tc_fence_after();
                float* dst = mine + P.w2 + (static_cast<int64_t>(l) * kFlowHidden + tid) * kFlowHidden;   // row j = tid of dW2[l]
#pragma unroll 1
                for (int c = 0; c < kFlowHidden; c += 32) {
                    uint32_t v[32];
                    tmem_ld32(tmem_w + trow + c, v);
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float4 o = *reinterpret_cast<float4*>(dst + c + j);
                        o.x += __uint_as_float(v[j]); o.y += __uint_as_float(v[j + 1]); o.z += __uint_as_float(v[j + 2]); o.w += __uint_as_float(v[j + 3]);
                        *reinterpret_cast<float4*>(dst + c + j) = o;
                    }
                }
                mine[P.w1 + l * kFlowHidden + tid] += sGrad[tid];
                mine[P.b1 + l * kFlowHidden + tid] += sGrad[128 + tid];
                mine[P.b2 + l * kFlowHidden + tid] += sGrad[256 + tid];
                mine[P.w3 + (l * 2) * kFlowHidden + tid] += sGrad[384 + tid];
                mine[P.w3 + (l * 2 + 1) * kFlowHidden + tid] += sGrad[512 + tid];
                if (tid < 2) mine[P.b3 + l * 2 + tid] += sGrad[640 + tid];
                tc_fence_before();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_slot), "r"(256u) : "memory");
}

// grad[p] = (1 / n) sum over the CTAs' slices in CTA order;  loss = -(1 / n) sum log q  (one block folds the log-densities)
static __global__ void __launch_bounds__(256) k_flow_grad_reduce(const float* __restrict__ partial, int n_slices, int64_t total, float inv_n,
                                                                 float* __restrict__ grad)
{
    const int64_t p = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p >= total) return;
    float s = 0.0f;
    const int64_t stride = (total + 3) & ~int64_t(3);
    for (int c = 0; c < n_slices; ++c) s += partial[static_cast<int64_t>(c) * stride + p];
    grad[p] = s * inv_n;
}

static __global__ void __launch_bounds__(1024) k_flow_loss(const float* __restrict__ lq, int64_t n, float* __restrict__ loss)
{
    // forward_kld = -mean(log q): float64 partials per thread, fixed-order tree
    __shared__ double part[1024];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) s += static_cast<double>(lq[i]);
    part[threadIdx.x] = s;
    __syncthreads();
    for (int off = 512; off > 0; off >>= 1) {
        if (threadIdx.x < off) part[threadIdx.x] += part[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) *loss = static_cast<float>(-part[0] / static_cast<double>(n));
}

// torch.optim.Adam (amsgrad = False): g += wd p; m = b1 m + (1 - b1) g; v = b2 v + (1 - b2) g^2;
// p -= (lr / (1 - b1^t)) m / (sqrt(v) / sqrt(1 - b2^t) + eps).  Skipped as a whole when the loss is not finite: the reference
// skips backward() then (GLMCMC_NFs.py:120-121) and Adam.step() leaves parameters without a gradient untouched.
static __global__ void __launch_bounds__(256) k_flow_adam(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v,
                                                          const float* __restrict__ g, int64_t total, const float* __restrict__ loss, float lr,
                                                          float beta1, float beta2, float eps, float wd, float bc1, float bc2_sqrt)
{
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    if (loss != nullptr && !isfinite(*loss)) return;
    const float pi = p[i];
    const float gi = fmaf(wd, pi, g[i]);
    const float mi = fmaf(beta1, m[i], (1.0f - beta1) * gi);
    const float vi = fmaf(beta2, v[i], (1.0f - beta2) * gi * gi);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
}

}  // namespace glabc
