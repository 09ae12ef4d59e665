// K4's forward kernels: sample() and log_prob() of the RealNVP flow (flow.cuh) as warp-specialised pipelines, k_flow_pipe
// (GLABC_FLOW_FAST) and k_flow_pipe_precise (GLABC_FLOW_PRECISE, further down).  DESIGN.md K4 has the measurements for
// which this layout replaced round 1's kernel, whose two thread groups each walked a tile through every phase in lock-step.
//
// The PHASES own the warps and the tiles of 128 samples flow past them:
//   * warps 16, 17        M1: wait on mbarriers and issue the hidden layer's tcgen05.mma for alternate tiles (one warp gets
//                            through its waits while the other's MMAs are in the tensor pipe's queue), commit to mbarriers,
//                            and prefetch the next coupling block's operands (W2 32 KB + a pre-packed 9 KB blob of w1 / b1 /
//                            b2 / W3 / b3, k_flow_pack_aux) with cp.async.bulk into the other half of a double buffer — no
//                            CTA-wide barrier and no staging code between coupling blocks;
//   * warp 18             M2: the output layer's MMAs;
//   * warps 8..15          Y: chunk input / output; layer 1 of every tile (HFMA2 -> A operand in TMEM), computed BEFORE the
//                            wait for the operand buffer so that only the tcgen05.st sits behind it;
//   * warps 4..7           E: the hidden layer's epilogue: accumulator -> ReLU -> FP16 pairs, written back into the slot;
//   * warps 0..3           U: (shift, log-scale) read-back and the affine update of the chain state in shared memory.
// What the measurements behind this layout say (profiles/micro/mma_cost.cu, B200):
//   * a tcgen05.mma issued by ONE diverged thread costs ~45 cycles of issue (the compiler's elect / R2UR.BROADCAST sequence
//     per instruction); issued by an elected lane of a CONVERGED warp with its operands prepared outside the branch, M128
//     N128 K16 runs at 64 cycles and M128 N16 K16 (A in TMEM) at 11.5 — the issuing warps therefore run their loops
//     converged (elect_one) — and the same N16 MMA with A in shared memory takes 39 cycles;
//   * b2 is added by the tensor cores: the accumulator of a tile is started by one extra K = 16 MMA of a constant operand
//     (ones in k = 0, 1) against [b2_hi, b2_lo, 0 ...] (both from shared memory): no bias loads or adds in the epilogue;
//   * the output layer (M128 N16 K128, eight K = 16 MMAs) goes into four independent 16-column accumulators (two MMAs
//     each), which the update sums;
//   * the same contraction on the CUDA cores (FFMA2) made the epilogue the bottleneck (7.2e8 samples/s against 1.2e9);
//   * Y is the critical role (layer 1: 64 HFMA2 per thread and tile): its w1 stays in registers across a block's tiles.
// TMEM (512 columns): three 128-column accumulator slots and two 64-column layer-1 operand buffers.  The epilogue writes
// the packed activations back INTO its accumulator slot (columns 0..63, each thread behind its own reads) and the
// output-layer MMAs put their partial sums into the same slot (columns 64..127), so the layer-1 buffer of a tile is free as
// soon as its first MMA completes and three tiles are in flight instead of two.
// Synchronisation is mbarriers only (full / empty pairs per resource, one state barrier per tile of the chunk); the two
// M1 warps and M2 interleave in the tensor pipe's queue in arrival order.
#pragma once
#include "flow.cuh"

namespace glabc {

constexpr int kPipeThreads = 19 * 32;
constexpr int kPipeSlots = 3;        // accumulator slots
constexpr int kPipeMinTiles = 2;
// per coupling block, pre-packed in global memory: [W3 as a 16 x 128 FP16 UMMA operand 4096][w1 FP16 pairs 256][b1 FP16 pairs 256]
// [b3 fp32 8 + pad 120][b2 as a 128 x 16 FP16 UMMA operand: k = 0 FP16(b2), k = 1 FP16(b2 - FP16(b2)), 4096]
constexpr int kAuxW1 = 4096, kAuxB1 = 4352, kAuxB3 = 4608, kAuxB2Op = 4736;
constexpr int kAuxFastBytes = kAuxB2Op + 4096;   // what the FAST kernel stages per coupling block
// ... followed by the PRECISE kernel's FP32 vectors: [W3 fp32 [2][128] 1024][w1 fp32 512][b1 fp32 512]; it stages [b3 .. end)
constexpr int kAuxW3F = kAuxFastBytes, kAuxW1F = kAuxW3F + 1024, kAuxB1F = kAuxW1F + 512;
constexpr int kAuxPreciseOff = kAuxB3, kAuxPreciseBytes = kFlowAuxBytes - kAuxPreciseOff;
static_assert(kAuxB1F + 512 == kFlowAuxBytes && kAuxPreciseBytes % 16 == 0 && kAuxPreciseOff % 16 == 0, "aux blob layout");
constexpr int kPipeOnesBytes = 4096;   // the constant A operand of the bias MMA: 128 x 16 FP16, ones in k = 0, 1
constexpr int kPipeStateFloats = 3 * kFlowTilesPerCta * kFlowTile;
constexpr int kPipeBars = 20 + kFlowTilesPerCta;
constexpr int kPipeSmemBytes = 2 * kFlowW2Bytes + 2 * kAuxFastBytes + kPipeOnesBytes + kPipeStateFloats * 4 + kPipeBars * 8 + 16;
enum : int { kBarWFull = 0, kBarAuxEmpty = 2, kBarA1Full = 4, kBarA1Empty = 6, kBarAccFull = 8, kBarActFull = 11, kBarOutFull = 14, kBarAccEmpty = 17, kBarStateFull = 20 };

static __global__ void __launch_bounds__(256) k_flow_pack_aux(const float* __restrict__ w1, const float* __restrict__ b1,
                                                              const float* __restrict__ b2, const float* __restrict__ w3,
                                                              const float* __restrict__ b3, uint8_t* __restrict__ aux)
{
    const int l = blockIdx.x, tid = threadIdx.x;
    uint8_t* a = aux + static_cast<size_t>(l) * kFlowAuxBytes;
    for (int i = tid; i < kFlowAuxBytes / 4; i += 256) reinterpret_cast<uint32_t*>(a)[i] = 0u;
    __syncthreads();
    {   // element (n, k) of the 16 x 128 K-major operand: rows 0 (shift) and 1 (log-scale), rows 2..15 zero
        const int n = tid >> 7, k = tid & 127;
        reinterpret_cast<__half*>(a)[((k >> 3) * 128 + n * 16 + (k & 7) * 2) / 2] = __float2half_rn(w3[(l * 2 + n) * kFlowHidden + k]);
    }
    if (tid < 64) reinterpret_cast<uint32_t*>(a + kAuxW1)[tid] = pack_half2(w1[l * kFlowHidden + 2 * tid], w1[l * kFlowHidden + 2 * tid + 1]);
    else if (tid < 128) reinterpret_cast<uint32_t*>(a + kAuxB1)[tid - 64] = pack_half2(b1[l * kFlowHidden + 2 * (tid - 64)], b1[l * kFlowHidden + 2 * (tid - 64) + 1]);
    else {   // row n of the bias operand (K-major core matrices, 8-row groups 256 B apart): k = 0 hi, k = 1 lo
        const int nn = tid - 128;
        const float v = b2[l * kFlowHidden + nn];
        const __half hi = __float2half_rn(v);
        __half* row = reinterpret_cast<__half*>(a + kAuxB2Op + (nn >> 3) * 256 + (nn & 7) * 16);
        row[0] = hi;
        row[1] = __float2half_rn(v - __half2float(hi));
    }
    if (tid < 2) reinterpret_cast<float*>(a + kAuxB3)[tid] = b3[l * 2 + tid];
    reinterpret_cast<float*>(a + kAuxW3F)[tid] = w3[l * 2 * kFlowHidden + tid];   // rows 0 (shift) and 1 (log-scale)
    if (tid < 128) reinterpret_cast<float*>(a + kAuxW1F)[tid] = w1[l * kFlowHidden + tid];
    else reinterpret_cast<float*>(a + kAuxB1F)[tid - 128] = b1[l * kFlowHidden + tid - 128];
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// shared-space loads by 32-bit address (a generic pointer into dynamic shared memory costs an S2R + LEA per use)
__device__ __forceinline__ float lds_f32(uint32_t a)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }

// keep a computed address in its register: without this the compiler re-derives shared-window addresses at every use
// (S2R SR_CgaCtaId + LEA, ~20 cycles of latency in front of each mbarrier wait)
__device__ __forceinline__ uint32_t opaque(uint32_t v)
{
    asm volatile("" : "+r"(v));
    return v;
}

// ring position of a running counter: index q % N and the parity of q / N, advanced without a division
template <int N>
struct Ring {
    uint32_t idx = 0, par = 0;
    __device__ __forceinline__ void next()
    {
        if (++idx == N) {
            idx = 0;
            par ^= 1u;
        }
    }
};

#ifdef GLABC_FLOW_TRACE
static __device__ long long g_pipe_trace[6][64][6];   // [role M1 (both threads) / U (warp 0) / Y (warp 8) / Y (warp 12) / M2 / E (warp 4)][step][stamp]
#define GLABC_PTR(role, step, i)                                                          \
    do {                                                                                  \
        if (blockIdx.x == 0 && lane == 0 && (step) >= 256 && (step) < 320) g_pipe_trace[role][(step)-256][i] = clock64(); \
    } while (0)
#else
#define GLABC_PTR(role, step, i)
#endif

__device__ __forceinline__ void tmem_ld32_async(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        :
        : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
          "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_ld2_async(uint32_t taddr, uint32_t& r0, uint32_t& r1)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(taddr) : "memory");
}

__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi)
{
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ uint64_t pack_u32x2(uint32_t lo, uint32_t hi)
{
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
    return r;
}
__device__ __forceinline__ float2 unpack_f32x2(uint64_t v)
{
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
// d += a * b on both fp32 lanes of a register pair (FFMA2)
__device__ __forceinline__ void ffma2(uint64_t& d, uint64_t a, uint64_t b)
{
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
}

template <bool SAMPLE>
__global__ void __launch_bounds__(kPipeThreads, 1) k_flow_pipe(const __grid_constant__ FlowDev W, const float* __restrict__ in, int64_t n,
                                                               float* __restrict__ out_theta, float* __restrict__ out_lq, int tpc)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sAux = smem + 2 * kFlowW2Bytes;
    uint8_t* sOnes = sAux + 2 * kAuxFastBytes;
    float* sState = reinterpret_cast<float*>(sOnes + kPipeOnesBytes);   // [3][tiles][128]: z1, z2, log q
    uint64_t* bars = reinterpret_cast<uint64_t*>(sState + kPipeStateFloats);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kPipeBars);
    // the warp index as a value the compiler knows to be warp-uniform (a broadcast from lane 0, as CUTLASS's
    // canonical_warp_idx_sync): the role branches become uniform branches (PRECISE: 4.3e8 -> 4.6e8 samples/s)
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    constexpr int TS = kFlowTilesPerCta * kFlowTile;
    const int T = tpc, L = W.n_blocks;
    const int64_t n_chunks = (n + static_cast<int64_t>(T) * kFlowTile - 1) / (static_cast<int64_t>(T) * kFlowTile);
    const int my_chunks = blockIdx.x < n_chunks ? static_cast<int>((n_chunks - 1 - blockIdx.x) / gridDim.x) + 1 : 0;
    const uint32_t bar0 = opaque(smem_u32(bars));
    auto bar = [&](int i) { return bar0 + 8u * static_cast<uint32_t>(i); };

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar(kBarWFull + i), 1);
            mbar_init(bar(kBarAuxEmpty + i), 384);
            mbar_init(bar(kBarA1Full + i), 256);
            mbar_init(bar(kBarA1Empty + i), 1);
        }
        for (int i = 0; i < kPipeSlots; ++i) {
            mbar_init(bar(kBarAccFull + i), 1);
            mbar_init(bar(kBarActFull + i), 128);
            mbar_init(bar(kBarOutFull + i), 1);
            mbar_init(bar(kBarAccEmpty + i), 128);
        }
        for (int i = 0; i < kFlowTilesPerCta; ++i) mbar_init(bar(kBarStateFull + i), 128);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // the bias MMA's constant A operand: element (r, k) = (k < 2), K-major core matrices, 8-row groups 256 B apart
    for (int i = tid; i < kPipeOnesBytes / 4; i += kPipeThreads) {
        const int byte = i * 4, in_row = byte & 15, kb = (byte >> 7) & 1;   // 16-byte rows: 8 halves; second core matrix: k = 8..15
        reinterpret_cast<uint32_t*>(sOnes)[i] = (kb == 0 && in_row == 0) ? 0x3C003C00u : 0u;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = opaque(*tmem_slot);    // accumulator slot s: columns 128 s ..; layer-1 operand buffer b: columns 384 + 64 b ..
    const uint32_t tmem_a1 = tmem + 384u;
    const float c2 = -1.8378770664093453f;       // -0.5 * 2 * log(2 pi)

    if (warp == 16 || warp == 17) {
        // ------------------------------------------------ M1: hidden-layer MMAs + operand prefetch ------------------------------------------------
        // two issuing threads, even and odd steps: while one sits in the tensor pipe's queue the other gets through its waits
        {
            const bool lead = elect_one();
            const uint32_t mine = static_cast<uint32_t>(warp - 16);
            constexpr uint32_t idesc = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);     // D = F32, A = B = F16, K-major, N = 128, M = 128
            const uint32_t sW2_addr = smem_u32(smem), sAux_addr = smem_u32(sAux);
            const uint64_t ones_desc = umma_desc(smem_u32(sOnes), 128, 256);
            const int total_blocks = my_chunks * L;
            auto load_block = [&](int gb) {   // coupling block gb of this CTA's sequence -> buffer gb & 1
                const int li = gb % L, l = SAMPLE ? li : L - 1 - li;
                const uint32_t b = static_cast<uint32_t>(gb & 1), full = bar(kBarWFull + (gb & 1));
                if (!lead) return;
                mbar_expect_tx(full, kFlowW2Bytes + kAuxFastBytes);
#pragma unroll
                for (int qd = 0; qd < 4; ++qd)
                    bulk_g2s(sW2_addr + b * kFlowW2Bytes + qd * (kFlowW2Bytes / 4),
                             reinterpret_cast<const uint8_t*>(W.w2p) + static_cast<int64_t>(l) * kFlowW2Bytes + qd * (kFlowW2Bytes / 4),
                             kFlowW2Bytes / 4, full);
                bulk_g2s(sAux_addr + b * kAuxFastBytes, W.aux + static_cast<int64_t>(l) * kFlowAuxBytes, kAuxFastBytes, full);
            };
            if (mine == 0 && total_blocks > 0) load_block(0);
            const int kload = T - 1 < 4 ? T - 1 : 4;
            Ring<2> a1;            // layer-1 operand buffer of step q
            Ring<kPipeSlots> sl;   // accumulator slot of step q
            int gb = 0, gb_seen = -1;
            uint32_t q = 0;
            for (int c = 0; c < my_chunks; ++c) {
                int t = 0;
                for (int s = 0; s < L * T; ++s, ++q) {
                    if ((q & 1u) == mine) {
                        GLABC_PTR(0, q, 0);
                        if (gb != gb_seen) {
                            mbar_wait(bar(kBarWFull + (gb & 1)), (gb >> 1) & 1);
                            gb_seen = gb;
                        }
                        mbar_wait(bar(kBarA1Full + a1.idx), a1.par);
                        GLABC_PTR(0, q, 1);
                        mbar_wait(bar(kBarAccEmpty + sl.idx), sl.par ^ 1u);
                        GLABC_PTR(0, q, 2);
                        tc_fence_after();
                        const uint32_t d = tmem + sl.idx * 128u, a = tmem_a1 + a1.idx * 64u;
                        const uint32_t wb = sW2_addr + static_cast<uint32_t>(gb & 1) * kFlowW2Bytes;
                        const uint64_t b2_desc = umma_desc(sAux_addr + static_cast<uint32_t>(gb & 1) * kAuxFastBytes + kAuxB2Op, 128, 256);
                        const uint64_t w2_desc = umma_desc(wb, 128, 2048);
                        const uint32_t bar_acc = bar(kBarAccFull + sl.idx), bar_a1 = bar(kBarA1Empty + a1.idx);
                        if (lead) {
                            // accumulator = b2 (ones x [b2_hi, b2_lo]), then += A W2^T
                            umma_f16_ss(d, ones_desc, b2_desc, idesc, 0u);
#pragma unroll
                            for (int k = 0; k < kFlowHidden / 16; ++k)
                                umma_f16_ts(d, a + k * 8, w2_desc + static_cast<uint64_t>(k * (256 >> 4)), idesc, 1u);   // the descriptor's address field: 16-byte units
                            umma_commit(bar_acc);
                            umma_commit(bar_a1);
                        }
                        __syncwarp();
                        GLABC_PTR(0, q, 3);
                        if (t == kload && gb + 1 < total_blocks) {   // block gb - 1 has drained: its buffer takes block gb + 1
                            if (gb >= 1) mbar_wait(bar(kBarAuxEmpty + ((gb - 1) & 1)), ((gb - 1) >> 1) & 1);
                            load_block(gb + 1);
                        }
                    }
                    a1.next();
                    sl.next();
                    if (++t == T) {
                        t = 0;
                        ++gb;
                    }
                }
            }
        }
    } else if (warp == 18) {
        // ------------------------------------------------ M2: output-layer MMAs ------------------------------------------------
        {
            const bool lead = elect_one();
            constexpr uint32_t idesc3 = (1u << 4) | ((16u >> 3) << 17) | ((128u >> 4) << 24);     // N = 16
            const uint32_t sAux_addr = smem_u32(sAux);
            Ring<kPipeSlots> sl;
            int gb = 0;
            [[maybe_unused]] int qs = 0;
            for (int c = 0; c < my_chunks; ++c) {
                int t = 0;
                for (int s = 0; s < L * T; ++s) {
                    GLABC_PTR(4, qs, 0);
                    if (t == 0) mbar_wait(bar(kBarWFull + (gb & 1)), (gb >> 1) & 1);
                    mbar_wait(bar(kBarActFull + sl.idx), sl.par);
                    GLABC_PTR(4, qs, 1);
                    tc_fence_after();
                    // activations: the slot's columns 0..63; K step k accumulates into partial sum k & 3 (columns 64 + 16 (k & 3) ..)
                    const uint32_t d = tmem + sl.idx * 128u;
                    const uint32_t w3b = sAux_addr + static_cast<uint32_t>(gb & 1) * kAuxFastBytes;
                    const uint64_t w3_desc = umma_desc(w3b, 128, 2048);
                    const uint32_t bar_out = bar(kBarOutFull + sl.idx);
                    if (lead) {
#pragma unroll
                        for (int k = 0; k < kFlowHidden / 16; ++k)
                            umma_f16_ts(d + 64u + static_cast<uint32_t>(k & 3) * 16u, d + k * 8,
                                        w3_desc + static_cast<uint64_t>(k * (256 >> 4)), idesc3, k >= 4 ? 1u : 0u);
                        umma_commit(bar_out);
                    }
                    __syncwarp();
                    GLABC_PTR(4, qs, 2);
                    sl.next();
                    if (++t == T) {
                        t = 0;
                        ++gb;
                    }
                    ++qs;
                }
            }
        }
    } else if (warp < 4) {
        // ------------------------------------------------ U: (shift, log-scale) read-back and the state update ------------------------------------------------
        const int quad = warp & 3, row = quad * 32 + lane;
        const uint32_t sState_addr = opaque(smem_u32(sState)), sAux_addr = opaque(smem_u32(sAux));
        const uint32_t lanebits = static_cast<uint32_t>(quad * 32) << 16;
        Ring<kPipeSlots> sl;
        int gb = 0;
        [[maybe_unused]] int qs = 0;
        for (int c = 0; c < my_chunks; ++c) {
            int t = 0;
            for (int s = 0; s < L * T; ++s, ++qs) {
                if (warp == 0) GLABC_PTR(1, qs, 0);
                mbar_wait(bar(kBarOutFull + sl.idx), sl.par);   // (this coupling block's operands are resident: its MMAs have run)
                if (warp == 0) GLABC_PTR(1, qs, 1);
                tc_fence_after();
                uint32_t p[8];   // four partial (shift, log-scale) sums: columns 64, 80, 96, 112 of the slot
                const uint32_t o = tmem + sl.idx * 128u + lanebits;
                tmem_ld2_async(o + 64u, p[0], p[1]);
                tmem_ld2_async(o + 80u, p[2], p[3]);
                tmem_ld2_async(o + 96u, p[4], p[5]);
                tmem_ld2_async(o + 112u, p[6], p[7]);
                // (the chain state after the wait: in a chunk's first coupling block it is Y's input, ordered by the barrier chain)
                const uint32_t st = sState_addr + static_cast<uint32_t>((t * kFlowTile + row) * 4);
                const uint32_t b3 = sAux_addr + static_cast<uint32_t>((gb & 1) * kAuxFastBytes + kAuxB3);
                float z1 = lds_f32(st), z2 = lds_f32(st + TS * 4), lq = lds_f32(st + 2 * TS * 4);
                const float b30 = lds_f32(b3), b31 = lds_f32(b3 + 4);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(bar(kBarAccEmpty + sl.idx));
                const float s0 = (__uint_as_float(p[0]) + __uint_as_float(p[2])) + (__uint_as_float(p[4]) + __uint_as_float(p[6]));
                const float s1 = (__uint_as_float(p[1]) + __uint_as_float(p[3])) + (__uint_as_float(p[5]) + __uint_as_float(p[7]));
                if (!SAMPLE) {  // Permute(swap)^-1 precedes the coupling's inverse
                    const float tmp = z1;
                    z1 = z2;
                    z2 = tmp;
                }
                const float sh = s0 + b30;  // shift     = param[:, 0::2]
                const float sc = s1 + b31;  // log-scale = param[:, 1::2]
                lq -= sc;   // log q -= log det (forward) / += log det of the inverse = -s
                if (SAMPLE) {
                    sts_f32(st, fmaf(z2, expf(sc), sh));  // z2 * exp(s) + shift, then Permute(swap)
                    sts_f32(st + TS * 4, z1);
                } else {
                    sts_f32(st, z1);
                    sts_f32(st + TS * 4, (z2 - sh) * expf(-sc));     // the coupling's inverse
                }
                sts_f32(st + 2 * TS * 4, lq);
                mbar_arrive(bar(kBarStateFull + t));   // Y: layer 1 of this tile in the next coupling block / the chunk's output
                if (warp == 0) GLABC_PTR(1, qs, 2);
                sl.next();
                if (++t == T) {   // b3 of this coupling block is behind this thread
                    t = 0;
                    mbar_arrive(bar(kBarAuxEmpty + (gb & 1)));
                    ++gb;
                }
            }
        }
    } else if (warp < 8) {
        // ------------------------------------------------ E: hidden-layer epilogue ------------------------------------------------
        const int quad = warp & 3;
        const uint32_t lanebits = static_cast<uint32_t>(quad * 32) << 16;
        Ring<kPipeSlots> sl;
        [[maybe_unused]] int qs = 0;
        for (int c = 0; c < my_chunks; ++c) {
            for (int s = 0; s < L * T; ++s, ++qs) {
                if (warp == 4) GLABC_PTR(5, qs, 0);
                mbar_wait(bar(kBarAccFull + sl.idx), sl.par);
                if (warp == 4) GLABC_PTR(5, qs, 1);
                tc_fence_after();
                // this row's 128 accumulator columns (b2 already added) -> ReLU -> 64 packed FP16 pairs, written back over columns
                // 0..63 — round r reads columns 32 r .. and writes 16 r .., always behind its own reads
                const uint32_t trow = tmem + sl.idx * 128u + lanebits;
                uint32_t v[2][32], hp[16];
                tmem_ld32_async(trow, v[0]);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    tmem_ld_wait();
                    if (r + 1 < 4) tmem_ld32_async(trow + (r + 1) * 32, v[(r + 1) & 1]);
                    const uint32_t* vv = v[r & 1];
#pragma unroll
                    for (int j = 0; j < 16; ++j) hp[j] = relu_pack_f16(__uint_as_float(vv[2 * j]), __uint_as_float(vv[2 * j + 1]));
                    tmem_st16(trow + r * 16, hp);
                }
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                tc_fence_before();
                mbar_arrive(bar(kBarActFull + sl.idx));
                if (warp == 4) GLABC_PTR(5, qs, 2);
                sl.next();
            }
        }
    } else {
        // ------------------------------------------------ Y: chunk input / output, layer 1 ------------------------------------------------
        const int w = warp - 8, quad = w & 3, half = w >> 2, row = quad * 32 + lane, ytid = tid - 256;
        const uint32_t lanebits = static_cast<uint32_t>(quad * 32) << 16;
        auto y_sync = [] { asm volatile("bar.sync 1, 256;" ::: "memory"); };
        const uint32_t sState_addr = opaque(smem_u32(sState)), sAux_addr = opaque(smem_u32(sAux));
        Ring<2> a1;
        int gb = 0;
        uint32_t wreg[32];   // w1 of this thread's 64 hidden units as FP16 pairs, reloaded once per coupling block
        for (int c = 0; c < my_chunks; ++c) {
            const int64_t chunk = blockIdx.x + static_cast<int64_t>(c) * gridDim.x;
            for (int r = ytid; r < T * kFlowTile; r += 256) {
                const int64_t idx = chunk * T * kFlowTile + r;
                float a = 0.0f, b = 0.0f, lq = 0.0f;
                if (idx < n) {
                    if (SAMPLE && in == nullptr) {   // q0's normals generated here (GLMCMC_NFs.py:72,127)
                        const RoundKeys rk = expand_key(make_uint2(W.seed_lo, W.seed_hi));
                        const uint4 wd = philox4x32_10(make_uint4(static_cast<uint32_t>(idx), static_cast<uint32_t>(idx >> 32), 0u, kSlotFlowEps), rk);
                        box_muller(wd.x, wd.y, a, b);
                    } else {
                        a = in[idx * 2];
                        b = in[idx * 2 + 1];
                    }
                    if (SAMPLE) {  // base DiagGaussian.forward: z = loc + exp(log_scale) * eps, log p from eps
                        lq = c2 - ((W.base_log_scale[0] + 0.5f * (a * a)) + (W.base_log_scale[1] + 0.5f * (b * b)));
                        a = W.base_loc[0] + expf(W.base_log_scale[0]) * a;
                        b = W.base_loc[1] + expf(W.base_log_scale[1]) * b;
                    }
                }
                sState[0 * TS + r] = a;
                sState[1 * TS + r] = b;
                sState[2 * TS + r] = lq;
            }
            y_sync();
            int t = 0;
            const int gb0 = gb;
            [[maybe_unused]] int qs = c * (L * T);
            for (int s = 0; s < L * T; ++s, ++qs) {
                if ((w & 3) == 0) GLABC_PTR(2 + half, qs, 0);
                {   // layer 1 (K = 1) of this step's tile: this thread's 64 hidden units -> 32 packed columns of the A operand
                    if (t == 0) {   // a new coupling block: its operands have landed; this thread's 64 units of w1 stay in registers
                        mbar_wait(bar(kBarWFull + (gb & 1)), (gb >> 1) & 1);
                        const uint32_t w1h = sAux_addr + static_cast<uint32_t>((gb & 1) * kAuxFastBytes + kAuxW1 + half * 128);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const uint4 ww = lds_v4(w1h + j * 16);
                            wreg[4 * j] = ww.x; wreg[4 * j + 1] = ww.y; wreg[4 * j + 2] = ww.z; wreg[4 * j + 3] = ww.w;
                        }
                    }
                    if (gb != gb0) mbar_wait(bar(kBarStateFull + t), (gb - 1) & 1);   // U has updated this tile in the previous coupling block
                    // the arithmetic needs no TMEM: it runs BEFORE the wait for the operand buffer, which leaves only the store behind it
                    const float z1 = lds_f32(sState_addr + static_cast<uint32_t>(((SAMPLE ? 0 : 1) * TS + t * kFlowTile + row) * 4));   // !SAMPLE: Permute(swap)^-1 precedes the inverse
                    // z1 as an FP16 hi + lo pair: rounding the INPUT to 11 bits would perturb all 128 hidden units coherently (the
                    // error of the block would be the network's derivative times 5e-4 |z1|); the roundings left are per-unit
                    const float z_hi = __half2float(__float2half_rn(z1));
                    const uint32_t zz = pack_half2(z_hi, z_hi), zl = pack_half2(z1 - z_hi, z1 - z_hi);
                    const uint32_t b1h = sAux_addr + static_cast<uint32_t>((gb & 1) * kAuxFastBytes + kAuxB1 + half * 128);
                    uint32_t hv[32];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint4 bb = lds_v4(b1h + j * 16);
                        hv[4 * j] = hfma2_relu(wreg[4 * j], zz, hfma2(wreg[4 * j], zl, bb.x));
                        hv[4 * j + 1] = hfma2_relu(wreg[4 * j + 1], zz, hfma2(wreg[4 * j + 1], zl, bb.y));
                        hv[4 * j + 2] = hfma2_relu(wreg[4 * j + 2], zz, hfma2(wreg[4 * j + 2], zl, bb.z));
                        hv[4 * j + 3] = hfma2_relu(wreg[4 * j + 3], zz, hfma2(wreg[4 * j + 3], zl, bb.w));
                    }
                    mbar_wait(bar(kBarA1Empty + a1.idx), a1.par ^ 1u);
                    if ((w & 3) == 0) GLABC_PTR(2 + half, qs, 1);
                    tc_fence_after();
                    tmem_st32(tmem_a1 + a1.idx * 64u + lanebits + half * 32, hv);
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                    tc_fence_before();
                    mbar_arrive(bar(kBarA1Full + a1.idx));
                    if ((w & 3) == 0) GLABC_PTR(2 + half, qs, 2);
                    a1.next();
                    if (++t == T) {   // w1 / b1 of this coupling block are behind this thread
                        t = 0;
                        mbar_arrive(bar(kBarAuxEmpty + (gb & 1)));
                        ++gb;
                    }
                }
            }
            for (int tt = 0; tt < T; ++tt) mbar_wait(bar(kBarStateFull + tt), (gb - 1) & 1);   // the last coupling block's updates
            for (int r = ytid; r < T * kFlowTile; r += 256) {
                const int64_t idx = chunk * T * kFlowTile + r;
                if (idx >= n) continue;
                const float a = sState[0 * TS + r], b = sState[1 * TS + r];
                float lq = sState[2 * TS + r];
                if (SAMPLE) {
                    out_theta[idx * 2] = a;
                    out_theta[idx * 2 + 1] = b;
                } else {  // + base.log_prob(z)
                    if (out_theta != nullptr) {   // the latent z = f^-1(x)
                        out_theta[idx * 2] = a;
                        out_theta[idx * 2 + 1] = b;
                    }
                    const float r0 = (a - W.base_loc[0]) / expf(W.base_log_scale[0]);
                    const float r1 = (b - W.base_loc[1]) / expf(W.base_log_scale[1]);
                    lq += c2 - ((W.base_log_scale[0] + 0.5f * (r0 * r0)) + (W.base_log_scale[1] + 0.5f * (r1 * r1)));
                }
                out_lq[idx] = lq;
            }
            y_sync();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------------
// GLABC_FLOW_PRECISE on the same pipeline (split precision: A = A_hi + A_lo, W2 = W_hi + W_lo as FP16 pairs, three MMAs per
// K step — flow.cuh).  A tile needs 128 accumulator + 64 + 64 operand columns, so two tiles are in flight (TMEM: slot s =
// columns 256 s ..: accumulator, A_hi, A_lo) and the tensor pipe's 25 MMAs per tile (1,600 cycles) set the pace; layers 1 and
// 3 stay FP32 on the CUDA cores:
//   * warps 16, 17  M1: bias MMA + 8 x (A_hi W_hi, A_lo W_hi, A_hi W_lo) for alternate tiles; operand prefetch (W_hi, W_lo 64 KB +
//                       the blob's FP32 part) into a double buffer;
//   * warps 8..15    Y: chunk input / output; FP32 layer 1, FP16 hi / lo split of every activation -> TMEM;
//   * warps 0..7     E: accumulator -> ReLU -> FP32 contraction with the two rows of W3 (FFMA2), the two halves of a row meet
//                       in shared memory, then the affine update of the chain state (half 0).
constexpr int kPipePSlots = 2;
constexpr int kPipeParts = 4;          // ring of partial-sum buffers between the two halves of a row
constexpr int kPipePBars = 16 + kFlowTilesPerCta;
constexpr int kPipePSmemBytes = 2 * 2 * kFlowW2Bytes + 2 * kAuxPreciseBytes + kPipeOnesBytes + kPipeStateFloats * 4 + kPipeParts * kFlowTile * 8 +
                                kPipePBars * 8 + 16;
static_assert(kPipePSmemBytes <= 232448, "shared memory of the PRECISE pipeline");
enum : int { kPBarWFull = 0, kPBarAuxEmpty = 2, kPBarA1Full = 4, kPBarA1Empty = 6, kPBarAccFull = 8, kPBarAccEmpty = 10, kPBarPartFull = 12,
             kPBarStateFull = 16 };

template <bool SAMPLE>
__global__ void __launch_bounds__(18 * 32, 1) k_flow_pipe_precise(const __grid_constant__ FlowDev W, const float* __restrict__ in, int64_t n,
                                                                  float* __restrict__ out_theta, float* __restrict__ out_lq, int tpc)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sAux = smem + 4 * kFlowW2Bytes;                      // [2][W_hi 32 KB | W_lo 32 KB] precede
    uint8_t* sOnes = sAux + 2 * kAuxPreciseBytes;
    float* sState = reinterpret_cast<float*>(sOnes + kPipeOnesBytes);   // [3][tiles][128]: z1, z2, log q
    float2* sPart = reinterpret_cast<float2*>(sState + kPipeStateFloats);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sPart + kPipeParts * kFlowTile);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kPipePBars);
    // the warp index as a value the compiler knows to be warp-uniform (a broadcast from lane 0, as CUTLASS's
    // canonical_warp_idx_sync): the role branches become uniform branches (PRECISE: 4.3e8 -> 4.6e8 samples/s)
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    constexpr int TS = kFlowTilesPerCta * kFlowTile;
    const int T = tpc, L = W.n_blocks;
    const int64_t n_chunks = (n + static_cast<int64_t>(T) * kFlowTile - 1) / (static_cast<int64_t>(T) * kFlowTile);
    const int my_chunks = blockIdx.x < n_chunks ? static_cast<int>((n_chunks - 1 - blockIdx.x) / gridDim.x) + 1 : 0;
    const uint32_t bar0 = opaque(smem_u32(bars));
    auto bar = [&](int i) { return bar0 + 8u * static_cast<uint32_t>(i); };
    // offsets inside the staged part of a block's blob
    constexpr int oB3 = kAuxB3 - kAuxPreciseOff, oB2Op = kAuxB2Op - kAuxPreciseOff, oW3 = kAuxW3F - kAuxPreciseOff,
                  oW1 = kAuxW1F - kAuxPreciseOff, oB1 = kAuxB1F - kAuxPreciseOff;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar(kPBarWFull + i), 1);
            mbar_init(bar(kPBarAuxEmpty + i), 512);
            mbar_init(bar(kPBarA1Full + i), 256);
            mbar_init(bar(kPBarA1Empty + i), 1);
            mbar_init(bar(kPBarAccFull + i), 1);
            mbar_init(bar(kPBarAccEmpty + i), 256);
        }
        for (int i = 0; i < kPipeParts; ++i) mbar_init(bar(kPBarPartFull + i), 128);
        for (int i = 0; i < kFlowTilesPerCta; ++i) mbar_init(bar(kPBarStateFull + i), 128);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < kPipeOnesBytes / 4; i += 18 * 32) {
        const int byte = i * 4, in_row = byte & 15, kb = (byte >> 7) & 1;
        reinterpret_cast<uint32_t*>(sOnes)[i] = (kb == 0 && in_row == 0) ? 0x3C003C00u : 0u;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = opaque(*tmem_slot);
    const float c2 = -1.8378770664093453f;       // -0.5 * 2 * log(2 pi)
    const uint32_t sState_addr = opaque(smem_u32(sState)), sAux_addr = opaque(smem_u32(sAux));

    if (warp == 16 || warp == 17) {
        // ------------------------------------------------ M1 ------------------------------------------------
        const bool lead = elect_one();
        const uint32_t mine = static_cast<uint32_t>(warp - 16);
        constexpr uint32_t idesc = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
        const uint32_t sW_addr = smem_u32(smem);
        const uint64_t ones_desc = umma_desc(smem_u32(sOnes), 128, 256);
        const int total_blocks = my_chunks * L;
        auto load_block = [&](int gb) {
            const int li = gb % L, l = SAMPLE ? li : L - 1 - li;
            const uint32_t b = static_cast<uint32_t>(gb & 1), full = bar(kPBarWFull + (gb & 1));
            if (!lead) return;
            mbar_expect_tx(full, 2 * kFlowW2Bytes + kAuxPreciseBytes);
#pragma unroll
            for (int qd = 0; qd < 4; ++qd) {
                bulk_g2s(sW_addr + b * 2 * kFlowW2Bytes + qd * (kFlowW2Bytes / 4),
                         reinterpret_cast<const uint8_t*>(W.w2p) + static_cast<int64_t>(l) * kFlowW2Bytes + qd * (kFlowW2Bytes / 4), kFlowW2Bytes / 4, full);
                bulk_g2s(sW_addr + b * 2 * kFlowW2Bytes + kFlowW2Bytes + qd * (kFlowW2Bytes / 4),
                         reinterpret_cast<const uint8_t*>(W.w2p_lo) + static_cast<int64_t>(l) * kFlowW2Bytes + qd * (kFlowW2Bytes / 4), kFlowW2Bytes / 4, full);
            }
            bulk_g2s(sAux_addr + b * kAuxPreciseBytes, W.aux + static_cast<int64_t>(l) * kFlowAuxBytes + kAuxPreciseOff, kAuxPreciseBytes, full);
        };
        if (mine == 0 && total_blocks > 0) load_block(0);
        const int kload = T - 1 < 2 ? T - 1 : 2;
        uint32_t par = 0;   // this warp's slot (= mine) has been used `uses` times: parity of uses
        int gb = 0, gb_seen = -1;
        uint32_t q = 0;
        for (int c = 0; c < my_chunks; ++c) {
            int t = 0;
            for (int s = 0; s < L * T; ++s, ++q) {
                if ((q & 1u) == mine) {
                    if (gb != gb_seen) {
                        mbar_wait(bar(kPBarWFull + (gb & 1)), (gb >> 1) & 1);
                        gb_seen = gb;
                    }
                    mbar_wait(bar(kPBarA1Full + mine), par);
                    mbar_wait(bar(kPBarAccEmpty + mine), par ^ 1u);
                    tc_fence_after();
                    const uint32_t d = tmem + mine * 256u, a_hi = d + 128u, a_lo = d + 192u;
                    const uint32_t wb = sW_addr + static_cast<uint32_t>(gb & 1) * 2 * kFlowW2Bytes;
                    const uint64_t b2_desc = umma_desc(sAux_addr + static_cast<uint32_t>(gb & 1) * kAuxPreciseBytes + oB2Op, 128, 256);
                    const uint64_t wh_desc = umma_desc(wb, 128, 2048), wl_desc = umma_desc(wb + kFlowW2Bytes, 128, 2048);
                    const uint32_t bar_acc = bar(kPBarAccFull + mine), bar_a1 = bar(kPBarA1Empty + mine);
                    if (lead) {
                        umma_f16_ss(d, ones_desc, b2_desc, idesc, 0u);   // accumulator = b2
#pragma unroll
                        for (int k = 0; k < kFlowHidden / 16; ++k) umma_f16_ts(d, a_hi + k * 8, wh_desc + static_cast<uint64_t>(k * 16), idesc, 1u);
#pragma unroll
                        for (int k = 0; k < kFlowHidden / 16; ++k) umma_f16_ts(d, a_lo + k * 8, wh_desc + static_cast<uint64_t>(k * 16), idesc, 1u);
#pragma unroll
                        for (int k = 0; k < kFlowHidden / 16; ++k) umma_f16_ts(d, a_hi + k * 8, wl_desc + static_cast<uint64_t>(k * 16), idesc, 1u);
                        umma_commit(bar_acc);
                        umma_commit(bar_a1);
                    }
                    __syncwarp();
                    par ^= 1u;
                    if (t == kload && gb + 1 < total_blocks) {
                        if (gb >= 1) mbar_wait(bar(kPBarAuxEmpty + ((gb - 1) & 1)), ((gb - 1) >> 1) & 1);
                        load_block(gb + 1);
                    }
                }
                if (++t == T) {
                    t = 0;
                    ++gb;
                }
            }
        }
    } else if (warp < 8) {
        // ------------------------------------------------ E: epilogue, output layer, state update ------------------------------------------------
        const int quad = warp & 3, half = warp >> 2, row = quad * 32 + lane;
        const uint32_t lanebits = static_cast<uint32_t>(quad * 32) << 16;
        Ring<kPipePSlots> sl;
        Ring<kPipeParts> pr;
        int gb = 0;
        for (int c = 0; c < my_chunks; ++c) {
            int t = 0;
            for (int s = 0; s < L * T; ++s) {
                if (t == 0) mbar_wait(bar(kPBarWFull + (gb & 1)), (gb >> 1) & 1);
                const uint32_t aux = sAux_addr + static_cast<uint32_t>(gb & 1) * kAuxPreciseBytes;
                const uint32_t w3a = aux + oW3 + half * 256, w3b = aux + oW3 + 512 + half * 256;   // rows 0 / 1, this thread's 64 columns
                mbar_wait(bar(kPBarAccFull + sl.idx), sl.par);
                tc_fence_after();
                const uint32_t trow = tmem + sl.idx * 256u + lanebits + half * 64;
                uint32_t v[2][16];
                uint64_t acc0[2] = {0ull, 0ull}, acc1[2] = {0ull, 0ull};
                tmem_ld16_async(trow, v[0]);
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    tmem_ld_wait();
                    if (cc + 1 < 4) tmem_ld16_async(trow + (cc + 1) * 16, v[(cc + 1) & 1]);
                    else {   // the slot's columns are in registers: the tile after next may overwrite it
                        tc_fence_before();
                        mbar_arrive(bar(kPBarAccEmpty + sl.idx));
                    }
                    const uint32_t* vv = v[cc & 1];
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const uint4 wa = lds_v4(w3a + (cc * 16 + j) * 4), wb = lds_v4(w3b + (cc * 16 + j) * 4);
                        const uint64_t h01 = pack_f32x2(fmaxf(__uint_as_float(vv[j]), 0.0f), fmaxf(__uint_as_float(vv[j + 1]), 0.0f));
                        const uint64_t h23 = pack_f32x2(fmaxf(__uint_as_float(vv[j + 2]), 0.0f), fmaxf(__uint_as_float(vv[j + 3]), 0.0f));
                        ffma2(acc0[0], h01, pack_u32x2(wa.x, wa.y));
                        ffma2(acc1[0], h01, pack_u32x2(wb.x, wb.y));
                        ffma2(acc0[1], h23, pack_u32x2(wa.z, wa.w));
                        ffma2(acc1[1], h23, pack_u32x2(wb.z, wb.w));
                    }
                }
                const float2 a00 = unpack_f32x2(acc0[0]), a01 = unpack_f32x2(acc0[1]), a10 = unpack_f32x2(acc1[0]), a11 = unpack_f32x2(acc1[1]);
                const float s0 = (a00.x + a00.y) + (a01.x + a01.y), s1 = (a10.x + a10.y) + (a11.x + a11.y);
                if (half == 1) {
                    sPart[pr.idx * kFlowTile + row] = make_float2(s0, s1);
                    mbar_arrive(bar(kPBarPartFull + pr.idx));
                } else {
                    const uint32_t st = sState_addr + static_cast<uint32_t>((t * kFlowTile + row) * 4);
                    float z1 = lds_f32(st), z2 = lds_f32(st + TS * 4), lq = lds_f32(st + 2 * TS * 4);
                    const float b30 = lds_f32(aux + oB3), b31 = lds_f32(aux + oB3 + 4);
                    mbar_wait(bar(kPBarPartFull + pr.idx), pr.par);
                    const float2 o = sPart[pr.idx * kFlowTile + row];
                    if (!SAMPLE) {  // Permute(swap)^-1 precedes the coupling's inverse
                        const float tmp = z1;
                        z1 = z2;
                        z2 = tmp;
                    }
                    const float sh = (s0 + o.x) + b30;  // shift     = param[:, 0::2]
                    const float sc = (s1 + o.y) + b31;  // log-scale = param[:, 1::2]
                    lq -= sc;
                    if (SAMPLE) {
                        sts_f32(st, fmaf(z2, expf(sc), sh));  // z2 * exp(s) + shift, then Permute(swap)
                        sts_f32(st + TS * 4, z1);
                    } else {
                        sts_f32(st, z1);
                        sts_f32(st + TS * 4, (z2 - sh) * expf(-sc));     // the coupling's inverse
                    }
                    sts_f32(st + 2 * TS * 4, lq);
                    mbar_arrive(bar(kPBarStateFull + t));
                }
                sl.next();
                pr.next();
                if (++t == T) {
                    t = 0;
                    mbar_arrive(bar(kPBarAuxEmpty + (gb & 1)));
                    ++gb;
                }
            }
        }
    } else {
        // ------------------------------------------------ Y: chunk input / output, FP32 layer 1 + hi / lo split ------------------------------------------------
        const int w = warp - 8, quad = w & 3, half = w >> 2, row = quad * 32 + lane, ytid = tid - 256;
        const uint32_t lanebits = static_cast<uint32_t>(quad * 32) << 16;
        auto y_sync = [] { asm volatile("bar.sync 1, 256;" ::: "memory"); };
        Ring<kPipePSlots> a1;
        int gb = 0;
        for (int c = 0; c < my_chunks; ++c) {
            const int64_t chunk = blockIdx.x + static_cast<int64_t>(c) * gridDim.x;
            for (int r = ytid; r < T * kFlowTile; r += 256) {
                const int64_t idx = chunk * T * kFlowTile + r;
                float a = 0.0f, b = 0.0f, lq = 0.0f;
                if (idx < n) {
                    if (SAMPLE && in == nullptr) {
                        const RoundKeys rk = expand_key(make_uint2(W.seed_lo, W.seed_hi));
                        const uint4 wd = philox4x32_10(make_uint4(static_cast<uint32_t>(idx), static_cast<uint32_t>(idx >> 32), 0u, kSlotFlowEps), rk);
                        box_muller(wd.x, wd.y, a, b);
                    } else {
                        a = in[idx * 2];
                        b = in[idx * 2 + 1];
                    }
                    if (SAMPLE) {
                        lq = c2 - ((W.base_log_scale[0] + 0.5f * (a * a)) + (W.base_log_scale[1] + 0.5f * (b * b)));
                        a = W.base_loc[0] + expf(W.base_log_scale[0]) * a;
                        b = W.base_loc[1] + expf(W.base_log_scale[1]) * b;
                    }
                }
                sState[0 * TS + r] = a;
                sState[1 * TS + r] = b;
                sState[2 * TS + r] = lq;
            }
            y_sync();
            int t = 0;
            const int gb0 = gb;
            for (int s = 0; s < L * T; ++s) {
                if (t == 0) mbar_wait(bar(kPBarWFull + (gb & 1)), (gb >> 1) & 1);
                if (gb != gb0) mbar_wait(bar(kPBarStateFull + t), (gb - 1) & 1);
                const float z1 = lds_f32(sState_addr + static_cast<uint32_t>(((SAMPLE ? 0 : 1) * TS + t * kFlowTile + row) * 4));
                const uint32_t aux = sAux_addr + static_cast<uint32_t>(gb & 1) * kAuxPreciseBytes;
                const uint32_t w1a = aux + oW1 + half * 256, b1a = aux + oB1 + half * 256;
                // FP32 layer 1, then the FP16 hi / lo split of every activation: 32 + 32 packed columns
                uint32_t hv[32], lv[32];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const uint4 wq = lds_v4(w1a + j * 16), bq = lds_v4(b1a + j * 16);
                    const float a0 = fmaxf(fmaf(__uint_as_float(wq.x), z1, __uint_as_float(bq.x)), 0.0f);
                    const float a1v = fmaxf(fmaf(__uint_as_float(wq.y), z1, __uint_as_float(bq.y)), 0.0f);
                    const float a2 = fmaxf(fmaf(__uint_as_float(wq.z), z1, __uint_as_float(bq.z)), 0.0f);
                    const float a3 = fmaxf(fmaf(__uint_as_float(wq.w), z1, __uint_as_float(bq.w)), 0.0f);
                    const uint32_t h01 = relu_pack_f16(a0, a1v), h23 = relu_pack_f16(a2, a3);   // saturating round to FP16
                    const float2 f01 = unpack_half2(h01), f23 = unpack_half2(h23);
                    hv[2 * j] = h01;
                    hv[2 * j + 1] = h23;
                    lv[2 * j] = pack_half2(a0 - f01.x, a1v - f01.y);
                    lv[2 * j + 1] = pack_half2(a2 - f23.x, a3 - f23.y);
                }
                mbar_wait(bar(kPBarA1Empty + a1.idx), a1.par ^ 1u);
                tc_fence_after();
                const uint32_t ta = tmem + a1.idx * 256u + 128u + lanebits + half * 32;
                tmem_st32(ta, hv);
                tmem_st32(ta + 64u, lv);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                tc_fence_before();
                mbar_arrive(bar(kPBarA1Full + a1.idx));
                a1.next();
                if (++t == T) {
                    t = 0;
                    mbar_arrive(bar(kPBarAuxEmpty + (gb & 1)));
                    ++gb;
                }
            }
            for (int tt = 0; tt < T; ++tt) mbar_wait(bar(kPBarStateFull + tt), (gb - 1) & 1);
            for (int r = ytid; r < T * kFlowTile; r += 256) {
                const int64_t idx = chunk * T * kFlowTile + r;
                if (idx >= n) continue;
                const float a = sState[0 * TS + r], b = sState[1 * TS + r];
                float lq = sState[2 * TS + r];
                if (SAMPLE) {
                    out_theta[idx * 2] = a;
                    out_theta[idx * 2 + 1] = b;
                } else {
                    if (out_theta != nullptr) {   // the latent z = f^-1(x): where the training step's backward sweep starts
                        out_theta[idx * 2] = a;
                        out_theta[idx * 2 + 1] = b;
                    }
                    const float r0 = (a - W.base_loc[0]) / expf(W.base_log_scale[0]);
                    const float r1 = (b - W.base_loc[1]) / expf(W.base_log_scale[1]);
                    lq += c2 - ((W.base_log_scale[0] + 0.5f * (r0 * r0)) + (W.base_log_scale[1] + 0.5f * (r1 * r1)));
                }
                out_lq[idx] = lq;
            }
            y_sync();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

}  // namespace glabc
