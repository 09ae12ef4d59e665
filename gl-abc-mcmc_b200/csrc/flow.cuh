// K4 — the RealNVP importance proposal of GLMCMC-NFs (reference GLMCMC_NFs.py:51-61,72,98,127; normflows
// pieces restated in SURVEY.md Appendix C): 32 x [AffineCouplingBlock(MLP([1,128,128,2])), Permute(swap)] over a
// trainable DiagGaussian(2) base.  sample(n) and log_prob(x) for large batches.
//
// What the flow kernels share: the sizes, the device view of the weights (FlowDev), W2's packing into the UMMA operand
// layout (k_flow_pack), and thin wrappers over the mbarrier, bulk-copy, tcgen05 (MMA, TMEM load / store) and FP16 pack
// instructions.  The forward kernels (sample, log_prob; FAST and PRECISE) are k_flow_pipe / k_flow_pipe_precise in
// flow_pipe.cuh, the training step's backward sweep is k_flow_bwd in flow_train.cuh.
//
// The 128 x 128 hidden layer of every coupling MLP runs on the tensor cores with FP16 operands (kind::f16, FP32 accumulate):
// FP16 and TF32 carry the same 10-bit mantissa, but kind::f16 runs at twice the tensor rate, and ReLU + saturation + rounding
// + packing of TWO activations is ONE instruction (F2FP.SATFINITE.RELU.F16.F32.PACK_AB).  Activations beyond 65504 saturate
// instead of overflowing.  sample() and log_prob() evaluate the SAME deterministic network (same roundings), so the
// log-density returned for a sample is the exact density of the map that produced it — importance weights stay exact
// whatever the operand precision; only the agreement with an fp32 evaluation of the weights is ~1e-3 (FAST mode).
// PRECISE mode (split precision, SURVEY.md 7.3(5)): A = A_hi + A_lo and W2 = W_hi + W_lo as FP16 pairs, three MMAs per K step
// (A_hi W_hi + A_lo W_hi + A_hi W_lo, FP32 accumulate; the dropped A_lo W_lo term is 2^-22 of the product), layers 1 and 3 and
// every vector in FP32 on the CUDA cores.  FP16 subnormals keep the lo parts to 3e-8 absolute, so the hidden layer carries
// ~22 significant bits and the flow's log-density agrees with a float64 evaluation to ~1e-6 (tests/test_flow_gpu.py): the
// tolerance north_star states (1e-5) — which single FP16 operands miss by 20-600x.
#pragma once
#include <cstdint>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "philox.cuh"

namespace glabc {

constexpr int kFlowHidden = 128;
constexpr int kFlowTile = 128;
// capacity (shared-memory state slots) of a CTA's chunk; the launcher picks the tiles per chunk at run time (<= this) so that a
// small batch still spreads over all SMs: 32 tiles per weight fetch measured 4 % faster than 16 on 8.4 M samples
constexpr int kFlowTilesPerCta = 32;
constexpr int kFlowW2Bytes = kFlowHidden * kFlowHidden * 2;   // W2 of one coupling block as FP16: 32 KB

// per coupling block, the small operands pre-packed for the flow kernels (flow_pipe.cuh: k_flow_pack_aux)
constexpr int kFlowAuxBytes = 10880;   // FAST reads bytes [0, 8832), PRECISE bytes [4608, 10880) of a block's blob

struct FlowDev {
    const float* w1;   // [L][128]
    const float* b1;   // [L][128]
    const float* w2p;  // [L][128*128] FP16, UMMA K-major / no-swizzle core-matrix layout (flow_pack_offset)
    const float* w2p_lo;  // PRECISE mode: FP16(W2 - FP16(W2)) in the same layout
    const float* b2;   // [L][128]
    const float* w3;   // [L][2][128]
    const float* b3;   // [L][2]
    const uint8_t* aux;   // [L][kFlowAuxBytes]: W3 and b2 as UMMA operands, w1 / b1 as FP16 pairs, b3, W3 / w1 / b1 in FP32 (k_flow_pack_aux)
    float base_loc[2], base_log_scale[2];
    int32_t n_blocks;
    // sample() without an eps buffer: the base normals of sample i are Box-Muller of Philox4x32-10(counter = (i, kSlotFlowEps), key = seed)
    uint32_t seed_lo, seed_hi;
};

constexpr uint32_t kSlotFlowEps = 0x60000000u;

// byte offset of element (row r, k) of a [128][128] FP16 operand in the K-major no-swizzle canonical layout:
// core matrix = 8 rows x 16 bytes (8 halves), core matrices contiguous along K (LBO = 128 B), 8-row groups 2 KB apart (SBO)
__host__ __device__ constexpr uint32_t flow_pack_offset(uint32_t r, uint32_t k)
{
    return (r >> 3) * 2048u + (k >> 3) * 128u + (r & 7u) * 16u + (k & 7u) * 2u;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"   // suspend-time hint: sleep in hardware, not in a spin loop
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity), "r"(0x989680u)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor: K-major, SWIZZLE_NONE, version 1 (cute::UMMA::SmemDescriptor bit layout)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4) | (static_cast<uint64_t>(lbo_bytes >> 4) << 16) |
           (static_cast<uint64_t>(sbo_bytes >> 4) << 32) | (1ull << 46);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
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
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 16 columns, asynchronous: the registers are valid after tmem_ld_wait()
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        :
        : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
          "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]),
          "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]),
          "r"(v[30]), "r"(v[31])
        : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem]^T with FP16 operands: K = 16 per instruction, A row i = TMEM lane i, 16 halves = 8 columns
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T with FP16 operands
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// one lane of a converged warp (the warp runs the issue loops together: a lone diverged thread pays ~45 cycles per
// tcgen05.mma for the compiler's elect / R2UR.BROADCAST sequence; from a converged warp the MMAs issue back to back)
__device__ __forceinline__ bool elect_one()
{
    uint32_t p;
    asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(p));
    return p != 0;
}

// relu(lo), relu(hi) -> saturated, rounded FP16 pair (lo in bits 0..15): one F2FP instruction
__device__ __forceinline__ uint32_t relu_pack_f16(float lo, float hi)
{
    uint32_t r;
    asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// relu(a * b + c) on two FP16 lanes at once (HFMA2.RELU): layer 1 of the coupling MLP directly in the A operand's format
__device__ __forceinline__ uint32_t hfma2_relu(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t hfma2(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi)
{
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_half2(uint32_t v) { return __half22float2(*reinterpret_cast<const __half2*>(&v)); }

// pack W2 [L][out=128][in=128] (torch Linear.weight) into the UMMA layout as FP16, and (w2p_lo non-null) the FP16 remainder
static __global__ void __launch_bounds__(256) k_flow_pack(const float* __restrict__ w2, float* __restrict__ w2p, float* __restrict__ w2p_lo,
                                                          int64_t total)
{
    const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (g >= total) return;
    const int64_t l = g / (kFlowHidden * kFlowHidden);
    const uint32_t e = static_cast<uint32_t>(g - l * kFlowHidden * kFlowHidden);
    const uint32_t r = e / kFlowHidden, k = e % kFlowHidden;
    const __half hi = __float2half_rn(w2[g]);
    reinterpret_cast<__half*>(w2p)[l * kFlowHidden * kFlowHidden + flow_pack_offset(r, k) / 2] = hi;
    if (w2p_lo != nullptr)
        reinterpret_cast<__half*>(w2p_lo)[l * kFlowHidden * kFlowHidden + flow_pack_offset(r, k) / 2] = __float2half_rn(w2[g] - __half2float(hi));
}

cudaError_t launch_flow_pack(const float* w2, float* w2p, float* w2p_lo, int n_blocks, cudaStream_t st);
cudaError_t launch_flow_pack_aux(const float* w1, const float* b1, const float* b2, const float* w3, const float* b3, uint8_t* aux,
                                 int n_blocks, cudaStream_t st);
cudaError_t launch_flow(const FlowDev& W, bool sample, bool precise, const float* in, int64_t n, float* out_theta, float* out_lq,
                        int sm_count, cudaStream_t st);

}  // namespace glabc
