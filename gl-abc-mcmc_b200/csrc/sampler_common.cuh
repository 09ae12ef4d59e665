// Pieces shared by the sampler kernels: the launch description, the trace writers and the
// per-chain statistics accumulators.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/glabc.h"
#include "model.cuh"
#include "philox.cuh"

namespace glabc {

// device view of glabc_run_t (validated and narrowed by the host side)
struct RunParams {
    int32_t n_chains;
    uint32_t first_step;   // first loop index i to perform (= step_base + 1)
    uint32_t last_step;    // last loop index (inclusive); last < first means no transition
    uint32_t chain_lo0, chain_hi0;  // global id of chain 0 (low/high words)
    RoundKeys rk;          // Philox round keys of the run's seed
    float gf;
    uint32_t gf_thr_hi;     // native mode: global iff (U_b16 << 16 | junk) < gf_thr_hi, U_b16 the 16-bit
                            // branch uniform and gf_thr_hi = ceil(gf * 2^16) << 16   (cf. B-15/B-16)
    int32_t gf_all_global;  // gf >= 1: every step is global (the threshold would not fit 32 bits)
    int32_t write_row0;
    int32_t trace_runs_16b;  // chain-major d = 2: every chain's 32-row run starts 16-byte aligned (chain_major_runs_16b)
    int64_t trace_rows, trace_chains, trace_chain_off, trace_row_base;
    float* theta;
    float* y;
    float* aux;
    float* trace;
    float* stats;
    const float* tape32;
    const double* tape64;
    float* debug;
    float* tape_dump;
    double* tape64_dump;
    int32_t n_candidates;
    // GLMALA (K3)
    int32_t trace_layout;
    double* state64;
    const float* tape_grad0;
    float* tape_grad0_dump;
    double* debug64;
};

__device__ __forceinline__ Stream chain_stream(const RunParams& r, int32_t chain)
{
    // 64-bit add of the chain index to the global base id
    const uint64_t gid = (static_cast<uint64_t>(r.chain_hi0) << 32 | r.chain_lo0) + static_cast<uint64_t>(chain);
    return Stream{static_cast<uint32_t>(gid), static_cast<uint32_t>(gid >> 32)};
}

// ---------------------------------------------------------------------------------------------
// Trace writers.  Row index = the reference's loop index i (row 0 = initial theta,
// GlobalMCMC.py:34-35); rows are relative to trace_row_base so a run can be chunked.
// ---------------------------------------------------------------------------------------------
template <int D>
struct VecOf { using type = float; };
template <> struct VecOf<2> { using type = float2; };
template <> struct VecOf<4> { using type = float4; };

template <int D>
__device__ __forceinline__ void store_row(float* dst, const float (&v)[D])
{
    if constexpr (D == 2) {
        *reinterpret_cast<float2*>(dst) = make_float2(v[0], v[1]);
    } else if constexpr (D == 4) {
        *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
        for (int k = 0; k < D; ++k) dst[k] = v[k];
    }
}

// TIME_MAJOR: trace[row][chain][d] — a warp's 32 chains are contiguous, one vector store per row.
template <int D>
struct TimeMajorWriter {
    float* next;  // &trace[next row][chain][0]; rows are written consecutively
    bool active;
    __device__ __forceinline__ TimeMajorWriter(const RunParams& r, int32_t chain, bool act, float*)
        : active(act)
    {
        const int64_t first_row = static_cast<int64_t>(r.first_step) - (r.write_row0 ? 1 : 0) - r.trace_row_base;
        next = r.trace + (first_row * r.trace_chains + r.trace_chain_off + chain) * D;
    }
    __device__ __forceinline__ void put(const RunParams& r, uint32_t, const float (&v)[D])
    {
        if (active) store_row<D>(next, v);
        next += r.trace_chains * D;
    }
    __device__ __forceinline__ void maybe_flush(const RunParams&, uint32_t) {}
    __device__ __forceinline__ void finish(const RunParams&) {}
    static constexpr int smem_floats_per_warp = 0;
};

// CHAIN_MAJOR: trace[chain][row][d] — out[c] is a reference-shaped [num_ite, d] chain.  A thread
// per chain would store with a stride of a whole chain, so each warp stages up to 32 rows of its
// 32 chains in shared memory (component-planar, row pitch 33 words: conflict-free both ways) and
// flushes them as 32 runs of 32*D contiguous floats, 128 B per store instruction.
template <int D>
struct ChainMajorWriter {
    static constexpr int kPitch = 33;
    static constexpr int kPlane = 32 * kPitch + (D > 1 ? 32 / D : 0);  // plane skew spreads banks on read
    static constexpr int smem_floats_per_warp = D * kPlane;
    float* tile;       // this warp's tile
    float* out;        // &trace[chain0_of_warp][0][0]
    int64_t chain_stride;
    uint32_t row0;     // absolute row of tile slot 0
    int32_t count;     // buffered rows
    int32_t lane;
    int32_t chains_in_warp;  // valid chains of this warp (tail warp may have < 32)

    __device__ __forceinline__ ChainMajorWriter(const RunParams& r, int32_t, bool, float* smem_warp)
        : tile(smem_warp), chain_stride(r.trace_rows * D), row0(0), count(0), lane(threadIdx.x & 31)
    {
        // warp-uniform geometry (tail lanes shadow another chain's state but must agree on the tile)
        const int32_t chain0 = blockIdx.x * blockDim.x + (threadIdx.x & ~31u);
        out = r.trace + (r.trace_chain_off + chain0) * chain_stride;
        chains_in_warp = min(32, r.n_chains - chain0);
    }

    __device__ __forceinline__ void put(const RunParams& r, uint32_t row, const float (&v)[D])
    {
        if (count == 0) row0 = row;
#pragma unroll
        for (int k = 0; k < D; ++k) tile[k * kPlane + count * kPitch + lane] = v[k];
        ++count;
    }

    // call after put(row): flushes on a 32-row boundary of the absolute row index, so every run a
    // chain receives is 32 rows long and 128B-aligned (the tile never holds more than 32 rows)
    __device__ __forceinline__ void maybe_flush(const RunParams& r, uint32_t row)
    {
        if (((row + 1u) & 31u) == 0u) flush(r);
    }

    __device__ __forceinline__ void flush(const RunParams& r)
    {
        __syncwarp();
        const int32_t n = count * D;  // floats per chain in this tile
        const int64_t off = (static_cast<int64_t>(row0) - r.trace_row_base) * D;
        for (int32_t c = 0; c < chains_in_warp; ++c) {
            float* dst = out + c * chain_stride + off;
            for (int32_t e = lane; e < n; e += 32) {
                const int32_t s = e / D, k = e - s * D;
                dst[e] = tile[k * kPlane + s * kPitch + c];
            }
        }
        __syncwarp();
        count = 0;
    }

    __device__ __forceinline__ void finish(const RunParams& r)
    {
        if (count > 0) flush(r);
    }

    // full-tile entry points of K1's steady loop: the row's slot is the loop position, and the tile
    // [first_row, first_row + 32) ends with one flush
    __device__ __forceinline__ void put_slot(uint32_t slot, const float (&v)[D])
    {
#pragma unroll
        for (int k = 0; k < D; ++k) tile[k * kPlane + slot * kPitch + lane] = v[k];
    }
    __device__ __forceinline__ void flush_tile(const RunParams& r, uint32_t first_row)
    {
        row0 = first_row;
        count = 32;
        flush(r);
    }
};

// D in {1, 2, 4}: a row is one 4/8/16-byte vector.  The tile is chain-major, [32 chains][kPitch]
// vectors, so a lane stores its chain's row with one STS into its own line of the tile, and a flush
// writes chain c's rows as one coalesced run (128/256/512 contiguous bytes for a full tile).
//  - full tile of a full warp, WIDE (D = 2 only) and runs 16-byte aligned (RunParams::trace_runs_16b):
//    a lane moves two rows of one chain as one LDS.128 / STG.128, lanes 0-15 chain c and 16-31 chain
//    c+1, so the tile is 16 STG.128 instead of 32 STG.64;
//  - full tile of a full warp otherwise: one STG per chain, lane = row;
//  - partial tile or tail warp: the same, predicated on lane < count.
// Banks (32 x 4 bytes): pitch 33 vectors is conflict-free both ways.  The 16-byte reads of WIDE need
// an even pitch: 34 float2 = 17 16-byte units.  The STS.64 of a step then runs in two half-warp phases
// in which lanes l and l + 8 meet in 8-byte bank pair 34 l mod 16 (2-way); each quarter-warp phase of
// the LDS.128 reads 8 consecutive 16-byte units of one chain (conflict-free), and the lane = row
// reads are consecutive (conflict-free).  WIDE pays where the trace writer is a large share of the
// issue budget (K1's steady loop); the samplers with heavier steps keep the conflict-free pitch.
template <int D, bool WIDE = false>
struct ChainMajorVecWriter {
    static_assert(!WIDE || D == 2, "the 16-byte flush moves two float2 rows per lane");
    using V = typename VecOf<D>::type;
    static constexpr int kPitch = WIDE ? 34 : 33;
    static constexpr int smem_floats_per_warp = 32 * kPitch * D;
    V* line;           // this lane's chain in the warp's tile (the tile is line - lane * kPitch)
    V* out;            // &trace[chain0_of_warp][0] - trace_row_base, in vector units: indexed by absolute row
    int64_t chain_stride;  // vectors per chain
    uint32_t row0;
    int32_t count, lane, chains_in_warp;

    __device__ __forceinline__ ChainMajorVecWriter(const RunParams& r, int32_t, bool, float* smem_warp)
        : chain_stride(r.trace_rows), row0(0), count(0), lane(threadIdx.x & 31)
    {
        const int32_t chain0 = blockIdx.x * blockDim.x + (threadIdx.x & ~31u);
        line = reinterpret_cast<V*>(smem_warp) + lane * kPitch;
        out = reinterpret_cast<V*>(r.trace) + ((r.trace_chain_off + chain0) * chain_stride - r.trace_row_base);
        chains_in_warp = min(32, r.n_chains - chain0);
    }

    static __device__ __forceinline__ V pack(const float (&v)[D])
    {
        if constexpr (D == 1) return v[0];
        else if constexpr (D == 2) return make_float2(v[0], v[1]);
        else return make_float4(v[0], v[1], v[2], v[3]);
    }

    __device__ __forceinline__ void put(const RunParams&, uint32_t row, const float (&v)[D])
    {
        if (count == 0) row0 = row;
        line[count] = pack(v);
        ++count;
    }

    __device__ __forceinline__ void maybe_flush(const RunParams& r, uint32_t row)
    {
        if (((row + 1u) & 31u) == 0u) flush(r);
    }

    __device__ __forceinline__ void flush(const RunParams& r)
    {
        flush_rows(r, row0, count);
        count = 0;
    }

    __device__ __forceinline__ void finish(const RunParams& r)
    {
        if (count > 0) flush(r);
    }

    // full-tile entry points of K1's steady loop: the row's slot is the loop position, and the tile
    // [first_row, first_row + 32) ends with one flush
    __device__ __forceinline__ void put_slot(uint32_t slot, const float (&v)[D]) { line[slot] = pack(v); }
    __device__ __forceinline__ void flush_tile(const RunParams& r, uint32_t first_row) { flush_rows(r, first_row, 32); }

    // rows [first_row, first_row + n) of the warp's chains; the tile holds them in slots [0, n)
    __device__ __forceinline__ void flush_rows(const RunParams& r, uint32_t first_row, int32_t n)
    {
        __syncwarp();
        const V* tile = line - lane * kPitch;
        if (n == 32 && chains_in_warp == 32) {
            if (WIDE && r.trace_runs_16b) {
                const int32_t h = lane >> 4, j = 2 * (lane & 15);
                const V* src = tile + h * kPitch + j;
                V* dst = out + h * chain_stride + first_row + j;
#pragma unroll
                for (int32_t c = 0; c < 32; c += 2)
                    *reinterpret_cast<float4*>(dst + c * chain_stride) = *reinterpret_cast<const float4*>(src + c * kPitch);
            } else {
                V* dst = out + first_row + lane;
#pragma unroll 8
                for (int32_t c = 0; c < 32; ++c) dst[c * chain_stride] = tile[c * kPitch + lane];
            }
        } else {
            V* dst = out + first_row + lane;
            for (int32_t c = 0; c < chains_in_warp; ++c)
                if (lane < n) dst[c * chain_stride] = tile[c * kPitch + lane];
        }
        __syncwarp();
    }
};

// RunParams::trace_runs_16b of a launch with a WIDE writer: a 32-row run of chain c starts at float2
// (trace_chain_off + c) * trace_rows + row - trace_row_base with row % 32 == 0, so every run is
// 16-byte aligned when the buffer is and trace_rows and trace_row_base are even.
inline bool chain_major_runs_16b(const RunParams& r)
{
    return (reinterpret_cast<uintptr_t>(r.trace) & 15u) == 0 && (r.trace_rows & 1) == 0 && (r.trace_row_base & 1) == 0;
}

// EVENTS: the chain as its moves (glabc.h GLABC_TRACE_EVENTS).  One scattered store per move instead of one row per step.
template <int D>
struct EventWriter {
    float* ev;        // &events[chain][0][0], entries of 1 + D floats
    uint32_t n;       // entries used so far + 1 (entry 0 is the header)
    uint32_t cap;     // trace_rows
    float last[D];
    bool active;
    static constexpr int smem_floats_per_warp = 0;
    __device__ __forceinline__ EventWriter(const RunParams& r, int32_t chain, bool act, float*)
        : ev(r.trace + (r.trace_chain_off + chain) * r.trace_rows * (1 + D)), n(1u), cap(static_cast<uint32_t>(r.trace_rows)), active(act)
    {
#pragma unroll
        for (int k = 0; k < D; ++k) last[k] = __int_as_float(0x7fc00000);   // NaN: the first row always differs
    }
    __device__ __forceinline__ void put(const RunParams&, uint32_t row, const float (&v)[D])
    {
        bool moved = false;
#pragma unroll
        for (int k = 0; k < D; ++k) moved |= !(v[k] == last[k]);
        if (moved) {
            if (active && n < cap) {
                float* e = ev + static_cast<int64_t>(n) * (1 + D);
                e[0] = __uint_as_float(row);
#pragma unroll
                for (int k = 0; k < D; ++k) e[1 + k] = v[k];
            }
            ++n;
#pragma unroll
            for (int k = 0; k < D; ++k) last[k] = v[k];
        }
    }
    __device__ __forceinline__ void maybe_flush(const RunParams&, uint32_t) {}
    __device__ __forceinline__ void finish(const RunParams&)
    {
        if (active) ev[0] = __uint_as_float(n - 1u);
    }
};

struct NoTraceWriter {
    __device__ __forceinline__ NoTraceWriter(const RunParams&, int32_t, bool, float*) {}
    template <int D>
    __device__ __forceinline__ void put(const RunParams&, uint32_t, const float (&)[D]) {}
    __device__ __forceinline__ void maybe_flush(const RunParams&, uint32_t) {}
    __device__ __forceinline__ void finish(const RunParams&) {}
    static constexpr int smem_floats_per_warp = 0;
};

// WIDE: the chain-major d = 2 writer with the 16-byte full-tile flush (ChainMajorVecWriter)
template <int D, int LAYOUT, bool WIDE = false> struct WriterFor;
template <int D, bool W> struct WriterFor<D, GLABC_TRACE_NONE, W> { using type = NoTraceWriter; };
template <int D, bool W> struct WriterFor<D, GLABC_TRACE_TIME_MAJOR, W> { using type = TimeMajorWriter<D>; };
template <int D, bool W> struct WriterFor<D, GLABC_TRACE_CHAIN_MAJOR, W> { using type = ChainMajorVecWriter<D, W && D == 2>; };
template <bool W> struct WriterFor<3, GLABC_TRACE_CHAIN_MAJOR, W> { using type = ChainMajorWriter<3>; };
template <int D, bool W> struct WriterFor<D, GLABC_TRACE_EVENTS, W> { using type = EventWriter<D>; };

// ---------------------------------------------------------------------------------------------
// Per-chain statistics (layout: GLABC_STAT_* in glabc.h)
// ---------------------------------------------------------------------------------------------
template <int D>
struct ChainStats {
    static constexpr int kTri = D * (D + 1) / 2;
    uint32_t n_global, acc_local, acc_global;
    float f_global, f_acc, f_acc_global;  // FAST path: the same counts kept as floats on the FMA pipe
                                          // (exact below 2^24 transitions per launch — host-enforced)
    float sum[D], sumsq[D], gram[kTri];

    __device__ __forceinline__ ChainStats()
        : n_global(0), acc_local(0), acc_global(0), f_global(0.0f), f_acc(0.0f), f_acc_global(0.0f)
    {
#pragma unroll
        for (int i = 0; i < D; ++i) sum[i] = sumsq[i] = 0.0f;
#pragma unroll
        for (int i = 0; i < kTri; ++i) gram[i] = 0.0f;
    }

    // theta_new is the post-decision state; delta = theta_new - theta_prev (zero unless moved)
    __device__ __forceinline__ void update(bool is_global, bool moved, const float (&theta_new)[D],
                                           const float (&theta_prev)[D])
    {
        n_global += is_global;
        acc_global += (moved && is_global);
        acc_local += (moved && !is_global);
        float dl[D];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            sum[i] += theta_new[i];
            sumsq[i] = fmaf(theta_new[i], theta_new[i], sumsq[i]);
            dl[i] = theta_new[i] - theta_prev[i];
        }
        int t = 0;
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = i; j < D; ++j, ++t) gram[t] = fmaf(dl[i], dl[j], gram[t]);
    }

    // glob, moved: 0/1 masks
    __device__ __forceinline__ void update_masked(float glob, float moved, const float (&theta_new)[D],
                                                  const float (&theta_prev)[D])
    {
        f_global += glob;
        f_acc += moved;
        f_acc_global = fmaf(moved, glob, f_acc_global);
        float dl[D];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            sum[i] += theta_new[i];
            sumsq[i] = fmaf(theta_new[i], theta_new[i], sumsq[i]);
            dl[i] = theta_new[i] - theta_prev[i];
        }
        int t = 0;
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = i; j < D; ++j, ++t) gram[t] = fmaf(dl[i], dl[j], gram[t]);
    }

    __device__ __forceinline__ void store(float* st, uint32_t n_steps) const
    {
        st[GLABC_STAT_STEPS] += static_cast<float>(n_steps);
        st[GLABC_STAT_GLOBAL_STEPS] += static_cast<float>(n_global) + f_global;
        st[GLABC_STAT_ACC_LOCAL] += static_cast<float>(acc_local) + (f_acc - f_acc_global);
        st[GLABC_STAT_ACC_GLOBAL] += static_cast<float>(acc_global) + f_acc_global;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            st[GLABC_STAT_SUM + i] += sum[i];
            st[GLABC_STAT_SUM + D + i] += sumsq[i];
        }
#pragma unroll
        for (int i = 0; i < kTri; ++i) st[GLABC_STAT_SUM + 2 * D + i] += gram[i];
    }
};

}  // namespace glabc
