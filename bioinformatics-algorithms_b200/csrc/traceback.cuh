// traceback.cuh -- one thread per pair walks the short16 record.
//
// Replaces hw2.cpp:158-188 (NW) / hw2.cpp:235-263 (SW) and overlapLongestExactMatch (hw2.cpp:267-278)
// for every pair of the batch.  The direction of a cell is decided by the reference's own comparisons
// (hw2.cpp:145-153 NW, hw2.cpp:214-222 SW) on the exact H of the cell and its three neighbours, which the
// delta record yields in O(1) per cell (one 16-byte chunk load + a popcount prefix sum from the anchor).
//
// Shaped for a WARP of 32 independent walks, where anything that is rare per thread happens almost every
// iteration somewhere in the warp, so every iteration runs the same code:
//   * NW walks one DP row per iteration (row_walk.h, shared with the CPU harness of the tests): both rows
//     are re-sought at the current column, then a branch-free scan over a window of up to 8 columns finds
//     where the row's run of 'l' moves ends and takes the terminal 'M' or 'D'.  A config-2 path is a
//     staircase (~150 climbs, runs of ~4.5 'l' moves), so this takes ~190 iterations per warp where a step
//     per cell took ~690 (the run along the last row is just the first row of the loop);
//   * SW takes one uniform branch-free step per cell (local paths are mostly diagonal, a row walk saves
//     nothing): both rows are re-sought every step (the chunk of the lower row was loaded as the upper row
//     one step earlier, so it hits L1) instead of carrying cursors whose chunk-boundary reloads and row
//     changes diverge; it starts from the end cell the fill kernel's epilogue already found (FillArgs::endcell);
//   * border tails are emitted in bulk.
// The generic cursor walkers in b2a_format.h stay the executable specification (CPU host model, wide32 warp walker).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "b2a_format.h"
#include "short16_fill.cuh"
#include "row_walk.h"

namespace b2a {

struct TbArgs {
    const uint8_t*  pat;
    const uint8_t*  txt;
    const uint64_t* pat_off;
    const uint64_t* txt_off;
    const PPDesc*   pps;
    const uint64_t* code_off;
    const Chunk*    codes;
    const uint32_t* rowbest;
    const int4*     endcell;    // local and semi-global modes, per pair: {score, end_i, end_j, 0} from the fill kernel
    PairResult*     results;    // indexed by pair
    uint32_t*       ops;        // packed 2-bit ops, may be null
    const uint64_t* ops_off;    // per pair word offset into ops
    uint32_t        n_pp;
    int32_t         R;
    int32_t         match, mismatch, gap, bias;
    int32_t         opt;
    int32_t         tie_hw4;    // global mode: tie order d > u > l (hw4.cpp:37-46) and overlap := hw4's distance
    const AlphaInfo* alpha;
    const uint8_t*  dirty;      // per pair-pair: 2 = skipped by the s16x2 fill kernels (served by wide32)
};

struct DevLoader {
    const Chunk* base;
    __device__ __forceinline__ Chunk operator()(uint64_t idx) const {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(base + idx));
        return Chunk{v.x, v.y, v.z, v.w};
    }
    __device__ __forceinline__ void prefetch(uint64_t idx) const {
        asm volatile("prefetch.global.L2 [%0];" :: "l"(base + idx));
    }
};

// row_walk.h's memory interface: read-only chunk and aligned text-word loads
struct DevMem {
    __device__ __forceinline__ Chunk chunk(const Chunk* p) const {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
        return Chunk{v.x, v.y, v.z, v.w};
    }
    __device__ __forceinline__ uint64_t word8(const uint8_t* p) const {
        return __ldg(reinterpret_cast<const unsigned long long*>(p));
    }
};

constexpr int TB_THREADS = 128;

// one pair's view of its half of a pair-pair record
template <int K>
struct S16View {
    using FM = Short16<K>;
    const Chunk* rec;
    uint32_t NC, R, rmagic, stride;    // stride = 32R: distance between consecutive chunks of a row
    uint32_t sel_lo, sel_hi;     // PRMT selectors of this pair's 16-bit half
    int gap;

    // first chunk of DP row i >= 1 (its chunks are 32R apart) and the lane that owned the row in the fill
    // (step q = j + L; no runtime division, see row_slot)
    __device__ __forceinline__ const Chunk* row_base(uint32_t i, uint32_t& L) const {
        const uint32_t x = i - 1u;
        L = (x * rmagic) >> 16;
        return rec + x;
    }
    // field string of a chunk (step rem at bit K*(CS-1-rem)) and its anchor
    __device__ __forceinline__ uint64_t unpack(const uint4& ch, int& anchor) const {
        const uint32_t lo = __byte_perm(ch.z, ch.y, sel_lo);              // (w1.half << 16) | w2.half
        const uint32_t hi = __byte_perm(ch.x, 0u, sel_hi);                // w0.half
        anchor = (int)__byte_perm(ch.w, 0u, sel_hi);
        return ((uint64_t)hi << 32) | lo;
    }
    // (tried and lost, per 1 M pairs: prefetch.global.L1 of the rows above 6.2 -> 7.9 ms NW / 2.7 -> 6.2 ms SW;
    //  ld.cg instead of ld.nc for the chunks 6.2 -> 7.2 ms NW; ld.cs 6.2 -> 8.9 ms)
    // exact (biased) H of cell (i, j), i >= 1, and its horizontal delta D = H(i,j) - H(i,j-1) - gap
    __device__ __forceinline__ void cell(uint32_t i, uint32_t j, int& H, int& D) const {
        uint32_t L;
        const Chunk* rb = row_base(i, L);
        const uint32_t q = j + L, c = q / (uint32_t)FM::CS, rem = q - c * (uint32_t)FM::CS;
        const uint4 ch = __ldg(reinterpret_cast<const uint4*>(rb + (size_t)c * stride));
        int anchor;
        const uint64_t X = unpack(ch, anchor);
        const int off = K * (FM::CS - 1 - (int)rem);
        D = (int)((uint32_t)(X >> off) & FM::MASK);
        H = anchor - (FM::CS - 1 - (int)rem) * gap - field_sum64<K>(X & ((1ull << off) - 1ull));
    }
};

#ifndef TB_MIN_CTAS
#define TB_MIN_CTAS 1
#endif
// SEMI (with LOCAL = false): the semi-global row walk from the end cell the fill's epilogue found (FillArgs::endcell)
template <int K, bool LOCAL, bool SEMI = false>
__global__ void __launch_bounds__(TB_THREADS, TB_MIN_CTAS)
short16_traceback_kernel(const TbArgs A)
{
    using FM = Short16<K>;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t pp = t >> 1;
    const int half = (int)(t & 1u);
    if (pp >= A.n_pp || A.dirty[pp] == 2) return;         // 2: more than 7 pattern symbols, no s16x2 record (wide32 serves the pair-pair)
    const PPDesc d = A.pps[pp];
    if (half && d.b == d.a) return;                       // singleton: the high half is a duplicate
    const uint32_t pair = half ? d.b : d.a;
    const uint8_t* __restrict__ P = A.pat + A.pat_off[pair];
    const uint8_t* __restrict__ T = A.txt + A.txt_off[pair];
    const int gap = A.gap, match = A.match, mismatch = A.mismatch;
    const uint32_t mh = pp_dim(d.m, half), nh = pp_dim(d.n, half);   // this pair's own shape; the record is laid out for max(n)
    OpsRunSink sink(A.ops ? A.ops + A.ops_off[pair] : nullptr);
    PairResult res;
    res.path = 1;

    if (SEMI) {
        RowWalkPair v{A.codes + A.code_off[pp], P, T, mh, nh, (uint32_t)A.R, (uint32_t)short16_rmagic(A.R), half,
                      match, mismatch, gap, A.bias, false};
        v.j_end = (uint32_t)A.endcell[pair].z;
        row_walk_global<K, DevMem, OpsRunSink, true>(v, DevMem{}, sink, res);
        sink.flush();
        A.results[pair] = res;
        return;
    }
    if (!LOCAL) {
        // ---- NW: one DP row per iteration (row_walk.h) ----
        const RowWalkPair v{A.codes + A.code_off[pp], P, T, mh, nh, (uint32_t)A.R, (uint32_t)short16_rmagic(A.R), half,
                            match, mismatch, gap, A.bias, A.tie_hw4 != 0};
        row_walk_global<K>(v, DevMem{}, sink, res);
        sink.flush();
        A.results[pair] = res;
        return;
    }

    // ---- SW: one uniform branch-free step per cell from the fill's end cell ----
    S16View<K> v{A.codes + A.code_off[pp], num_chunks(pp_max(d.n), FM::CS), (uint32_t)A.R, (uint32_t)short16_rmagic(A.R), 32u * (uint32_t)A.R,
                 half ? 0x7632u : 0x5410u, half ? 0x4432u : 0x4410u, gap};
    const int4 e = A.endcell[pair];
    res.score = e.x; res.end_i = (uint32_t)e.y; res.end_j = (uint32_t)e.z;
    uint32_t i = res.end_i, j = res.end_j, nops = 0;
    if (e.x == 0) { i = 0; j = 0; }                       // hw2.cpp:202-203: best cell stays (0,0), empty alignment
    int cur = 0, best = 0;
    while (i > 0u && j > 0u) {
        int H, D, Hu, Du;
        v.cell(i, j, H, D);
        v.cell(i > 1u ? i - 1u : 1u, j, Hu, Du);
        if (i == 1u) { Hu = 0; Du = -gap; }                                                  // border row, hw2.cpp:196-197
        if (H == 0) break;                                                                   // hw2.cpp:239
        const int Hd = Hu - Du - gap;
        const uint8_t pc = P[i - 1u];
        const bool eq = pc == T[j - 1u];
        const int dv = Hd + (eq ? match : mismatch);                                         // hw2.cpp:208
        const uint32_t op = H == dv ? OP_M : (H == Hu + gap ? OP_D : OP_I);                  // hw2.cpp:214-222 (H != 0 here)
        cur = (op == OP_M && eq && pc != (uint8_t)'-') ? cur + 1 : 0;                        // hw2.cpp:267-278
        best = max(best, cur);
        i -= op != OP_I; j -= op != OP_D;
        sink.put(op); ++nops;
    }
    sink.flush();
    res.start_i = i; res.start_j = j; res.n_ops = nops;
    res.overlap = best;
    A.results[pair] = res;
}

} // namespace b2a
