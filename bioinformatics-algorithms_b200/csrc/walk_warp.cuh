// walk_warp.cuh -- warp-cooperative traceback over the delta record (device only).
//
// The per-thread walkers in b2a_format.h follow the path one cell at a time: a chain of dependent
// chunk loads, fine when a batch supplies a thread per pair, hopeless for ONE 100 kb x 100 kb pair
// (200 k dependent steps).  Here a warp walks one pair.  The direction of a cell depends only on the
// exact H of the cell and of its three neighbours, all of which the record yields in O(1) per cell
// (RowCursor::seek), so the 32 lanes evaluate the directions of the next 32 cells of a HYPOTHESIS --
// the path continues diagonally (cells (i-k, j-k)), vertically ((i-k, j)) or horizontally ((i, j-k)) --
// in parallel with the reference's own comparisons (hw2.cpp:145-153 NW, hw2.cpp:214-222 SW).  The
// leading lanes that confirm the hypothesis are accepted in one go, the first lane that does not
// contributes its own (different) move, and the walk resumes from there.  Every accepted move was
// decided by exactly the test the reference applies to that cell, so the path is the reference's.
// One iteration = one round of independent 16-byte loads; the chunks of the next diagonal window are
// prefetched into L2 while the current one is evaluated.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "b2a_format.h"

namespace b2a {

// 2-bit op writer with warp-uniform state; only `writer` (lane 0) touches memory
struct WarpOpsSink {
    uint32_t* out;
    uint32_t word, fill;
    uint64_t pos;
    bool writer;
    __device__ __forceinline__ WarpOpsSink(uint32_t* o, bool w) : out(o), word(0), fill(0), pos(0), writer(w) {}
    __device__ __forceinline__ void put_run(uint32_t op, uint32_t cnt) {
        while (cnt) {
            const uint32_t take = min(cnt, 16u - fill);
            if (op) {
                const uint32_t span = take == 16u ? 0xFFFFFFFFu : ((1u << (2u * take)) - 1u);
                word |= ((op * 0x55555555u) & span) << (2u * fill);
            }
            fill += take; cnt -= take;
            if (fill == 16u) { if (out && writer) out[pos] = word; ++pos; word = 0; fill = 0; }
        }
    }
    __device__ __forceinline__ void flush() { if (fill && out && writer) out[pos] = word; }
};

// longest-exact-match bookkeeping (overlapLongestExactMatch, hw2.cpp:267-278) for t accepted 'M'
// columns whose exactness is bit k of `em` (k = 0 first)
__device__ __forceinline__ void overlap_run(uint32_t em, uint32_t t, int& cur, int& best) {
    if (t == 0) return;
    const uint32_t span = t >= 32u ? 0xFFFFFFFFu : ((1u << t) - 1u);
    const uint32_t m = em & span;
    if (m == span) { cur += (int)t; best = max(best, cur); return; }
    const int lead = __ffs(~m) - 1;                         // leading exact columns continue the open run
    cur += lead; best = max(best, cur);
    uint32_t x = m; int len = 0;
    while (x) { x &= x >> 1; ++len; }                       // longest run of ones inside the window
    best = max(best, len);
    cur = __clz(~(m << (32u - t)));                         // exact columns at the far end stay open
}

enum : int { HYP_DIAG = 0, HYP_UP = 1, HYP_LEFT = 2 };

template <class FM, class Loader, bool LOCAL>
__device__ __forceinline__ void warp_prefetch_window(const PairView& v, const Loader& ld, uint32_t i, uint32_t j, int lane) {
    // rows i-32-lane (and the one above the last) around the continued diagonal
    if (i > 32u + (uint32_t)lane) {
        const uint32_t pi = i - 32u - (uint32_t)lane, pj = j > 32u + (uint32_t)lane ? j - 32u - (uint32_t)lane : 1u;
        uint32_t L;
        const uint64_t base = chunk_index<FM>(v, pi, 0, L);
        ld.prefetch(base + (uint64_t)((pj + L * (uint32_t)FM::SKEW) / (uint32_t)FM::CS) * chunk_stride<FM>(v));
    }
}

// Walks from (i, j) until the reference's loop would stop; returns the stop cell in (i, j).  `cur` is the exact-match run that is open
// at (i, j) (0 at the start of an alignment; a checkpointed walk carries it from one sub-problem to the next).
// (Measured and dropped in round 2: rounds that decide the cells of THREE neighbouring diagonals per lane, so that a window survives one
//  indel and continues on the shifted diagonal.  Fewer rounds, but three seeks + three decisions per lane made a round 1.8x as expensive:
//  the 100 kb pair of config 4 went from 7.0 to 8.0 ms.  A round is bound by its ~110 instructions per lane, not by the load latency.)
// SEMI (with LOCAL = false): NW decisions over the semi-global record, whose row 0 is free (H = 0, D = -gap: the cursor's SW border).
template <class FM, class Loader, bool LOCAL, bool SEMI = false>
__device__ __forceinline__ void warp_walk(const PairView& v, const Loader& ld, WarpOpsSink& sink, uint32_t& i, uint32_t& j,
                                           uint32_t& nops, int& best, uint32_t& mism, int& cur)
{
    const int lane = (int)(threadIdx.x & 31u);
    const bool hw4 = !LOCAL && (v.opt & 4) != 0;            // tie order d > u > l (hw4.cpp:37-46) instead of hw2's d > l > u
    int hyp = HYP_DIAG;
    uint32_t last_op = OP_M;
    while (i > 0 && j > 0) {
        const uint32_t di = hyp == HYP_LEFT ? 0u : (uint32_t)lane, dj = hyp == HYP_UP ? 0u : (uint32_t)lane;
        const bool valid = i > di && j > dj;                       // the hypothesised cell is inside the matrix
        uint32_t op = OP_M; bool stop = false, exact = false, differ = false;
        if (valid) {
            const uint32_t ci = i - di, cj = j - dj;
            RowCursor<FM, Loader, LOCAL || SEMI> rc, ru;
            rc.seek(v, ld, ci, cj);
            ru.seek(v, ld, ci - 1u, cj);
            const int H = rc.H, Hl = H - rc.D() - v.gap;            // H(ci, cj-1); frozen lanes make this the border at cj == 1
            const int Hu = ru.H, Hd = Hu - ru.D() - v.gap;          // H(ci-1, cj), H(ci-1, cj-1)
            const uint8_t pc = v.p[ci - 1u];
            const bool eq = pc == v.t[cj - 1u];
            const int dv = Hd + (eq ? v.match : v.mismatch);
            if (LOCAL) {                                            // hw2.cpp:239, :214-222
                stop = H == 0;
                op = H == dv ? OP_M : (H == Hu + v.gap ? OP_D : OP_I);
            } else if (!hw4) {                                      // hw2.cpp:142-153: d, then l if strictly larger, then u if strictly larger
                int val = dv;
                if (Hl + v.gap > val) { val = Hl + v.gap; op = OP_I; }
                if (Hu + v.gap > val) op = OP_D;
            } else {                                                // hw4.cpp:37-46: d, then u if strictly larger, then l if strictly larger
                int val = dv;
                if (Hu + v.gap > val) { val = Hu + v.gap; op = OP_D; }
                if (Hl + v.gap > val) op = OP_I;
            }
            exact = eq && pc != (uint8_t)'-';
            differ = !eq;
        }
        if (hyp == HYP_DIAG) warp_prefetch_window<FM, Loader, LOCAL>(v, ld, i, j, lane);
        const uint32_t want = hyp == HYP_DIAG ? OP_M : (hyp == HYP_UP ? OP_D : OP_I);
        const uint32_t ok = __ballot_sync(0xFFFFFFFFu, valid && !stop && op == want);
        const uint32_t t = ok == 0xFFFFFFFFu ? 32u : (uint32_t)(__ffs(~ok) - 1);     // leading lanes confirming the hypothesis
        if (t) {
            sink.put_run(want, t); nops += t;
            if (want == OP_M) {
                overlap_run(__ballot_sync(0xFFFFFFFFu, exact), t, cur, best);
                mism += (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, differ) & (t >= 32u ? 0xFFFFFFFFu : ((1u << t) - 1u)));
                i -= t; j -= t;
            }
            else { cur = 0; if (want == OP_D) i -= t; else j -= t; }
            last_op = want;
        }
        if (t == 32u) continue;
        // lane t is the first cell off the hypothesis: it is the path's current cell; apply its own move
        const uint32_t v_t = __shfl_sync(0xFFFFFFFFu, (uint32_t)valid, (int)t);
        if (!v_t) break;                                            // i == 0 or j == 0: the caller finishes the border
        const uint32_t s_t = __shfl_sync(0xFFFFFFFFu, (uint32_t)stop, (int)t);
        if (s_t) break;                                             // local: H == 0
        const uint32_t op_t = __shfl_sync(0xFFFFFFFFu, op, (int)t);
        const uint32_t ex_t = __shfl_sync(0xFFFFFFFFu, (uint32_t)exact, (int)t);
        const uint32_t df_t = __shfl_sync(0xFFFFFFFFu, (uint32_t)differ, (int)t);
        sink.put_run(op_t, 1u); ++nops;
        if (op_t == OP_M) { mism += df_t; if (ex_t) { if (++cur > best) best = cur; } else cur = 0; --i; --j; }
        else { cur = 0; if (op_t == OP_D) --i; else --j; }
        // gap runs are short unless proven otherwise: switch hypothesis only after two equal gap moves in a row
        hyp = op_t == OP_M ? HYP_DIAG : (op_t == last_op ? (op_t == OP_D ? HYP_UP : HYP_LEFT) : HYP_DIAG);
        last_op = op_t;
    }
}

// first row-major arg-max (hw2.cpp:225-229) with the whole warp: per-row maxima -> first best row,
// then every lane rebuilds a share of that row's chunks backwards from their anchors
template <class FM, class Loader>
__device__ __forceinline__ void warp_find_local_end(const PairView& v, const Loader& ld, int& M, uint32_t& bi, uint32_t& bj) {
    const int lane = (int)(threadIdx.x & 31u);
    M = 0; bi = 0; bj = 0;
    if (v.n == 0 || v.m == 0) return;
    int mloc = 0; uint32_t iloc = 0xFFFFFFFFu;
    for (uint32_t i = (uint32_t)lane + 1u; i <= v.m; i += 32u) {
        uint32_t L;
        const uint32_t slot = row_slot<FM>(v, i, L);
        const int rb = rowbest_of<FM>(v.rowbest[(uint64_t)slot * 32u + L], v.half);
        if (rb > mloc) { mloc = rb; iloc = i; }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const int om = __shfl_xor_sync(0xFFFFFFFFu, mloc, o);
        const uint32_t oi = __shfl_xor_sync(0xFFFFFFFFu, iloc, o);
        if (om > mloc || (om == mloc && oi < iloc)) { mloc = om; iloc = oi; }
    }
    if (mloc == 0) return;                                          // hw2.cpp:202-203: best cell stays (0,0)
    M = mloc; bi = iloc;
    uint32_t L;
    const uint64_t rowbase = chunk_index<FM>(v, bi, 0, L);
    L *= (uint32_t)FM::SKEW;                                        // the row's step offset: column j sits at step q = j + L
    const uint32_t c0 = (L + 1u) / (uint32_t)FM::CS, c1 = (L + v.n) / (uint32_t)FM::CS;   // chunks holding columns 1..n
    uint32_t cand = 0xFFFFFFFFu;                                    // smallest step q with H == M
    for (uint32_t c = c0 + (uint32_t)lane; c <= c1; c += 32u) {
        const Chunk ch = ld(rowbase + (uint64_t)c * chunk_stride<FM>(v));
        const uint64_t X = chunk_string<FM>(ch, v.half);
        int H = anchor_of<FM>(ch, v.half);
        for (int rem = FM::CS - 1; rem >= 0; --rem) {
            const uint32_t q = c * (uint32_t)FM::CS + (uint32_t)rem;
            if (H == M && q >= L + 1u && q <= L + v.n) cand = min(cand, q);
            const int off = FM::K * (FM::CS - 1 - rem);
            const int D = FM::K == 32 ? (int)(uint32_t)(X >> off) : (int)((uint32_t)(X >> off) & FM::MASK);
            H -= D + v.gap;
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) cand = min(cand, __shfl_xor_sync(0xFFFFFFFFu, cand, o));
    bj = cand - L;
}

} // namespace b2a
