// row_walk.h -- the short16 NW traceback, one DP row per iteration.
//
// Shared by short16_traceback_kernel<K,false> (device) and the CPU harness of tests/test_row_walker_cpu.py (host), so
// both execute the same function on the same record.  The generic cursor walker walk_global() in b2a_format.h stays the
// executable specification; this is the same decision per cell (hw2.cpp:145-153, or hw4.cpp:37-46), resolved for a whole
// window of one row at a fixed cost.
//
// Notation: D_i(j) = H(i,j) - H(i,j-1) - gap >= 0 is the stored field, V(j) = H(i,j) - H(i-1,j), s = match / mismatch.
//   'M'  <=>  H == diagonal  <=>  V(j) + D_{i-1}(j) + gap == s(i,j)
//   hw2: otherwise 'I' <=> D_i(j) == 0, else 'D';   hw4: otherwise 'D' <=> V(j) == gap, else 'I'.
// An 'I' move has D_i(j) == 0 (H came from the left), so along a run of 'I' moves  V(j-1) = V(j) + D_{i-1}(j):  once V is
// known at the run's first column, the run depends only on the two rows' fields, the text bytes and the one pattern byte.
//
// One iteration at (i, j): seek rows i and i-1 at column j (one chunk load + a popcount prefix from the anchor each; the
// lower row's chunk was the upper row's one iteration earlier, so it hits L1), load the text bytes T[j-8 .. j-1] as two
// aligned 8-byte words, then decide up to W columns j, j-1, ... with a fully unrolled branch-free scan that sets one stop
// bit per column (the run is the count of trailing zeros): no trip count that depends on the data, so the 32 walks of a
// warp stay converged.  The window stops at the nearer chunk edge of the two
// rows (rows i and i-1 may belong to different fill lanes, whose chunk edges are one column apart).  The iteration emits
// the window's run of 'I' moves and, if the run ends inside the window, its terminal 'M' or 'D', which climbs a row.
// A config-2 NW path (150 x 1000, linear gap) is a staircase of ~150 climbs with runs of ~4.5 'I' moves in between, so
// the walk takes ~190 iterations per pair where the per-cell walker took ~680 steps plus the run along the last row.
#pragma once
#include <stdint.h>
#include "b2a_format.h"

namespace b2a {

// one pair (one 16-bit half) of a short16 pair-pair record, global mode
struct RowWalkPair {
    const Chunk*   rec;         // the pair-pair's record: chunk (row i, c) at c*32R + (i-1)
    const uint8_t* P;           // pattern (rows)
    const uint8_t* T;           // text (columns); read as aligned 8-byte words, never outside the words holding T[0 .. n-1]
    uint32_t m, n;              // this pair's own shape (the record is laid out for the pair-pair's max(n))
    uint32_t R, rmagic;         // rows per lane, ceil(65536 / R)
    int half;                   // 0 = low 16 bits of every word, 1 = high
    int match, mismatch, gap, bias;
    bool hw4;                   // tie order d > u > l (hw4.cpp:37-46) and overlap := hw4's distance
};

// 2-bit op writer with bulk runs: op t of a pair lands in bits 2*(t%16) of word t/16 (traceback order)
struct OpsRunSink {
    uint32_t* out;              // may be null: ops are counted but not stored
    uint32_t word, fill, pos;
    B2A_HD explicit OpsRunSink(uint32_t* o) : out(o), word(0), fill(0), pos(0) {}
    B2A_HD void put(uint32_t op) {
        word |= op << (2u * fill);
        if (++fill == 16u) { if (out) out[pos] = word; ++pos; word = 0; fill = 0; }
    }
    B2A_HD void put_run(uint32_t op, uint32_t cnt) {
        while (cnt) {
            const uint32_t take = cnt < 16u - fill ? cnt : 16u - fill;
            if (op) word |= ((op * 0x55555555u) & (take == 16u ? 0xFFFFFFFFu : ((1u << (2u * take)) - 1u))) << (2u * fill);
            fill += take; cnt -= take;
            if (fill == 16u) { if (out) out[pos] = word; ++pos; word = 0; fill = 0; }
        }
    }
    B2A_HD void flush() { if (fill && out) out[pos] = word; }
};

// field string of one half of a short16 chunk (step rem at bit K*(CS-1-rem)) and its anchor
B2A_HD uint64_t s16_unpack(const Chunk& ch, int half, int& anchor) {
#if defined(__CUDA_ARCH__)
    const uint32_t sel_lo = half ? 0x7632u : 0x5410u, sel_hi = half ? 0x4432u : 0x4410u;
    const uint32_t lo = __byte_perm(ch.w2, ch.w1, sel_lo);           // (w1.half << 16) | w2.half
    const uint32_t hi = __byte_perm(ch.w0, 0u, sel_hi);              // w0.half
    anchor = (int)__byte_perm(ch.anchor, 0u, sel_hi);
    return ((uint64_t)hi << 32) | lo;
#else
    anchor = anchor_of<Short16<2>>(ch, half);
    return chunk_string<Short16<2>>(ch, half);                       // (the word layout does not depend on K)
#endif
}

// Seek row i >= 1 at column j: exact (biased) H(i,j), the field string shifted so that column j - t sits at bit K*t, and
// rem = the step of column j inside its chunk (columns j .. j-rem share the chunk).
template <int K, class Mem>
B2A_HD void rw_seek(const RowWalkPair& v, const Mem& mem, uint32_t i, uint32_t j, uint64_t& X, int& H, uint32_t& rem) {
    using FM = Short16<K>;
    const uint32_t x = i - 1u, L = (x * v.rmagic) >> 16;             // lane that owned the row in the fill (x / R, see row_slot)
    const uint32_t q = j + L, c = q / (uint32_t)FM::CS;
    rem = q - c * (uint32_t)FM::CS;
    int anchor;
    X = s16_unpack(mem.chunk(v.rec + x + (uint64_t)c * (32u * v.R)), v.half, anchor);
    const int off = K * (FM::CS - 1 - (int)rem);
    H = anchor - (FM::CS - 1 - (int)rem) * v.gap - field_sum64<K>(X & ((1ull << off) - 1ull));
    X >>= off;
}

// number of trailing zero bits (x != 0)
B2A_HD int ctz32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __ffs((int)x) - 1;
#else
    return __builtin_ctz(x);
#endif
}

// byte k (k = 0..7) of the result has bit 7 set iff byte k of x equals pc
B2A_HD uint64_t eq_bytes(uint64_t x, uint8_t pc) {
#if defined(__CUDA_ARCH__)
    const uint32_t p4 = pc * 0x01010101u;
    return ((uint64_t)__vcmpeq4((uint32_t)(x >> 32), p4) << 32) | __vcmpeq4((uint32_t)x, p4);
#else
    const uint64_t y = x ^ (pc * 0x0101010101010101ull);
    return ~(((y & 0x7F7F7F7F7F7F7F7Full) + 0x7F7F7F7F7F7F7F7Full) | y) & 0x8080808080808080ull;
#endif
}

// Needleman-Wunsch traceback of one pair (hw2.cpp:158-188 + overlapLongestExactMatch hw2.cpp:267-278, or hw4.cpp:52-68).
// Mem: Chunk chunk(const Chunk*) and uint64_t word8(const uint8_t* 8-byte aligned).  Returns the number of iterations.
template <int K, class Mem, class Sink>
B2A_HD uint32_t row_walk_global(const RowWalkPair& v, const Mem& mem, Sink& sink, PairResult& res) {
    using FM = Short16<K>;
    constexpr int W = FM::CS < 8 ? FM::CS : 8;                        // columns per window (the text window holds 8)
    uint32_t i = v.m, j = v.n, nops = 0, mism = 0, iters = 0;
    int cur = 0, best = 0;
    {
        uint64_t X; int H; uint32_t rem;
        rw_seek<K>(v, mem, i, j, X, H, rem);
        res.score = H - v.bias;                                       // hw2.cpp:186
    }
    const uintptr_t t0 = (uintptr_t)v.T & ~(uintptr_t)7;
    while (i > 0u && j > 0u) {
        ++iters;
        uint64_t Xa, Xb; int H, Hu; uint32_t ra, rb;
        rw_seek<K>(v, mem, i, j, Xa, H, ra);
        rw_seek<K>(v, mem, i > 1u ? i - 1u : 1u, j, Xb, Hu, rb);
        if (i == 1u) { Hu = v.bias + (int)j * v.gap; Xb = 0; rb = W - 1; }     // border row 0: D = 0 (hw2.cpp:131-136)
        // text bytes T[j-1-t] for t = 0..7: byte 7-t of E
        const uint32_t x = j - 1u;
        const uintptr_t a = ((uintptr_t)v.T + x) & ~(uintptr_t)7;
        const uint32_t sh = (uint32_t)((uintptr_t)v.T + x - a);
        const uint64_t hi = mem.word8((const uint8_t*)a);
        const uint64_t lo = mem.word8((const uint8_t*)(a == t0 ? a : a - 8u));   // (a == t0: the window holds no byte left of a)
        const uint64_t E = sh == 7u ? hi : (lo >> (8u * (sh + 1u))) | (hi << (56u - 8u * sh));
        const uint8_t pc = v.P[i - 1u];
        const uint64_t Z = eq_bytes(E, pc);
        uint32_t lim = ra < rb ? ra : rb;
        if (x < lim) lim = x;
        if (lim > W - 1u) lim = W - 1u;                               // window: columns j - lim .. j
        // every column's decision as if the run reached it (V accumulates unconditionally: past the first stop it is
        // meaningless and unused); the run is the number of columns before the first stop, bit lim+1 ends the window
        int V = H - Hu;
        uint32_t stops = 1u << (lim + 1u), diag = 0;
#pragma unroll
        for (int t = 0; t < W; ++t) {
            const int du = (int)((uint32_t)(Xb >> (K * t)) & FM::MASK);
            const int da = (int)((uint32_t)(Xa >> (K * t)) & FM::MASK);
            const bool eq = (Z >> (8 * (7 - t) + 7)) & 1u;
            const bool isM = V + du + v.gap == (eq ? v.match : v.mismatch);
            const bool stop = isM || (v.hw4 ? V == v.gap : da != 0);
            stops |= (uint32_t)stop << t;
            diag |= (uint32_t)isM << t;
            V += du;
        }
        const uint32_t run = (uint32_t)ctz32(stops);
        const bool term = run <= lim;                                 // else the window is exhausted: the run goes on next iteration
        const uint32_t op = (diag >> run) & 1u ? OP_M : OP_D;
        const bool eqt = (Z >> (8u * (7u - (run & 7u)) + 7u)) & 1u;
        sink.put_run(OP_I, run); nops += run; j -= run;
        if (run) cur = 0;
        if (term) {
            mism += (op == OP_M && !eqt);
            cur = (op == OP_M && eqt && pc != (uint8_t)'-') ? cur + 1 : 0;   // hw2.cpp:267-278
            best = cur > best ? cur : best;
            sink.put(op); ++nops;
            --i; j -= op == OP_M;
        }
    }
    sink.put_run(OP_D, i); nops += i;                                 // column 0 holds 'u' (hw2.cpp:128)
    sink.put_run(OP_I, j); nops += j;                                 // row 0 holds 'l'    (hw2.cpp:134)
    res.end_i = v.m; res.end_j = v.n; res.start_i = 0; res.start_j = 0; res.n_ops = nops;
    res.overlap = v.hw4 ? (int)(nops - (v.m + v.n - nops) + mism) : best;   // gap columns = n_ops - M columns, M columns = m + n - n_ops
    return iters;
}

} // namespace b2a
