// wide32.cuh -- int32 kernel family: intra-pair tiled anti-diagonal wavefront for pairs the s16x2
// record cannot hold (long patterns, general byte alphabets, large scores).
//
// Replaces the same reference loops as short16 (hw2.cpp:138-156 / :205-231) for ONE pair spread over
// many warps: the DP matrix is cut into BANDS of 128 pattern rows (32 lanes x 4 rows); a warp sweeps
// its band along the text as a skewed wavefront (__shfl_up_sync carries the in-warp diagonal
// dependency) and hands the band's bottom row to the band below through L2 as SELF-VALIDATING 64-bit
// entries {H, tag}: value and validity travel in one atomic word, so neither side needs a fence or a
// separate progress flag (an earlier st.release/ld.acquire counter design spent 60 % of a single long
// pair's time in membar/long-scoreboard stalls, profiles/r01_ncu_wide32_c4.md).  The consumer loads
// its column of the next 32-column block one block ahead and only re-polls if the tag is not there yet.
// tag = epoch * 2^20 + band + 1: the two boundary buffers of a pair alternate between bands, the epoch
// changes with every launch, the host clears the buffers when the epoch wraps or the buffer moves.
// Bands are handed out by a ticket counter in (band, pair) order, so the band a warp waits for was
// always claimed earlier by a warp that is already running: no cooperative launch is needed and
// nothing can deadlock.
// The traceback record is the same delta/anchor chunk format as short16 (b2a_format.h, Wide32<K>),
// written with the same ring-arithmetic word trick; K = 32 stores raw deltas and covers any scoring.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "b2a_format.h"
#include "short16_fill.cuh"
#include "walk_warp.cuh"

namespace b2a {

struct WidePair {
    uint64_t pat_off, txt_off;      // byte offsets of the pair's sequences
    uint64_t code_off;              // first chunk of the pair's record
    uint64_t bound_off;             // entry index of the pair's 2 boundary rows (each bound_stride long); multi-band pairs only
    uint64_t rowbest_off;           // uint32 index, nbands*128 entries
    uint32_t m, n, pair, nbands;
    uint32_t bound_stride;
    // ---- checkpointed long pairs (b2a_api.cu wide_ckpt): the pair may be a SUB-PROBLEM, rows row_base+1 .. row_base+m of a longer pattern ----
    uint32_t row_base;              // rows above the sub-problem (0 for a whole pair): the left border is H(i, 0) = (row_base + i) gap
    uint64_t top_off;               // index into WideArgs::ck of the stored row above row 1 (entries 0..n); ~0 = the real border row 0
    uint64_t ck_off;                // where this launch keeps checkpoint rows: ck[ck_off + (g * ck_stride) + j] = H((g + 1) ck_every bands, j)
    uint32_t ck_every, ck_stride;   // keep the bottom row of every ck_every-th band (0 = none); entries per kept row
    // a sub-problem may also start at a kept COLUMN: columns col_base+1 .. col_base+n of a longer text
    uint32_t col_base;              // columns left of the sub-problem (0 for a whole pair): the top border is H(0, j) = (col_base + j) gap
    uint32_t col_shift;             // pass 1 keeps every 2^col_shift-th column (0 = none) ...
    uint64_t left_off;              // index into WideArgs::ck of the stored column left of column 1 (one entry per row of the sub-problem); ~0 = none
    uint64_t colck_off;             // ... at ck[colck_off + (j / 2^col_shift - 1) * col_stride + row]
    uint32_t col_stride, pad;
};
constexpr uint64_t WIDE_NO_TOP = ~0ull;
struct WideTask { uint32_t wp, band; };

struct WideArgs {
    const uint8_t*  pat;
    const uint8_t*  txt;
    const WidePair* pairs;
    const WideTask* tasks;
    uint32_t        n_tasks;
    uint32_t*       ticket;
    Chunk*          codes;
    uint64_t*       bound;          // tagged boundary entries: (tag << 32) | (uint32) H
    uint32_t*       rowbest;
    int32_t*        final_score;    // per wide pair: H(m, n) (global mode)
    int32_t         match, mismatch, gap;
    uint32_t        radix;
    uint32_t        epoch_tag;      // epoch << 20
    int32_t*        ck;             // checkpoint rows (plain int32 H values), see WidePair
    const AlphaInfo* alpha;         // used by the ALPHA4 variant only
    int32_t*        final_col;      // per wide pair, semi-global mode: j* (final_score then holds H(m, j*))
};

constexpr int WIDE_WARPS = 4;
#ifndef WIDE_MID_UNROLL
#define WIDE_MID_UNROLL 32     // unroll of the F-2 middle steps of a delta word (tuned on config 4 / config 5, bench.py --config c4 / c5)
#endif
constexpr int MID_UNROLL = WIDE_MID_UNROLL;

__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p));       // no "memory" clobber: nothing else is ordered by it
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(uint64_t* p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v));
}
// Waits until this lane's tagged boundary entry (if it `need`s one) carries `tag`; `v` is a copy loaded a block
// earlier.  WARP-UNIFORM on purpose: every lane leaves the loop in the same iteration (__all_sync).  A per-lane
// polling loop left the warp split into sub-warps that then executed the whole next block of shuffle-synchronised
// steps one group after the other (3.5x slower first block of every band, measured with per-band globaltimer stamps in round 1).
// Re-polls back off so that hundreds of waiting bands of one long pair do not flood L2.
__device__ __forceinline__ uint32_t bound_wait(const uint64_t* p, uint64_t v, uint32_t tag, bool need) {
    uint32_t ns = 32;
    for (;;) {
        const bool ok = !need || (uint32_t)(v >> 32) == tag;
        if (__all_sync(0xFFFFFFFFu, ok)) break;
        __nanosleep(ns); ns = min(ns * 2u, 256u);
        if (!ok) v = ld_relaxed_u64(p);
    }
    return (uint32_t)v;
}
__device__ __forceinline__ uint32_t prmt32(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// K: delta width; LOCAL: Smith-Waterman; STORE: write the traceback record; ALPHA4: pattern alphabet
// has <= 4 symbols and scores fit int8, so the substitution score is one PRMT from a 4-entry table.
//
// A lane owns R rows and computes them C columns at a time (a register tile of R x C cells per MACRO-STEP): the bottom-row values of
// the lane above for those C columns arrive through C independent shuffles and the tile's cells form a small wavefront of their own.
// C = 1 for every launch that writes a record (the lanes follow each other one column apart); C = 4 for the score-only launches, where
// many pairs are in flight and the tile's shorter instruction stream per cell pays (config 5 linear: 3684 -> 4001 GCUPS).  For ONE long
// pair C = 4 is slower (measured, see b2a_format.h wide_skew).
// KEEPCOL: pass 1 of a checkpointed pair, which also keeps every 2^col_shift-th column (a test in the innermost loop: 4 % on the 120-pair
// score-only launch when it was a run-time flag, so only that pass instantiates it).
// SEMI (with LOCAL = false): semi-global mode.  Row 0 is free (H(0, j) = 0), the interior is NW's (no floor), and the lane holding
// row m tracks the first strict maximum of that row as it sweeps (columns 0..n) -> final_score / final_col, which serves the
// score-only launches too.  Whole pairs only: checkpointed pairs are refused by the host for this mode.
template <int K, bool LOCAL, bool STORE, bool ALPHA4, bool KEEPCOL = false, bool SEMI = false>
__global__ void __launch_bounds__(WIDE_WARPS * 32)
wide32_fill_kernel(const WideArgs A)
{
    static_assert(!(LOCAL && SEMI) && !(KEEPCOL && SEMI), "semi-global: whole pairs, NW cells");
    using FM = Wide32<K>;
    constexpr int C = STORE ? FM::SKEW : WIDE_TILE_SCORE_ONLY;                   // score-only launches (instantiated with K = 2) use the tile
    static_assert(STORE || K == 2, "score-only kernels are launched with K = 2: no record, the word structure only paces the loop");
    constexpr int R = WIDE_R, F = FM::F, CS = FM::CS, CPB = 32 / CS;               // CPB: chunks per 32-step block
    constexpr uint32_t RING = C == 1 ? 64u : 256u, RMASK = RING - 1u;               // live columns of a block: [q0 - 31 C, q0 + 31]
    static_assert(32 * C + 32 <= (int)RING, "ring too small for the lane skew");
    __shared__ __align__(16) uint2 s_ring[WIDE_WARPS][RING];   // per 1-based column j (slot j & RMASK): {text entry, H(top row, j)}
    __shared__ int32_t s_out[WIDE_WARPS][32];                  // bottom-row values lane 31 produced during the current block
    __shared__ uint32_t s_tbl4[256];
    uint8_t sym[4] = {0, 0, 0, 0};
    if (ALPHA4) {
        const int nsym = A.alpha->nsym;
#pragma unroll
        for (int c = 0; c < 4; ++c) sym[c] = A.alpha->sym[c];
        for (int b = threadIdx.x; b < 256; b += blockDim.x) {
            uint32_t w = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int sc = (c < nsym && sym[c] == (uint8_t)b) ? A.match : A.mismatch;
                w |= ((uint32_t)sc & 0xFFu) << (8 * c);
            }
            s_tbl4[b] = w;
        }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint2* ring = s_ring[warp];
    int32_t* outb = s_out[warp];
    const int gap = A.gap;
    const uint32_t radix = A.radix, g32 = (uint32_t)gap;
    uint32_t geo = 0, bpow = 1;
    if (K < 32) {
#pragma unroll
        for (int t = 0; t < F; ++t) geo = geo * radix + 1u;
#pragma unroll
        for (int t = 0; t < F - 1; ++t) bpow *= radix;
    }
    const uint32_t negGc = 0u - g32 * geo, negBpow = 0u - bpow, radm1 = radix - 1u;

    for (;;) {
        uint32_t tk = 0;
        if (lane == 0) tk = atomicAdd(A.ticket, 1u);
        tk = __shfl_sync(0xFFFFFFFFu, tk, 0);
        if (tk >= A.n_tasks) break;
        const WideTask task = A.tasks[tk];
        const WidePair wp = A.pairs[task.wp];
        const uint32_t m = wp.m, n = wp.n, band = task.band;
        const uint8_t* pp = A.pat + wp.pat_off;
        const uint8_t* tt = A.txt + wp.txt_off;
        const uint32_t row0 = band * 32u * R + (uint32_t)lane * R;          // 0-based first row of this lane
        uint32_t pc[R];
        int32_t H[R], best[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const uint32_t i0 = row0 + r;
            if (ALPHA4) {
                uint32_t c = 0;
                if (i0 < m) { const uint8_t x = pp[i0];
#pragma unroll
                    for (int k = 1; k < 4; ++k) if (x == sym[k]) c = k; }
                pc[r] = c | ((8u | c) << 4) | ((8u | c) << 8) | ((8u | c) << 12);
            } else pc[r] = i0 < m ? (uint32_t)pp[i0] : 0xFFFFFFFFu;         // junk rows never match
            H[r] = LOCAL ? 0 : (int32_t)(wp.row_base + i0 + 1) * gap;        // hw2.cpp:125-130
            if (wp.left_off != WIDE_NO_TOP && i0 < m) H[r] = A.ck[wp.left_off + i0];   // sub-problem at a kept column: the stored H(i, col_base)
            best[r] = 0;
        }
        const uint64_t* bin = A.bound + wp.bound_off + (uint64_t)((band + 1u) & 1u) * wp.bound_stride;
        uint64_t* bout = A.bound + wp.bound_off + (uint64_t)(band & 1u) * wp.bound_stride;
        const uint32_t tag_in = A.epoch_tag + band;                          // what the band above writes
        const uint64_t tag_out = (uint64_t)(A.epoch_tag + band + 1u) << 32;
        const bool has_next = band + 1 < wp.nbands;
        const uint32_t nblk = (n + 31u * C + 1u + 31u) / 32u;                // lane 31 reaches column n at step n + 31 C
        const uint32_t NC = num_chunks(n, CS, C);
        Chunk* rec = A.codes + wp.code_off;
        const int32_t* top = wp.top_off != WIDE_NO_TOP ? A.ck + wp.top_off : nullptr;      // band 0 of a sub-problem reads the row above it
        // H(row above the band, column 0 of the (sub-)problem): a border cell, or a kept value when the sub-problem starts inside the matrix
        int32_t top0 = LOCAL ? 0 : (int32_t)(wp.row_base + band * 32u * R + wp.col_base) * gap;   // row_base or col_base is 0 whenever this formula is used
        if (band == 0) { if (top) top0 = top[0]; }
        else if (wp.left_off != WIDE_NO_TOP) top0 = A.ck[wp.left_off + band * 32u * R - 1u];
        int32_t dgn = top0;                                                  // bottom row of the lane above, one column left of the tile
        int32_t outv[C];                                                     // this lane's bottom row at the C columns of its last tile
#pragma unroll
        for (int c = 0; c < C; ++c) outv[c] = H[R - 1];                      // before its first column a lane shows its border value
        // SEMI: row m (0-based im inside the last band) belongs to lane im / R, register im % R; its best starts at column 0
        const uint32_t im = m - 1u - band * 32u * R;
        const bool own_m = SEMI && band + 1u == wp.nbands && (uint32_t)lane == im / R;
        const uint32_t rm = im % R;
        int32_t ebest = (int32_t)m * gap;
        uint32_t ej = 0;
        uint64_t nx = 0;                                                     // this lane's entry of the next block, loaded a block ahead
        if (band != 0 && lane >= 1 && (uint32_t)lane <= n) nx = ld_relaxed_u64(bin + lane);

        // text byte of 1-based column j, fetched one block ahead (0x100 = outside the text); the score-table
        // lookup waits until the byte is staged, so the global load has a whole block to arrive
        auto text_byte = [&](uint32_t j) -> uint32_t { return (j == 0 || j > n) ? 0x100u : (uint32_t)tt[j - 1]; };
        auto text_entry = [&](uint32_t x) -> uint32_t {                      // ring payload
            if (x & 0x100u) return ALPHA4 ? 0u : 0xFFFFFF00u;
            return ALPHA4 ? s_tbl4[x] : x;
        };
        uint32_t tnext = text_byte((uint32_t)lane);

        for (uint32_t kb = 0; kb < nblk; ++kb) {
            const uint32_t q0 = kb * 32u;
            // ---- stage columns q0 .. q0+31 of the text and of the band above into the ring ----
            int32_t bnd;
            const uint32_t jcol = q0 + (uint32_t)lane;
            if (band == 0) {
                if (top) bnd = (jcol >= 1 && jcol <= n) ? top[jcol] : top0;
                else bnd = (LOCAL || SEMI) ? 0 : (int32_t)(wp.col_base + jcol) * gap;  // hw2.cpp:131-136; semi-global: free row 0
            } else {
                const bool need = jcol >= 1 && jcol <= n;
                const int32_t got = (int32_t)bound_wait(bin + jcol, nx, tag_in, need);
                bnd = need ? got : top0;
                const uint32_t jn = jcol + 32u;
                if (jn <= n) nx = ld_relaxed_u64(bin + jn);
            }
            __syncwarp();
            ring[jcol & RMASK] = make_uint2(text_entry(tnext), (uint32_t)bnd);
            __syncwarp();
            tnext = text_byte(q0 + 32u + (uint32_t)lane);                    // prefetch the next block's text
            // RAMP = false: every lane is inside its column range for the whole block (steady state).  RAMP = true: lanes
            // outside 1 <= j <= n keep their H frozen -- done with selects, NOT a branch: a branch per step stops
            // the scheduler from overlapping the shuffle / shared-memory latencies of neighbouring steps (2.4x slower).
            const bool steady = q0 >= 31u * C + 1u && q0 + 31u <= n;
            // One macro-step: the tile of R rows x C columns at lane-steps qm .. qm + C - 1 (columns qm - lane C + c).
            // POS: where the C steps sit inside their delta word: 0 = first, 1 = middle, 2 = last, 3 = the whole word.
            auto macro = [&](uint32_t qm, uint32_t (&S)[R], auto pos_tag, auto ramp_tag) {
                constexpr bool RAMP = decltype(ramp_tag)::value;
                constexpr int POS = decltype(pos_tag)::value;
                const uint32_t j0 = qm - (uint32_t)lane * C;                 // may wrap below zero: such columns are inactive
                uint2 e[C];
                if (C == 4) {
                    const uint4* e4 = reinterpret_cast<const uint4*>(ring + (j0 & RMASK));   // j0 is a multiple of 4: 32-byte aligned
                    const uint4 lo = e4[0], hi = e4[1];
                    e[0] = make_uint2(lo.x, lo.y); e[1 % C] = make_uint2(lo.z, lo.w); e[2 % C] = make_uint2(hi.x, hi.y); e[3 % C] = make_uint2(hi.z, hi.w);
                } else {
#pragma unroll
                    for (int c = 0; c < C; ++c) e[c] = ring[(j0 + (uint32_t)c) & RMASK];
                }
                int32_t upv[C];
#pragma unroll
                for (int c = 0; c < C; ++c) upv[c] = __shfl_up_sync(0xFFFFFFFFu, outv[c], 1);
                if (lane == 0) {
#pragma unroll
                    for (int c = 0; c < C; ++c) upv[c] = (int32_t)e[c].y;    // the band above (or the border row 0); also H(top, 0) at column 0
                }
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const bool active = !RAMP || (uint32_t)(j0 + (uint32_t)c - 1u) < n;
                    int32_t dg = dgn, u = upv[c];
                    dgn = upv[c];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const int32_t s = ALPHA4 ? (int32_t)prmt32(e[c].x, 0u, pc[r]) : (pc[r] == e[c].x ? A.match : A.mismatch);
                        const int32_t ds = dg + s;
                        dg = H[r];
                        const int32_t a = __viaddmax_s32(H[r], gap, ds);
                        int32_t h = LOCAL ? __viaddmax_s32_relu(u, gap, a) : __viaddmax_s32(u, gap, a);
                        if (RAMP) h = active ? h : H[r];
                        if (LOCAL) best[r] = max(best[r], h);    // a frozen H is a border 0 or a value already counted
                        H[r] = h; u = h;
                    }
                    if (SEMI) {                                                  // first strict maximum of row m, left to right
                        int32_t hv = H[0];
#pragma unroll
                        for (int r = 1; r < R; ++r) if (rm == (uint32_t)r) hv = H[r];
                        const uint32_t jc = j0 + (uint32_t)c;
                        if (own_m && jc - 1u < n && hv > ebest) { ebest = hv; ej = jc; }
                    }
                    outv[c] = H[R - 1];
                    if (lane == 31) outb[(qm + (uint32_t)c) & 31u] = H[R - 1];   // bottom row of the band (published per block)
                    if (KEEPCOL) {                                               // pass 1 of a checkpointed pair: keep every 2^col_shift-th column
                        const uint32_t jc = j0 + (uint32_t)c;
                        if ((jc & ((1u << wp.col_shift) - 1u)) == 0u && jc - 1u < n) {
#pragma unroll
                            for (int r = 0; r < R; ++r)
                                if (row0 + r < m) A.ck[wp.colck_off + (uint64_t)((jc >> wp.col_shift) - 1u) * wp.col_stride + row0 + r] = H[r];
                        }
                    }
                    // what the step contributes to the delta word's Horner sum: start it (S = H), S = S * 2^K + H, or nothing (last step)
                    constexpr bool first_of_word = (POS == 0 || POS == 3);
                    constexpr bool last_of_word = (POS == 2 || POS == 3);
                    const bool is_first = first_of_word && c == 0, is_last = last_of_word && c == C - 1;
                    if (STORE && K < 32 && !(is_last && F > 1) && F > 1) {
#pragma unroll
                        for (int r = 0; r < R; ++r) S[r] = is_first ? (uint32_t)H[r] : S[r] * radix + (uint32_t)H[r];
                    }
                }
            };
            // The F steps of one delta word = F / C macro-steps.  Deliberately NOT one straight-line block per chunk: fully unrolled
            // the two flavours were 38 KB of code and every band of a long pair paid ~6 us of instruction-fetch stalls for its first
            // (cold) ramp block -- a cost that chains over all bands of the pair.
            auto word_steps = [&](uint32_t qw, uint32_t (&S)[R], auto ramp_tag) {
                if (F <= C) { macro(qw, S, std::integral_constant<int, 3>{}, ramp_tag); return; }
                macro(qw, S, std::integral_constant<int, 0>{}, ramp_tag);
#pragma unroll MID_UNROLL
                for (int f = C; f < F - C; f += C) macro(qw + (uint32_t)f, S, std::integral_constant<int, 1>{}, ramp_tag);
                macro(qw + (uint32_t)(F - C), S, std::integral_constant<int, 2>{}, ramp_tag);
            };

#pragma unroll 1
            for (int cb = 0; cb < CPB; ++cb) {
                uint32_t w0[R];
#pragma unroll
                for (int wi = 0; wi < 2; ++wi) {
                    uint32_t S[R], pre[R];
#pragma unroll
                    for (int r = 0; r < R; ++r) pre[r] = K == 32 ? (0u - (uint32_t)H[r] - g32) : (uint32_t)H[r] * negBpow + negGc;
                    const uint32_t qw = q0 + (uint32_t)(cb * CS + wi * F);
                    // Both flavours are straight-line code of the same speed: the last blocks of band b wait for the last
                    // block of band b-1, so a slow ramp flavour is paid once PER BAND on the critical path of a long pair.
                    if (steady) word_steps(qw, S, std::false_type{});
                    else word_steps(qw, S, std::true_type{});
                    if (STORE) {
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const uint32_t w = (K < 32 && F > 1 ? S[r] * radm1 : 0u) + (uint32_t)H[r] + pre[r];
                            if (wi == 0) w0[r] = w;
                            else {
                                const uint32_t c = kb * CPB + cb;
                                if (c < NC) {
                                    const uint4 v = make_uint4(w0[r], w, 0u, (uint32_t)H[r]);
                                    *reinterpret_cast<uint4*>(&rec[(((uint64_t)band * R + r) * NC + c) * 32u + lane]) = v;
                                }
                            }
                        }
                    }
                }
            }
            // publish the 32 bottom-row values of this block as tagged entries: ONE coalesced 64-bit store per lane
            // per block instead of a store per step (the per-step stores cost 8 % on the 120 x 100 kb batch)
            if (has_next) {
                __syncwarp();
                const uint32_t jc = q0 + (uint32_t)lane - 31u * C;            // lane 31 was at this column at step q0 + lane
                if (jc - 1u < n) st_relaxed_u64(bout + jc, tag_out | (uint32_t)outb[lane]);
                // checkpointed long pairs: every ck_every-th band also keeps its bottom row (columns 0..n) for the re-fill pass
                if (wp.ck_every && (band + 1u) % wp.ck_every == 0u && jc <= n)
                    A.ck[wp.ck_off + (uint64_t)((band + 1u) / wp.ck_every - 1u) * wp.ck_stride + jc] = outb[lane];
                __syncwarp();
            }
        }
        if (LOCAL) {
#pragma unroll
            for (int r = 0; r < R; ++r) A.rowbest[wp.rowbest_off + ((uint64_t)band * R + r) * 32u + lane] = (uint32_t)best[r];
        } else if (band + 1 == wp.nbands) {
            const uint32_t ib = (m - 1u) - band * 32u * R;
            if ((uint32_t)lane == ib / R) {
                const uint32_t rm = ib % R;
                int32_t v = H[0];
#pragma unroll
                for (int r = 1; r < R; ++r) if (rm == (uint32_t)r) v = H[r];
                if (SEMI) { A.final_score[task.wp] = ebest; A.final_col[task.wp] = (int32_t)ej; }
                else A.final_score[task.wp] = v;
            }
        }
        __syncwarp();
    }
}

// ---- traceback over the wide32 record: one thread per pair ----
struct WideTbArgs {
    const uint8_t*  pat;
    const uint8_t*  txt;
    const WidePair* pairs;
    uint32_t        n_wide;
    const Chunk*    codes;
    const uint32_t* rowbest;
    const int32_t*  final_score;
    PairResult*     results;
    uint32_t*       ops;
    const uint64_t* ops_off;
    int32_t         match, mismatch, gap;
    int32_t         score_only;
    int32_t         opt;            // bit 2 (value 4): hw4 tie order d > u > l, overlap := hw4's distance
    const int32_t*  final_col;      // semi-global mode: end column j* per wide pair
};

struct WideLoader {
    const Chunk* base;
    __device__ __forceinline__ Chunk operator()(uint64_t idx) const {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(base + idx));
        return Chunk{v.x, v.y, v.z, v.w};
    }
    __device__ __forceinline__ void prefetch(uint64_t idx) const {
        asm volatile("prefetch.global.L2 [%0];" :: "l"(base + idx));
    }
};

constexpr int WIDE_TB_WARPS = 2;

// One WARP per pair (walk_warp.cuh); score-only batches just gather the scores the fill kernel left.
// SEMI (with LOCAL = false): semi-global, from (m, j*) up to row 0; m = 0 or n = 0 never reach the fill (no bands).
template <int K, bool LOCAL, bool SEMI = false>
__global__ void __launch_bounds__(WIDE_TB_WARPS * 32)
wide32_traceback_kernel(const WideTbArgs A)
{
    using FM = Wide32<K>;
    const int lane = (int)(threadIdx.x & 31u);
    const uint32_t t = blockIdx.x * WIDE_TB_WARPS + (threadIdx.x >> 5);
    if (t >= A.n_wide) return;
    const WidePair wp = A.pairs[t];
    PairResult res;
    if (A.score_only) {
        res = PairResult{0, 0, 0, 0, 0, 0, 0, 2};
        if (LOCAL) {
            int M = 0;
            for (uint32_t k = (uint32_t)lane; k < wp.nbands * 32u * WIDE_R; k += 32u) {   // k = (band*R + r)*32 + L; rows beyond m are junk
                const uint32_t L = k & 31u, br = k >> 5, r = br % WIDE_R, band = br / WIDE_R;
                if (band * 32u * WIDE_R + L * WIDE_R + r >= wp.m) continue;
                M = max(M, (int)A.rowbest[wp.rowbest_off + k]);
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) M = max(M, __shfl_xor_sync(0xFFFFFFFFu, M, o));
            res.score = M;
        } else if (SEMI) {
            const bool cells = wp.m && wp.n;
            res.score = cells ? A.final_score[t] : (int32_t)wp.m * A.gap; res.end_i = wp.m; res.end_j = cells ? (uint32_t)A.final_col[t] : 0u;
        } else { res.score = (wp.m && wp.n) ? A.final_score[t] : (int32_t)(wp.m + wp.n) * A.gap; res.end_i = wp.m; res.end_j = wp.n; }
        if (lane == 0) A.results[wp.pair] = res;
        return;
    }
    const Chunk* rec = A.codes + wp.code_off;
    const PairView v{rec, A.rowbest + wp.rowbest_off, A.pat + wp.pat_off, A.txt + wp.txt_off,
                     wp.m, wp.n, num_chunks(wp.n, FM::CS, FM::SKEW), WIDE_R, 0, A.match, A.mismatch, A.gap, 0, A.opt, 0};
    const WideLoader ld{rec};
    WarpOpsSink sink(A.ops ? A.ops + A.ops_off[wp.pair] : nullptr, lane == 0);
    uint32_t i, j, nops = 0, mism = 0;
    int best = 0, cur = 0;
    if (LOCAL) {
        int M; uint32_t bi, bj;
        warp_find_local_end<FM>(v, ld, M, bi, bj);
        res.score = M; res.end_i = bi; res.end_j = bj;
        i = bi; j = bj;
        if (M != 0) warp_walk<FM, WideLoader, true>(v, ld, sink, i, j, nops, best, mism, cur);
    } else if (SEMI) {
        const bool cells = wp.m && wp.n;
        i = wp.m; j = cells ? (uint32_t)A.final_col[t] : 0u;
        res.end_i = i; res.end_j = j;
        res.score = cells ? A.final_score[t] : (int32_t)i * A.gap;
        warp_walk<FM, WideLoader, false, true>(v, ld, sink, i, j, nops, best, mism, cur);
        sink.put_run(OP_D, i); nops += i; i = 0;                                           // column 0 holds 'u'; row 0 is free: no 'I' tail
    } else {
        i = wp.m; j = wp.n;
        res.end_i = i; res.end_j = j;
        res.score = (i && j) ? A.final_score[t] : (int32_t)(i + j) * A.gap;               // hw2.cpp:186 / borders :125-136
        warp_walk<FM, WideLoader, false>(v, ld, sink, i, j, nops, best, mism, cur);
        sink.put_run(OP_D, i); nops += i; i = 0;                                           // column 0 holds 'u' (hw2.cpp:128)
        sink.put_run(OP_I, j); nops += j; j = 0;                                           // row 0 holds 'l'    (hw2.cpp:134)
    }
    sink.flush();
    res.start_i = i; res.start_j = j; res.n_ops = nops; res.path = 2;
    res.overlap = (!LOCAL && (A.opt & 4)) ? (int)(nops - (wp.m + wp.n - nops) + mism) : best;       // hw4.cpp:141-152
    if (lane == 0) A.results[wp.pair] = res;
}

// ---- checkpointed long pairs: the walk of one pair, carried across its sub-problems (b2a_api.cu wide_ckpt_run) ----
struct CkptWalk {
    uint32_t i, j;              // current cell, ABSOLUTE row / column
    uint32_t nops, mism;
    int32_t  cur, best;         // open / longest exact-match run (hw2.cpp:267-278)
    uint32_t word, fill;        // 2-bit op writer
    uint64_t pos;
    int32_t  score, done;
    uint32_t end_i, end_j;
};
struct CkptWalkArgs {
    const uint8_t*  pat;
    const uint8_t*  txt;
    const WidePair* pair;       // the sub-problem that has just been filled (record at codes + code_off)
    const Chunk*    codes;
    const uint32_t* rowbest;
    const int32_t*  ck;
    CkptWalk*       st;
    PairResult*     result;     // the pair's record, written when the walk is complete
    uint32_t*       ops;        // the pair's op words, may be null
    uint32_t        m_total, n_total;
    int32_t         match, mismatch, gap, opt;
    int32_t         first;      // local mode: this sub-problem holds the end cell; find it (hw2.cpp:225-229) before walking
};

// first row of the first row-major maximum (hw2.cpp:225-229) from the per-row maxima of a whole-pair score-only fill: st->i / st->score
__global__ void __launch_bounds__(32) wide32_first_best_row_kernel(const uint32_t* __restrict__ rowbest, uint32_t m, CkptWalk* st)
{
    const uint32_t lane = threadIdx.x & 31u;
    int mloc = 0; uint32_t iloc = 0xFFFFFFFFu;
    for (uint32_t i = lane + 1u; i <= m; i += 32u) {
        const uint32_t x = i - 1u;
        const int rb = (int)rowbest[(uint64_t)((x >> 7) * 4u + (x & 3u)) * 32u + ((x >> 2) & 31u)];   // [(band R + r) 32 + L], R = 4
        if (rb > mloc) { mloc = rb; iloc = i; }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const int om = __shfl_xor_sync(0xFFFFFFFFu, mloc, o);
        const uint32_t oi = __shfl_xor_sync(0xFFFFFFFFu, iloc, o);
        if (om > mloc || (om == mloc && oi < iloc)) { mloc = om; iloc = oi; }
    }
    if (lane == 0) { st->score = mloc; st->i = mloc ? iloc : 0u; }
}

template <int K, bool LOCAL>
__global__ void __launch_bounds__(32) wide32_ckpt_walk_kernel(const CkptWalkArgs A)
{
    using FM = Wide32<K>;
    const int lane = (int)(threadIdx.x & 31u);
    const WidePair wp = *A.pair;
    CkptWalk s = *A.st;
    const Chunk* rec = A.codes + wp.code_off;
    PairView v{rec, A.rowbest + wp.rowbest_off, A.pat + wp.pat_off, A.txt + wp.txt_off,
               wp.m, wp.n, num_chunks(wp.n, FM::CS, FM::SKEW), WIDE_R, 0, A.match, A.mismatch, A.gap, 0, A.opt, 0};
    v.top = wp.top_off != WIDE_NO_TOP ? A.ck + wp.top_off : nullptr;
    if (!LOCAL && !v.top) v.bias = (int)wp.col_base * A.gap;        // the real border row 0, seen from column col_base: H(0, j) = (col_base + j) gap
    const WideLoader ld{rec};
    WarpOpsSink sink(A.ops, lane == 0);
    sink.word = s.word; sink.fill = s.fill; sink.pos = s.pos;
    uint32_t i = s.i - wp.row_base, j = s.j - wp.col_base;       // the sub-problem's own row / column index
    int best = s.best, cur = s.cur;
    bool walk = true;
    if (LOCAL && A.first) {
        int M; uint32_t bi, bj;
        warp_find_local_end<FM>(v, ld, M, bi, bj);                // rows above this sub-problem hold no earlier maximum: the first pass chose row s.i
        s.score = M; s.end_i = wp.row_base + bi; s.end_j = wp.col_base + bj;
        i = bi; j = bj;
        if (M == 0) { s.end_i = s.end_j = 0; i = 0; j = 0; walk = false; s.done = 1; }
    }
    if (walk) {
        warp_walk<FM, WideLoader, LOCAL>(v, ld, sink, i, j, s.nops, best, s.mism, cur);
        if (LOCAL) {
            // stopped inside the sub-problem (H == 0), or at the real left / top border: the alignment is complete (hw2.cpp:239)
            if ((i > 0 && j > 0) || (j == 0 && wp.col_base == 0) || (i == 0 && wp.row_base == 0)) s.done = 1;
        } else if (j == 0 && wp.col_base == 0) {
            const uint32_t up = wp.row_base + i;                 // column 0 holds 'u' all the way up (hw2.cpp:128)
            sink.put_run(OP_D, up); s.nops += up; i = 0; s.done = 2;
        } else if (i == 0 && wp.row_base == 0) {
            const uint32_t lf = wp.col_base + j;                 // row 0 holds 'l' all the way left (hw2.cpp:134)
            sink.put_run(OP_I, lf); s.nops += lf; j = 0; s.done = 3;
        }
    }
    s.i = s.done == 2 ? 0u : wp.row_base + i; s.j = s.done == 3 ? 0u : wp.col_base + j; s.best = best; s.cur = cur;
    s.word = sink.word; s.fill = sink.fill; s.pos = sink.pos;
    if (s.done) {
        sink.flush();
        PairResult res;
        res.score = s.score; res.end_i = s.end_i; res.end_j = s.end_j; res.start_i = s.i; res.start_j = s.j;
        res.n_ops = s.nops; res.path = 2;
        res.overlap = (!LOCAL && (A.opt & 4)) ? (int)(s.nops - (A.m_total + A.n_total - s.nops) + s.mism) : s.best;   // hw4.cpp:141-152
        if (lane == 0) *A.result = res;
    }
    if (lane == 0) *A.st = s;
}

} // namespace b2a
