// short16_fill.cuh -- inter-pair batched DP fill for short pairs (sm_100a).
//
// Replaces the fill loops hw2.cpp:138-156 (NW) and hw2.cpp:205-231 (SW) for every pair of a batch.
// One warp owns one PAIR-PAIR: two pairs of identical shape whose cells travel in the low/high
// halves of s16x2 registers.  Lane L owns pattern rows L*R+1 .. L*R+R; the warp sweeps the text
// as a skewed wavefront (lane L is at column q-L at step q), the row below a lane's band receives
// its boundary through one __shfl_up_sync per step.  Per packed cell pair the ALU pipe sees
//     PRMT            substitution score of both pairs from the text's 4-entry score tables
//     VIADD.16x2      diagonal + score
//     VIADDMNMX.S16x2 max(left + gap, .)
//     VIADDMNMX.S16x2(.RELU for SW)  max(up + gap, .)   [+ VIMNMX.S16x2 row maximum for SW]
// and the FMA pipe one IMAD that folds the new H into the row's delta word (see b2a_format.h
// encode_word: the word of horizontal deltas is a polynomial in the packed H values, evaluated in
// 32-bit ring arithmetic, so no masking, shifting or compare instruction is spent on traceback data).
// NW runs the recurrence on S = H - (i + j) * gap (+ const): both borders become one constant, "left + gap" and "up + gap"
// become plain S values and the diagonal's -2*gap folds into the score table, so a packed cell pair costs
//     PRMT   VIADDMNMX.S16x2 (max(diag + s', left))   VIMNMX.S16x2 (max(., up))
// -- and the plain packed max issues at full rate, while VIADD.16x2 / VIADDMNMX / VIMNMX3 are half rate on sm_100
// (scripts/mb.py).  Horizontal differences of S ARE the stored deltas, the anchor is converted back to H when a chunk
// is stored: the record is bit-identical to the H-space formulation (white-box test against tests/hostmodel.cpp).
// SW stays in H space: its per-row maximum and its floor at 0 do not survive the transform.
// Every 3 words a lane stores one 16-byte chunk {w0,w1,w2,anchor} per row at chunk index (c*32 + lane)*R + r
// (b2a_format.h: consecutive DP rows are 16 bytes apart, which is what the traceback wants); the R stores of a warp
// fill 512R contiguous bytes between them.  (Cache hints on these stores -- st.cs, st.wt, st.cg -- change nothing: 2-bit and 4-bit
// deltas, NW and SW, all within 0.2 %, profiles/r02_store_hints.log.  The 4-bit record's cost is its word bookkeeping, twice per 24 steps.)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "b2a_format.h"

namespace b2a {

// Pattern alphabet of a segment, produced on the device (alphabet kernels in b2a_api.cu) so that the host never has
// to wait for it: the PRMT score tables hold 4 symbols -- the segment's four most frequent pattern bytes.  If the
// segment holds others too (too_many: an 'N' in a read), the pair-pairs that contain one are flagged per pair-pair
// (FillArgs::dirty); the s16x2 kernels skip exactly those and the host hands their pairs to wide32 afterwards.
struct AlphaInfo { uint32_t mask[8]; uint8_t sym[4]; int32_t nsym; int32_t too_many; };

struct FillArgs {
    const uint8_t*  pat;        // concatenated pattern bytes
    const uint8_t*  txt;        // concatenated text bytes
    const uint64_t* pat_off;    // per pair, n_pairs+1
    const uint64_t* txt_off;
    const PPDesc*   pps;        // pair-pairs of this launch (all with the same R)
    const uint64_t* code_off;   // per pair-pair: first chunk of its record
    Chunk*          codes;
    uint32_t*       rowbest;    // local mode: [n_pp][R][32]
    int4*           endcell;    // local mode, per PAIR: {score, end_i, end_j, 0} = first row-major maximum (hw2.cpp:225-229);
                                // semi-global mode: {score, m, j*, 0}, j* = first maximum of row m
    uint32_t        n_pp;
    int32_t         match, mismatch, gap, bias;
    uint32_t        radix;      // 2^K, passed at run time so the word update stays an IMAD (FMA pipe)
    const AlphaInfo* alpha;     // device-resident: the (<= 4) table symbols of this segment
    uint8_t*        dirty;      // per pair-pair of this launch: 0 = the four table symbols cover its patterns (4-symbol kernel), 1 = they do
                                // not: the 8-symbol kernel (A8) serves it, or raises it to 2 = more than 7 distinct pattern symbols: wide32
    const uint32_t* dirty_list; // the pair-pairs with dirty == 1, compacted (dirty_compact_kernel): the 8-symbol kernel's warps take list[0 .. *dirty_cnt)
    const uint32_t* dirty_cnt;
};

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));   // default mode: selector bit 3 replicates the sign
    return d;
}
__device__ __forceinline__ uint32_t pack2(int v) { return ((uint32_t)v & 0xFFFFu) | ((uint32_t)v << 16); }

constexpr int FILL_WARPS = 4;
#ifndef FILL_MIN_CTAS
#define FILL_MIN_CTAS 6          // measured (1 M pairs): 6 / 7 / 8 CTAs per SM (80 / 72 / 64 registers) give NW 21.4 / 21.6 / 21.3 ms and
                                 // SW 25.5 / 26.6 / 26.6 ms -- the kernel waits on the DPX pipe, not on occupancy
#endif

// A8 = false: the segment's four table symbols, one PRMT per cell pair from the column's score-table words (the common case).
// A8 = true : the pair-pairs those tables do not cover (FillArgs::dirty == 1, e.g. a read with an 'N').  Every pair gets its own codes:
//             its (<= 7) distinct pattern bytes are numbered 0..6 in byte order, text bytes the pattern does not hold get code 7.  Equal
//             symbols have equal codes, so the score is PRMT(T, rowsel ^ colsel) from ONE constant table T = [match, mismatch x 7]:
//             the selector nibbles of a row XOR those of the column, nibble 0 picks `match`.  One more ALU instruction (the XOR) per cell
//             pair; the record is the same.  More than 7 pattern symbols: dirty := 2, the pair-pair goes to wide32.
// SEMI (with LOCAL = false): semi-global mode, H space like SW (table scores s, the gap constant in the word, anchor = H) but
// biased (H + bias, A.bias from the global plan), no floor, row 0 = bias (free leading text), column 0 = bias + i*gap.  (NW's S space
// would fit too -- only lane 0's row-0 `up` would grow by |gap| per step -- but that one extra live register makes the R = 4, 5 / K = 2
// instances spill under the 80-register cap.)  The epilogue finds the end cell -- the first maximum of the pair's own row m over
// columns 0..n -- while the record is hot.
template <int R, int K, bool LOCAL, bool A8, bool SEMI = false>
__global__ void __launch_bounds__(FILL_WARPS * 32, (R <= 5 ? FILL_MIN_CTAS : 1))
short16_fill_kernel(const FillArgs A)
{
    static_assert(!(LOCAL && SEMI), "one mode per instantiation");
    constexpr bool HSP = LOCAL || SEMI;                      // the recurrence runs on H (not on NW's S = H - (i + j) gap)
    constexpr int F = Geo<K>::F, CS = Geo<K>::CS;
    // Per warp a MIRRORED ring of the last 128 text columns' entries -- score-table words (tableA, tableB), or the column's selector
    // nibbles (A8) --: entry x lives in slots x & 127 and (x & 127) + 128, so a chunk reads CS consecutive slots from one base with
    // immediate offsets and never wraps.  (The first version kept the whole text's tables, 8 KB per warp: shared memory capped the SM at 24 warps.)
    using RingT = typename std::conditional<A8, uint32_t, uint2>::type;
    __shared__ RingT s_ring[FILL_WARPS][256];
    __shared__ uint32_t s_tbl4[A8 ? 1 : 256];            // byte -> 4 int8 scores against sym[0..3]
    __shared__ uint8_t s_code[A8 ? FILL_WARPS : 1][2][A8 ? 256 : 1];   // A8: byte -> code of pair a / pair b

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t pp = blockIdx.x * FILL_WARPS + warp;
    uint8_t sym[4] = {0, 0, 0, 0};
    if (A8) {
        if (!A.alpha->too_many) return;                  // uniform: the segment has no pair-pair outside its four symbols
        if (pp >= *A.dirty_cnt) return;                  // warp-uniform: the flagged pair-pairs are served in list order, full CTAs
        pp = A.dirty_list[pp];
    } else {
        const int nsym = A.alpha->nsym;
#pragma unroll
        for (int c = 0; c < 4; ++c) sym[c] = A.alpha->sym[c];
        for (int b = threadIdx.x; b < 256; b += blockDim.x) {
            uint32_t w = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int sc = ((c < nsym && sym[c] == (uint8_t)b) ? A.match : A.mismatch) - (HSP ? 0 : 2 * A.gap);
                w |= ((uint32_t)sc & 0xFFu) << (8 * c);
            }
            s_tbl4[b] = w;
        }
        __syncthreads();
        if (pp >= A.n_pp || A.dirty[pp]) return;         // warp-uniform
    }
    RingT* ring = s_ring[warp];

    const PPDesc d = A.pps[pp];
    const uint32_t ma = pp_dim(d.m, 0), mb = pp_dim(d.m, 1), na = pp_dim(d.n, 0), nb = pp_dim(d.n, 1);
    const uint32_t m = pp_max(d.m), n = pp_max(d.n);                  // the sweep covers both pairs; the shorter one gets junk cells
    const uint8_t* pa = A.pat + A.pat_off[d.a];
    const uint8_t* pb = A.pat + A.pat_off[d.b];
    const uint8_t* ta = A.txt + A.txt_off[d.a];
    const uint8_t* tb = A.txt + A.txt_off[d.b];

    uint32_t staged = 0;                                  // text indices [0, staged) have been staged (multiple of 32)
    // bytes of the next block, one block ahead; 0x100 = beyond this pair's own text (mixed-shape pair-pairs): scores as a mismatch against
    // every pattern symbol, whatever bytes the alphabet holds (a NUL pad would MATCH a NUL pattern symbol)
    uint32_t nxa = (uint32_t)lane < na ? ta[lane] : 0x100u, nxb = (uint32_t)lane < nb ? tb[lane] : 0x100u;
    const uint32_t mmw = ((uint32_t)(A.mismatch - (HSP ? 0 : 2 * A.gap)) & 0xFFu) * 0x01010101u;
    // A8: the constant score table, byte 0 = match, bytes 1..7 = mismatch (NW: both minus 2 gap, see above)
    const uint32_t t8lo = (mmw & 0xFFFFFF00u) | ((uint32_t)(A.match - (HSP ? 0 : 2 * A.gap)) & 0xFFu), t8hi = mmw;
    if (A8) {
        // codes of both pairs: presence mask of the pattern's bytes (one warp-wide OR per mask word), code = rank among the present bytes
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
            const uint8_t* ph = h ? pb : pa;
            const uint32_t mh = h ? mb : ma;
            uint32_t msk[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            for (int r = 0; r < R; ++r) {
                const uint32_t i0 = (uint32_t)lane * R + r;
                if (i0 < mh) { const uint32_t x = ph[i0];
#pragma unroll
                    for (int w = 0; w < 8; ++w) if ((x >> 5) == (uint32_t)w) msk[w] |= 1u << (x & 31u); }
            }
            uint32_t nsym8 = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) { msk[w] = __reduce_or_sync(0xFFFFFFFFu, msk[w]); nsym8 += (uint32_t)__popc(msk[w]); }
            if (nsym8 > 7u) { if (lane == 0) A.dirty[pp] = 2; return; }          // warp-uniform: wide32 serves this pair-pair
            // lane L fills the codes of bytes 8L .. 8L+7 (all inside mask word L / 4)
            uint32_t below = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) if (w < (lane >> 2)) below += (uint32_t)__popc(msk[w]);
            uint32_t mine = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) if (w == (lane >> 2)) mine = msk[w];
            const uint32_t base = ((uint32_t)lane & 3u) * 8u;
            for (uint32_t b = 0; b < 8u; ++b) {
                const uint32_t bit = base + b;
                const bool present = (mine >> bit) & 1u;
                s_code[warp][h][lane * 8 + b] = present ? (uint8_t)(below + (uint32_t)__popc(mine & ((1u << bit) - 1u))) : (uint8_t)7;
            }
        }
        __syncwarp();
    }
    auto col_code = [&](int h, uint32_t x) -> uint32_t { return (x & 0x100u) ? 7u : (uint32_t)s_code[A8 ? warp : 0][h][A8 ? x : 0]; };
    auto stage_block = [&]() {
        const uint32_t slot = (staged + (uint32_t)lane) & 127u;
        RingT e;
        if constexpr (A8) e = col_code(0, nxa) * 0x11u | col_code(1, nxb) * 0x1100u;      // selector nibbles: pair a in 0-1, pair b in 2-3
        else e = make_uint2((nxa & 0x100u) ? mmw : s_tbl4[nxa], (nxb & 0x100u) ? mmw : s_tbl4[nxb]);
        __syncwarp();
        ring[slot] = e; ring[slot + 128u] = e;
        __syncwarp();
        staged += 32u;
        const uint32_t x = staged + (uint32_t)lane;
        nxa = x < na ? ta[x] : 0x100u; nxb = x < nb ? tb[x] : 0x100u;
    };

    // PRMT selectors of this lane's rows: byte0 = tableA[codeA], byte1 = its sign, byte2 = tableB[codeB], byte3 = its sign
    uint32_t sel[R], H[R], best[R];
    const uint32_t g2 = pack2(A.gap);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t i0 = (uint32_t)lane * R + r;     // 0-based row
        uint32_t ca = 0, cb = 0;
        if (A8) {
            if (i0 < ma) ca = s_code[A8 ? warp : 0][0][A8 ? pa[i0] : 0];
            if (i0 < mb) cb = s_code[A8 ? warp : 0][1][A8 ? pb[i0] : 0];
            sel[r] = ca | ((8u | ca) << 4) | (cb << 8) | ((8u | cb) << 12);     // XORed with the column's nibbles: 0 = equal symbols
        } else {
            if (i0 < ma) { const uint8_t xa = pa[i0];
#pragma unroll
                for (int c = 1; c < 4; ++c) if (xa == sym[c]) ca = c; }
            if (i0 < mb) { const uint8_t xb = pb[i0];
#pragma unroll
                for (int c = 1; c < 4; ++c) if (xb == sym[c]) cb = c; }
            sel[r] = ca | ((8u | ca) << 4) | ((4u + cb) << 8) | ((12u + cb) << 12);
        }
        // LOCAL: H of the column-0 border (0, hw2.cpp:196-197).  NW: S of the frozen border H(i, 0) = i*gap (hw2.cpp:125-130) as
        // seen from this lane's column before step 0, j = -1 - lane: Z - (lane + 1)|gap|; it grows by |gap| per frozen step
        // and reaches Z = 32|gap| at column 0 (every border cell has S = Z).
        // SEMI: the biased border H(i, 0) = bias + i*gap, frozen until the lane reaches column 1.
        H[r] = LOCAL ? 0u : (SEMI ? pack2(A.bias + (int)(i0 + 1u) * A.gap) : pack2((31 - lane) * -A.gap));
        best[r] = 0u;
    }
    __syncwarp();

    const uint32_t NC = num_chunks(n, CS);
    Chunk* rec = A.codes + A.code_off[pp];
    const uint32_t radix = A.radix;
    const uint32_t g32 = (uint32_t)A.gap * 65537u;
    uint32_t geo = 0, bpow = 1;
#pragma unroll
    for (int t = 0; t < F; ++t) geo = geo * radix + 1u;
#pragma unroll
    for (int t = 0; t < F - 1; ++t) bpow *= radix;
    // delta word = sum B^(F-1-t) (P_t - P_{t-1} - g): in S space the differences already exclude the gap, so the constant term goes
    const uint32_t negGc = HSP ? 0u - g32 * geo : 0u, negBpow = 0u - bpow, radm1 = radix - 1u;
    const uint32_t ag2 = pack2(-A.gap), Z = pack2(-32 * A.gap);         // NW: |gap| packed; S of every border cell
    const uint32_t top = SEMI ? pack2(A.bias) : 0u;                     // SEMI: biased H of every row-0 cell (free leading text)
    // NW: stored anchor = H + bias = S + (i + j)*gap + (bias - 32|gap|), i + j = lane*(R-1) + r + 1 + q at step q
    const int abase = ((int)lane * (R - 1) + 1) * A.gap + A.bias + 32 * A.gap;
    auto anchor_of_S = [&](uint32_t Sv, int r, uint32_t q) { return __vadd2(Sv, pack2(abase + (r + (int)q) * A.gap)); };

    uint32_t dgn = LOCAL ? 0u : (SEMI ? top : pack2((31 - lane) * -A.gap));   // value the row above had one column to the left (SEMI: overwritten before the lane's first column)

    // one wavefront step for this lane; `active` is false only in the ramp chunks (lanes outside their column range keep H frozen).
    // (A select-based, branch-free ramp -- what wide32 needs -- was measured here: NW fill -1.0 %, SW +0.6 %, i.e. nothing: with 24 warps
    // per SM the 4 ramp chunks of 43 hide their latencies behind other warps.)
    auto step = [&](const RingT* tcol, int k, uint32_t q, uint32_t (&S)[R], int f, bool active) {
        uint32_t up = __shfl_up_sync(0xFFFFFFFFu, H[R - 1], 1);
        if (lane == 0) up = LOCAL ? 0u : (SEMI ? top : Z);              // row 0 border, hw2.cpp:131-136 (S = Z) / :196-197 / semi-global
        const uint32_t dg0 = dgn;
        dgn = up;
        if (active) {
            const RingT tw = tcol[k];                                   // tables / selector nibbles of column j = q - lane (text index j - 1)
            uint32_t dg = dg0, u = up;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                uint32_t s;
                if constexpr (A8) s = prmt(t8lo, t8hi, sel[r] ^ tw);
                else s = prmt(tw.x, tw.y, sel[r]);
                uint32_t h;
                if (LOCAL) {
                    const uint32_t ds = __vadd2(dg, s);
                    dg = H[r];
                    const uint32_t a = __viaddmax_s16x2(H[r], g2, ds);
                    h = __viaddmax_s16x2_relu(u, g2, a);
                    best[r] = __vmaxs2(best[r], h);
                } else if (SEMI) {
                    const uint32_t ds = __vadd2(dg, s);
                    dg = H[r];
                    const uint32_t a = __viaddmax_s16x2(H[r], g2, ds);   // max(diag + s, left + gap)
                    h = __viaddmax_s16x2(u, g2, a);                      // max(., up + gap)
                } else {
                    const uint32_t a = __viaddmax_s16x2(dg, s, H[r]);   // max(diag + s - 2 gap, left)   in S space
                    dg = H[r];
                    h = __vmaxs2(a, u);                                  // max(., up)
                }
                H[r] = h; u = h;
            }
        } else if (!HSP) {
            // a frozen H is a growing S (the lane's column still moves): keeps the record identical to the H-space formulation
#pragma unroll
            for (int r = 0; r < R; ++r) H[r] = __vadd2(H[r], ag2);
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (f == 0) S[r] = H[r];
            else if (f < F - 1) S[r] = S[r] * radix + H[r];
        }
    };

    for (uint32_t c = 0; c < NC; ++c) {
        const uint32_t q0 = c * CS;
        while (staged < q0 + CS) stage_block();                        // steps q0 .. q0+CS-1 read text indices q0-32 .. q0+CS-2
        const RingT* tcol = ring + ((q0 - (uint32_t)lane - 1u) & 127u);  // tcol[k] = entry of text index q0 + k - lane - 1
        uint32_t w0[R], w1[R];
        if (q0 >= 32u && q0 + CS - 1 <= n) {
            // steady state: every lane is inside its row range for the whole chunk
#pragma unroll
            for (int wi = 0; wi < 3; ++wi) {
                uint32_t S[R], pre[R];
#pragma unroll
                for (int r = 0; r < R; ++r) pre[r] = H[r] * negBpow + negGc;
#pragma unroll
                for (int f = 0; f < F; ++f) step(tcol, wi * F + f, q0 + wi * F + f, S, f, true);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const uint32_t w = (F > 1 ? S[r] * radm1 : 0u) + H[r] + pre[r];
                    if (wi == 0) w0[r] = w; else if (wi == 1) w1[r] = w;
                    else {
                        const uint32_t anchor = HSP ? H[r] : anchor_of_S(H[r], r, q0 + CS - 1);
                        const uint4 v = make_uint4(w0[r], w1[r], w, anchor);
                        *reinterpret_cast<uint4*>(&rec[((size_t)c * 32u + lane) * R + r]) = v;
                    }
                }
            }
        } else {
            // ramp-up / ramp-down chunks: lanes outside 1 <= q - lane <= n keep their H frozen
#pragma unroll 1
            for (int wi = 0; wi < 3; ++wi) {
                uint32_t S[R], pre[R];
#pragma unroll
                for (int r = 0; r < R; ++r) pre[r] = H[r] * negBpow + negGc;
#pragma unroll
                for (int f = 0; f < F; ++f) {
                    const uint32_t q = q0 + wi * F + f;
                    step(tcol, wi * F + f, q, S, f, (uint32_t)(q - lane - 1u) < n);
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const uint32_t w = (F > 1 ? S[r] * radm1 : 0u) + H[r] + pre[r];
                    uint32_t* cw = reinterpret_cast<uint32_t*>(&rec[((size_t)c * 32u + lane) * R + r]);
                    cw[wi] = w;
                    if (wi == 2) cw[3] = HSP ? H[r] : anchor_of_S(H[r], r, q0 + CS - 1);
                }
            }
        }
    }
    if (LOCAL) {
#pragma unroll
        for (int r = 0; r < R; ++r) A.rowbest[((size_t)pp * R + r) * 32u + lane] = best[r];
        // ---- end cell of both pairs (hw2.cpp:202-203, :225-229: first strict maximum in row-major order), found by
        // the warp while the record is still hot: per-row maxima -> first best row, then the row's chunks are rebuilt
        // backwards from their anchors by the lanes in parallel.  ~2 % of the fill; the traceback kernel (one thread
        // per pair) used to spend more than its whole walk on this search.
        __syncwarp();                                            // the chunk stores above are visible to the whole warp
        const PPDesc de = A.pps[pp];                              // re-read: keeping the per-half shapes live through the sweep cost 4 %
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const uint32_t mh = pp_dim(de.m, half), nh = pp_dim(de.n, half);     // this pair's own shape
            int mloc = 0; uint32_t iloc = 0xFFFFFFFFu;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int v = (int)((best[r] >> (16 * half)) & 0xFFFFu);
                const uint32_t i = (uint32_t)lane * R + r + 1u;
                if (i <= mh && v > mloc) { mloc = v; iloc = i; }
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                const int om = __shfl_xor_sync(0xFFFFFFFFu, mloc, o);
                const uint32_t oi = __shfl_xor_sync(0xFFFFFFFFu, iloc, o);
                if (om > mloc || (om == mloc && oi < iloc)) { mloc = om; iloc = oi; }
            }
            uint32_t bi = 0, bj = 0;
            if (mloc > 0) {
                bi = iloc;
                const uint32_t Lb = (bi - 1u) / R;
                const Chunk* row = rec + (bi - 1u);                   // chunk c of DP row bi sits at c*32R + (bi-1)
                const int floor_anchor = mloc + (CS - 1) * A.gap;     // H falls by at most |gap| per step to the right
                uint32_t cand = 0xFFFFFFFFu;                          // smallest step q of the row with H == max
                for (uint32_t c = (uint32_t)lane; c < NC; c += 32u) {
                    const uint4 ch = __ldcg(reinterpret_cast<const uint4*>(row + (size_t)c * (32u * R)));
                    const int sh = 16 * half;
                    int Hq = (int)((ch.w >> sh) & 0xFFFFu);
                    if (Hq < floor_anchor) continue;
                    const uint64_t X = ((uint64_t)((ch.x >> sh) & 0xFFFFu) << 32) | ((uint64_t)((ch.y >> sh) & 0xFFFFu) << 16) | ((ch.z >> sh) & 0xFFFFu);
                    for (int rem = CS - 1; rem >= 0; --rem) {
                        const uint32_t q = c * CS + (uint32_t)rem;
                        if (Hq == mloc && q - Lb - 1u < nh) cand = min(cand, q);   // columns 1..n only (frozen steps outside repeat border values)
                        Hq -= (int)((uint32_t)(X >> (K * (CS - 1 - rem))) & Geo<K>::MASK) + A.gap;
                    }
                }
#pragma unroll
                for (int o = 16; o; o >>= 1) cand = min(cand, __shfl_xor_sync(0xFFFFFFFFu, cand, o));
                bj = cand - Lb;
            }
            if (lane == 0) A.endcell[half ? de.b : de.a] = make_int4(mloc, (int)bi, (int)bj, 0);
        }
    }
    if (SEMI) {
        // ---- semi-global end cell of both pairs: the first maximum of the pair's own row m over columns 0..n.  As in the SW
        // epilogue the lanes rebuild that row's chunks backwards from their anchors; only steps q with 0 <= q - Lb <= n count, so the
        // junk columns of a mixed-shape pair-pair never do.  Column 0 is step Lb, where the lane still held the border bias + m*gap.
        __syncwarp();                                            // the chunk stores above are visible to the whole warp
        const PPDesc de = A.pps[pp];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const uint32_t mh = pp_dim(de.m, half), nh = pp_dim(de.n, half);
            const uint32_t Lb = (mh - 1u) / R;                        // lane that owned row m: column j sits at step q = j + Lb
            const Chunk* row = rec + (mh - 1u);
            const int sh = 16 * half;
            int bv = -1;                                              // biased H >= 0
            uint32_t bq = 0xFFFFFFFFu;
            for (uint32_t c = (uint32_t)lane; c < NC; c += 32u) {
                const uint4 ch = __ldcg(reinterpret_cast<const uint4*>(row + (size_t)c * (32u * R)));
                int Hq = (int)((ch.w >> sh) & 0xFFFFu);
                const uint64_t X = ((uint64_t)((ch.x >> sh) & 0xFFFFu) << 32) | ((uint64_t)((ch.y >> sh) & 0xFFFFu) << 16) | ((ch.z >> sh) & 0xFFFFu);
                for (int rem = CS - 1; rem >= 0; --rem) {
                    const uint32_t q = c * CS + (uint32_t)rem;
                    if (q - Lb <= nh && (Hq > bv || (Hq == bv && q < bq))) { bv = Hq; bq = q; }
                    Hq -= (int)((uint32_t)(X >> (K * (CS - 1 - rem))) & Geo<K>::MASK) + A.gap;
                }
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                const int ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o);
                const uint32_t oq = __shfl_xor_sync(0xFFFFFFFFu, bq, o);
                if (ov > bv || (ov == bv && oq < bq)) { bv = ov; bq = oq; }
            }
            if (lane == 0) A.endcell[half ? de.b : de.a] = make_int4(bv - A.bias, (int)mh, (int)(bq - Lb), 0);
        }
    }
}

} // namespace b2a
