// b2a_format.h -- HBM layout of the DP record and the tie-exact traceback that reads it.
// Shared by the CUDA kernels (device) and by the host-side format model used in CPU tests
// (tests/hostmodel.cpp), so the decoder logic is exercised without a GPU.  No CUDA types here.
//
// What is stored (see DESIGN.md "DP record"):
//   The fill kernels never write H or direction letters.  Per DP row they write the HORIZONTAL
//   DELTAS  D(i,j) = H(i,j) - H(i,j-1) - gap, which for a linear gap always lie in
//   [0, max(match,mismatch) - 2*gap]  (K = 2, 4, 8, 16 bits; K = 32 stores the raw signed delta and
//   therefore holds ANY scoring), plus one absolute anchor H per chunk.  The traceback rebuilds the
//   exact H of the three neighbours of each visited cell and then applies the reference's own
//   comparisons (hw2.cpp:145-153 for NW, hw2.cpp:214-222 for SW), so ties break exactly as in the
//   reference by construction.
//
// Geometry (both kernel families): a BAND is 32 lanes x R rows; lane L owns rows
//   i = band*32R + L*R + r + 1, r = 0..R-1.  At (lane-)step q lane L is at column j = q - L*SKEW
//   (active iff 1 <= j <= n, otherwise its H registers are frozen, which makes D = -gap, still in
//   range).  SKEW = 1: the lanes follow each other one column apart (one shuffle per column).  SKEW = 4
//   (wide32, K <= 8): a lane computes R x 4 cells per macro-step from four independent shuffles, so the
//   next lane is four columns behind (a register tile instead of a single column: 4-5x the cells per
//   dependent shuffle, which is what a single long pair -- one warp per band -- is bound by).  A word holds F = WBITS/K steps, a 16-byte chunk holds NWORDS words + the anchor
//   (= H after the chunk's last step) and covers CS = NWORDS*F steps.
//   wide32 : chunk index of (band, r, c, L) = ((band*R + r)*NC + c)*32 + L  -> a warp stores 512 contiguous bytes;
//            the chunks of one row are 32 apart.
//   short16: chunk index of (row i, c) = c*32R + (i-1) = (c*32 + L)*R + r: ROW-MAJOR inside a chunk column, so the
//            chunks of consecutive DP rows are 16 bytes apart.  A traceback path climbs one row per step: with
//            this order a 128-byte line holds 8 rows of it (an earlier r-major order put every row change into a
//            different line: L1 hit rate 16-35 %, 2.5x the DRAM traffic).  The chunks of one row are 32R apart.
//
//   short16 family: two pairs of identical shape in the low/high 16-bit halves of every word
//                   (WBITS = 16, NWORDS = 3, one band, R = ceil(m/32) <= 8, K in {2,4,8}).
//   wide32  family: one pair per warp-band, int32 (WBITS = 32, NWORDS = 2, R = 4, any m and n,
//                   K in {2,4,8,16,32}).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define B2A_HD __host__ __device__ __forceinline__
#else
#define B2A_HD inline
#endif

namespace b2a {

struct alignas(16) Chunk { uint32_t w0, w1, w2, anchor; };

// pair-pair descriptor (short16): pairs a and b (b == a for an unpaired singleton).  m = m_a | m_b << 16, n = n_a | n_b << 16:
// the two pairs may differ in shape.  The warp sweeps max(m) x max(n); cells right of / below a half's own (m, n) are junk that
// never feeds its real cells (the recurrence only looks left and up), and only the epilogue and the walker use the true shapes.
struct PPDesc { uint32_t a, b, m, n; };
B2A_HD uint32_t pp_dim(uint32_t packed, int half) { return half ? packed >> 16 : packed & 0xFFFFu; }
B2A_HD uint32_t pp_max(uint32_t packed) { const uint32_t lo = packed & 0xFFFFu, hi = packed >> 16; return lo > hi ? lo : hi; }
B2A_HD uint32_t pp_pack(uint32_t lo, uint32_t hi) { return lo | (hi << 16); }

// one record per pair; mirrors b2a_result in include/b2align.h (static_assert in b2a_api.cu)
struct PairResult {
    int32_t score; uint32_t end_i, end_j, start_i, start_j; int32_t overlap; uint32_t n_ops; uint32_t path;
};

enum : uint32_t { OP_M = 0, OP_D = 1, OP_I = 2 };

template <int K_, int WBITS_, int NWORDS_, int SKEW_ = 1> struct Fmt {
    static_assert(K_ == 2 || K_ == 4 || K_ == 8 || K_ == 16 || K_ == 32, "delta width");
    static_assert(WBITS_ % K_ == 0 && (WBITS_ == 16 || WBITS_ == 32), "word width");
    static_assert(SKEW_ == 1 || (WBITS_ / K_) % SKEW_ == 0, "a macro-step never straddles a delta word");
    static constexpr int K = K_, WBITS = WBITS_, NWORDS = NWORDS_, SKEW = SKEW_;
    static constexpr int F = WBITS_ / K_;       // steps per word
    static constexpr int CS = NWORDS_ * F;      // steps per 16-byte chunk
    static constexpr uint32_t MASK = K_ == 32 ? 0xFFFFFFFFu : ((1u << (K_ & 31)) - 1u);
};
// Lane skew of the wide32 RECORD.  4 was built and measured (profiles/r02_wide32_tile.md): the 4-column register tile raises the
// throughput of many concurrent pairs by 9 % but makes ONE long pair slower (13.1 vs 10.0 ms at 100 kb): the bottom row of a band
// exists 31 lane-to-lane hand-offs after its top row whatever the tile width, and a 4-column macro-step takes 3.5x as long as a
// single step.  So kernels that write a record keep skew 1; the score-only kernels (no record, many pairs) use the tile.
constexpr int wide_skew(int /*K*/) { return 1; }
constexpr int WIDE_TILE_SCORE_ONLY = 4;
template <int K> using Short16 = Fmt<K, 16, 3>;
template <int K> using Wide32 = Fmt<K, 32, 2, wide_skew(K)>;
template <int K> using Geo = Short16<K>;        // the short16 kernels' name for their geometry

constexpr int WIDE_R = 4;                        // rows per lane in the wide32 family (band = 128 rows)

// chunks per DP row: lane 31 reaches column n at step n + 31*skew
B2A_HD uint32_t num_chunks(uint32_t n, int CS, int skew = 1) { return (n + 31u * (uint32_t)skew + (uint32_t)CS) / (uint32_t)CS; }

// number of distinct D values of a scoring scheme; 0 if the delta-range lemma does not apply
B2A_HD long delta_span(int match, int mismatch, int gap) {
    const long smax = match > mismatch ? match : mismatch;
    if (gap > 0 || smax < 0) return 0;
    return smax - 2L * gap + 1;
}
// smallest K the short16 record supports, 0 if none
B2A_HD int delta_bits(int match, int mismatch, int gap) {
    const long W = delta_span(match, mismatch, gap);
    if (W <= 0) return 0;
    if (W <= 4) return 2;
    if (W <= 16) return 4;
    if (W <= 256) return 8;
    return 0;
}
// K for the wide32 record: always defined (32 = raw signed deltas, no lemma needed)
B2A_HD int delta_bits_wide(int match, int mismatch, int gap) {
    const long W = delta_span(match, mismatch, gap);
    if (W <= 0) return 32;
    if (W <= 4) return 2;
    if (W <= 16) return 4;
    if (W <= 256) return 8;
    if (W <= 65536) return 16;
    return 32;
}

// Can the s16x2 record hold an m x n pair-class under this scoring?  Chooses rows-per-lane R,
// the delta width K and the bias that keeps every stored H of the (junk-extended) matrix in
// [0, 32767] (needed both for the s16 arithmetic and for the ring-exact word encoding).
struct Short16Plan { int K, R, bias; };
constexpr int SHORT16_MAX_R = 16;         // rows per lane -> patterns up to 512 bases
// rows per lane for an m-row pattern: every value up to 8, then 10, 12, 16 (fewer kernel instances; the extra rows are junk rows)
B2A_HD int short16_R(uint32_t m) {
    const int r = (int)((m + 31u) / 32u);
    return r <= 8 ? r : (r <= 10 ? 10 : (r <= 12 ? 12 : 16));
}
// mode: 0 global, 1 local, 2 semi-global.  Semi-global takes the global plan: with gap <= 0 every semi-global H lies in
// i*gap <= H(i,j) <= min(i,j)*max(match,0), inside the range the global bias and checks already cover, and its fill (H space,
// table scores s) needs no more than the global fill (S space, scores s - 2 gap), so one plan serves every run of a batch.
B2A_HD bool short16_plan(int mode, uint32_t m, uint32_t n, int match, int mismatch, int gap, Short16Plan& pl) {
    if (mode == 2) mode = 0;
    if (m == 0 || n == 0 || m > 32u * SHORT16_MAX_R || n > 30000u) return false;     // (the int16 range test below is the real limit on n)
    pl.K = delta_bits(match, mismatch, gap);
    if (pl.K == 0) return false;
    if (match > 127 || match < -128 || mismatch > 127 || mismatch < -128) return false;   // PRMT score tables are int8
    pl.R = short16_R(m);
    const long rows = 32L * pl.R;
    const long smax = match > mismatch ? match : mismatch, smin = match < mismatch ? match : mismatch;
    const long margin = (long)(-gap) + (smin < 0 ? -smin : 0) + 1;
    const long top = (rows < (long)n ? rows : (long)n) * (smax > 0 ? smax : 0) + margin;
    long bias = 0;
    if (mode == 0) bias = (rows + (long)n) * (long)(-gap) + margin;
    if (bias + top > 32767) return false;
    // NW fill works on S = H - (i + j) gap + 32|gap| (short16_fill.cuh): frozen lanes run up to 31 columns past either end,
    // and the score table holds s - 2 gap as int8
    if (mode == 0 && (bias + top + 64L * (long)(-gap) > 32767 || smax - 2L * gap > 127 || smin - 2L * gap < -128)) return false;
    pl.bias = (int)bias;
    return true;
}

B2A_HD int popc32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// sum of the K-bit fields of a word (K < 32)
template <int K> B2A_HD int field_sum(uint32_t x) {
    if (K == 2) return popc32(x & 0x55555555u) + 2 * popc32(x & 0xAAAAAAAAu);
    if (K == 4) { const uint32_t b = (x & 0x0F0F0F0Fu) + ((x >> 4) & 0x0F0F0F0Fu); return (int)((b * 0x01010101u) >> 24); }
    if (K == 8) { const uint32_t h = (x & 0x00FF00FFu) + ((x >> 8) & 0x00FF00FFu); return (int)((h + (h >> 16)) & 0xFFFFu); }
    if (K == 16) return (int)((x & 0xFFFFu) + (x >> 16));
    return (int)x;
}

// Read-only view of one pair inside its record.
struct PairView {
    const Chunk*    codes;     // this pair's (pair-pair's) chunk block
    const uint32_t* rowbest;   // per-row maxima (local mode): [(band*R + r)*32 + L]
    const uint8_t*  p;         // pattern bytes (rows)
    const uint8_t*  t;         // text bytes (columns)
    uint32_t m, n, NC;
    int R, half;               // half: short16 only, 0 = low 16 bits, 1 = high
    int match, mismatch, gap, bias;
    int opt;                   // walker bits: 1 = batch runs of 'l' moves, 2 = L2-prefetch rows ahead, 4 = hw4 tie order d > u > l
    int rmagic;                // short16: ceil(65536 / R)
    const int32_t* top = nullptr;   // checkpointed sub-problems (wide32): exact H of the row above row 1, top[j] for columns 0..n; null = the
                                    // real border row 0 (H = bias + j*gap global / 0 local)
};

template <class FM> B2A_HD uint32_t word_of(const Chunk& ch, int wi, int half) {
    const uint32_t w = wi == 0 ? ch.w0 : (wi == 1 ? ch.w1 : ch.w2);
    return FM::WBITS == 16 ? ((w >> (half * 16)) & 0xFFFFu) : w;
}
template <class FM> B2A_HD int anchor_of(const Chunk& ch, int half) {
    return FM::WBITS == 16 ? (int)((ch.anchor >> (half * 16)) & 0xFFFFu) : (int)ch.anchor;
}
template <class FM> B2A_HD int rowbest_of(uint32_t v, int half) {
    return FM::WBITS == 16 ? (int)((v >> (half * 16)) & 0xFFFFu) : (int)v;
}
template <class FM> B2A_HD int field_of(uint32_t word, int f) {           // field of in-word step f
    if (FM::K == 32) return (int)word;
    return (int)((word >> (FM::K * (FM::F - 1 - f))) & FM::MASK);
}

// H (biased) and D of the cell computed at in-chunk step `rem`
template <class FM>
B2A_HD void decode_step(const Chunk& ch, int half, int gap, int rem, int& H, int& D) {
    const int wi = rem / FM::F, f = rem - wi * FM::F;
    const uint32_t w = word_of<FM>(ch, wi, half);
    D = field_of<FM>(w, f);
    int sum = 0;
    if (FM::K < 32) {
        const int off = FM::K * (FM::F - 1 - f);
        sum = field_sum<FM::K>(w & ((1u << (off & 31)) - 1u));
    }
    for (int k = wi + 1; k < FM::NWORDS; ++k) sum += FM::K == 32 ? (int)word_of<FM>(ch, k, half) : field_sum<FM::K>(word_of<FM>(ch, k, half));
    H = anchor_of<FM>(ch, half) - (FM::CS - 1 - rem) * gap - sum;
}

// (row i, chunk c) -> chunk index, and the lane L that owns the row.  No runtime divisions: the wide32
// family has R = 4 (shifts); short16 has a single band and R <= 16, where x / R == (x * rmagic) >> 16
// exactly for x < 512 (rmagic = 65536 / R rounded up; checked exhaustively in tests).
template <class FM>
B2A_HD uint32_t row_slot(const PairView& v, uint32_t i, uint32_t& L) {     // band*R + r, and the owning lane
    const uint32_t x = i - 1u;
    if (FM::WBITS == 32) { L = (x >> 2) & 31u; return (x >> 7) * 4u + (x & 3u); }
    L = (x * (uint32_t)v.rmagic) >> 16;
    return x - L * (uint32_t)v.R;
}
template <class FM>
B2A_HD uint32_t chunk_stride(const PairView& v) {                          // distance between consecutive chunks of one row
    return FM::WBITS == 32 ? 32u : 32u * (uint32_t)v.R;
}
template <class FM>
B2A_HD uint64_t chunk_index(const PairView& v, uint32_t i, uint32_t c, uint32_t& L) {
    const uint32_t slot = row_slot<FM>(v, i, L);
    if (FM::WBITS == 32) return ((uint64_t)slot * v.NC + c) * 32u + L;
    return (uint64_t)c * (32u * (uint32_t)v.R) + (i - 1u);
}
B2A_HD int short16_rmagic(int R) { return (65536 + R - 1) / R; }

B2A_HD int popc64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}
// sum of the K-bit fields of a 64-bit field string
template <int K> B2A_HD int field_sum64(uint64_t x) {
    if (K == 2) return popc64(x & 0x5555555555555555ull) + 2 * popc64(x & 0xAAAAAAAAAAAAAAAAull);
    if (K == 32) return (int)((uint32_t)x + (uint32_t)(x >> 32));
    return field_sum<K>((uint32_t)x) + field_sum<K>((uint32_t)(x >> 32));
}
// the chunk's delta words as one field string: step rem of the chunk sits at bit K*(CS-1-rem)
template <class FM> B2A_HD uint64_t chunk_string(const Chunk& ch, int half) {
    if (FM::WBITS == 32) return ((uint64_t)ch.w0 << 32) | ch.w1;
    const int sh = half * 16;
    return ((uint64_t)((ch.w0 >> sh) & 0xFFFFu) << 32) | ((uint64_t)((ch.w1 >> sh) & 0xFFFFu) << 16) | ((ch.w2 >> sh) & 0xFFFFu);
}

// (chunks of a row are chunk_stride() apart)
// A cursor on one DP row of the record: knows the exact H at its column and can step LEFT for the
// price of one field extraction (H(i,j-1) = H(i,j) - D(i,j) - gap); a chunk is (re)loaded only when
// the column crosses a chunk boundary.  Seeking (a new row) costs one chunk load + one popcount sum
// from the chunk's anchor.  Row 0 is a virtual cursor: H = bias + j*gap (global) / 0 (local), no loads.
template <class FM, class Loader, bool LOCAL>
struct RowCursor {
    static constexpr int BITS = FM::K * FM::CS;      // 48 (short16) or 64 (wide32)
    uint64_t X;         // field string of the current chunk
    uint64_t cidx;      // index of the current chunk (chunks of a row are 32 apart); 0 on the border row
    int H, off, c;      // off = bit offset of the current field
    int dborder;        // D of the virtual row 0 (0 global, -gap local; from the checkpoint row of a sub-problem), unused otherwise
    bool border;
    B2A_HD void seek(const PairView& v, const Loader& ld, uint32_t i, uint32_t j) {
        if (i == 0) {
            border = true; X = 0; off = 0; cidx = 0;
            if (v.top) {                                             // row 0 of a checkpointed sub-problem: stored values (top[0..n]), not the border formula
                c = (int)j;                                          // (c doubles as the column on this row)
                H = v.top[j];
                dborder = j ? H - v.top[j - 1] - v.gap : 0;
            } else { c = 0; H = LOCAL ? 0 : v.bias + (int)j * v.gap; dborder = LOCAL ? -v.gap : 0; }
            return;
        }
        border = false; dborder = 0;
        uint32_t L;
        const uint64_t base = chunk_index<FM>(v, i, 0, L);
        const uint32_t q = j + L * (uint32_t)FM::SKEW;
        c = (int)(q / (uint32_t)FM::CS);
        const int rem = (int)(q - (uint32_t)c * (uint32_t)FM::CS);
        cidx = base + (uint64_t)c * chunk_stride<FM>(v);
        const Chunk ch = ld(cidx);
        X = chunk_string<FM>(ch, v.half);
        off = FM::K * (FM::CS - 1 - rem);
        const uint64_t low = off ? (X & (~0ull >> (64 - off))) : 0ull;
        H = anchor_of<FM>(ch, v.half) - (FM::CS - 1 - rem) * v.gap - field_sum64<FM::K>(low);
    }
    B2A_HD int D() const {
        if (border) return dborder;
        return FM::K == 32 ? (int)(uint32_t)(X >> off) : (int)((uint32_t)(X >> off) & FM::MASK);
    }
    // move to column j-1 (caller guarantees j >= 1)
    B2A_HD void left(const PairView& v, const Loader& ld) {
        if (border && v.top) {                                       // step along the checkpoint row
            if (c > 0) { --c; H = v.top[c]; dborder = c ? H - v.top[c - 1] - v.gap : 0; }
            return;
        }
        H -= D() + v.gap;
        off += FM::K;
        if (off == BITS) {
            off = 0;
            if (!border && c > 0) { --c; cidx -= chunk_stride<FM>(v); X = chunk_string<FM>(ld(cidx), v.half); }
            // c == 0: step q = 0, nothing further left is ever read
            else if (!border) off = BITS - FM::K;
        }
    }
};

// The walk is a chain of dependent chunk loads (one per row change).  The path is mostly diagonal, so the
// chunks of the next few rows up are predictable: ask for them PF rows ahead (L2 prefetch, no register cost).
constexpr uint32_t WALK_PF = 6;
template <class FM, class Loader>
B2A_HD void prefetch_row(const PairView& v, const Loader& ld, uint32_t i, uint32_t j) {
    if (i == 0) return;
    uint32_t L;
    const uint64_t base = chunk_index<FM>(v, i, 0, L);
    ld.prefetch(base + (uint64_t)((j + L * (uint32_t)FM::SKEW) / (uint32_t)FM::CS) * chunk_stride<FM>(v));
}

// ---- Needleman-Wunsch traceback, hw2.cpp:158-181 on reconstructed H; directions per hw2.cpp:145-153 ----
template <class FM, class Loader, class Sink>
B2A_HD void walk_global(const PairView& v, Loader ld, Sink& sink, PairResult& res) {
    uint32_t i = v.m, j = v.n, nops = 0;
    int cur = 0, best = 0;
    RowCursor<FM, Loader, false> rc, ru;                             // rows i and i-1 at column j
    rc.seek(v, ld, (i && j) ? i : 0, j);
    if (i == 0 || j == 0) rc.H = v.bias + (int)(i + j) * v.gap;      // border, hw2.cpp:125-136
    res.score = rc.H - v.bias;                                       // hw2.cpp:186
    if (i && j) ru.seek(v, ld, i - 1, j);
    if (v.opt & 2) for (uint32_t k = 2; k < 2 + WALK_PF && k <= i; ++k) prefetch_row<FM>(v, ld, i - k, j > k ? j - k + 1 : 1);
    while (i > 0 && j > 0) {
        const int Hl = rc.H - rc.D() - v.gap;                       // H(i, j-1); frozen lanes make this the border at j == 1
        const int Hu = ru.H, Hd = Hu - ru.D() - v.gap;              // H(i-1, j), H(i-1, j-1)
        const uint8_t pc = v.p[i - 1];
        const bool eq = pc == v.t[j - 1];
        int val = Hd + (eq ? v.match : v.mismatch);                  // hw2.cpp:142
        uint32_t op = OP_M;                                          // hw2.cpp:145
        if (v.opt & 4) {                                             // hw4's order d > u > l (hw4.cpp:37-46)
            if (Hu + v.gap > val) { val = Hu + v.gap; op = OP_D; }
            if (Hl + v.gap > val) { op = OP_I; }
        } else {
            if (Hl + v.gap > val) { val = Hl + v.gap; op = OP_I; }   // hw2.cpp:146-149 'l'
            if (Hu + v.gap > val) { op = OP_D; }                     // hw2.cpp:150-153 'u'
        }
        if (op == OP_I && (v.opt & 1) && !(v.opt & 4)) {
            // a run of 'l' moves stays inside the two chunks in registers: no memory traffic until a chunk edge
            cur = 0;
            for (;;) {
                rc.left(v, ld); ru.left(v, ld);
                --j; sink.put(OP_I); ++nops;
                if (j == 0 || rc.off == 0 || ru.off == 0) break;
                const int hl = rc.H - rc.D(), hd = ru.H - ru.D() - v.gap + (pc == v.t[j - 1] ? v.match : v.mismatch);
                if (!(hl > hd && !(ru.H + v.gap > hl))) break;       // next cell is not 'l' (same tests as above)
            }
            continue;
        }
        if (op == OP_M && eq && pc != (uint8_t)'-') { if (++cur > best) best = cur; } else cur = 0;   // hw2.cpp:267-278
        if (op != OP_D) { rc.left(v, ld); ru.left(v, ld); --j; }     // 'M' and 'I' both move one column left
        if (op != OP_I) {                                            // 'M' and 'D' both move one row up
            rc = ru; --i;
            if (i > 0) ru.seek(v, ld, i - 1, j);
            if ((v.opt & 2) && i > 1 + WALK_PF) prefetch_row<FM>(v, ld, i - 1 - WALK_PF, j > WALK_PF ? j - WALK_PF : 1);
        }
        sink.put(op);
        ++nops;
    }
    for (; i > 0; --i, ++nops) sink.put(OP_D);                       // column 0 holds 'u' (hw2.cpp:128)
    for (; j > 0; --j, ++nops) sink.put(OP_I);                       // row 0 holds 'l' (hw2.cpp:134)
    res.end_i = v.m; res.end_j = v.n; res.start_i = 0; res.start_j = 0;
    res.overlap = best; res.n_ops = nops;
}

// first row-major arg-max (hw2.cpp:225-229) from the per-row maxima + a left-to-right rebuild of one row
template <class FM, class Loader>
B2A_HD void find_local_end(const PairView& v, Loader ld, int& M, uint32_t& bi, uint32_t& bj) {
    M = 0; bi = 0; bj = 0;
    if (v.n == 0) return;                                           // no cells: the fill kernels wrote nothing
    for (uint32_t i = 1; i <= v.m; ++i) {
        uint32_t L;
        const uint32_t slot = row_slot<FM>(v, i, L);
        const int rb = rowbest_of<FM>(v.rowbest[(uint64_t)slot * 32u + L], v.half);
        if (rb > M) { M = rb; bi = i; }
    }
    if (M == 0) { bi = 0; return; }                                 // hw2.cpp:202-203: best cell stays (0,0)
    uint32_t L;
    const uint64_t rowbase = chunk_index<FM>(v, bi, 0, L);
    L *= (uint32_t)FM::SKEW;                                        // from here on: the row's step offset (q = j + L)
    int run = 0;                                                    // H(bi, 0) = 0
    uint32_t q = L + 1u;
    while (q <= L + v.n && bj == 0) {
        const uint32_t c = q / (uint32_t)FM::CS;
        const Chunk ch = ld(rowbase + (uint64_t)c * chunk_stride<FM>(v));
        uint32_t rem = q - c * (uint32_t)FM::CS;
        for (; rem < (uint32_t)FM::CS && q <= L + v.n; ++rem, ++q) {
            const int wi = (int)rem / FM::F, f = (int)rem - wi * FM::F;
            run += field_of<FM>(word_of<FM>(ch, wi, v.half), f) + v.gap;
            if (run == M) { bj = q - L; break; }
        }
    }
}

// ---- Smith-Waterman traceback hw2.cpp:239-257 from a known end cell ----
template <class FM, class Loader, class Sink>
B2A_HD void walk_local_from(const PairView& v, Loader ld, Sink& sink, PairResult& res, int M, uint32_t bi, uint32_t bj) {
    res.score = M; res.overlap = 0; res.n_ops = 0;
    if (M == 0) { res.end_i = res.end_j = res.start_i = res.start_j = 0; return; }
    uint32_t i = bi, j = bj, nops = 0;
    int cur = 0, best = 0;
    RowCursor<FM, Loader, true> rc, ru;                              // SW borders are 0 (hw2.cpp:193-197)
    rc.seek(v, ld, i, j);
    ru.seek(v, ld, i - 1, j);
    if (v.opt & 2) for (uint32_t k = 2; k < 2 + WALK_PF && k <= i; ++k) prefetch_row<FM>(v, ld, i - k, j > k ? j - k + 1 : 1);
    while (i > 0 && j > 0 && rc.H != 0) {                            // hw2.cpp:239
        const int H = rc.H, Hl = H - rc.D() - v.gap;
        const int Hu = ru.H, Hd = Hu - ru.D() - v.gap;
        const uint8_t pc = v.p[i - 1];
        const bool eq = pc == v.t[j - 1];
        uint32_t op;                                                 // hw2.cpp:214-222 (H != 0 here)
        if (H == Hd + (eq ? v.match : v.mismatch)) op = OP_M;
        else if (H == Hu + v.gap) op = OP_D;
        else op = OP_I;
        if (op == OP_M && eq && pc != (uint8_t)'-') { if (++cur > best) best = cur; } else cur = 0;
        if (op != OP_D) { rc.left(v, ld); ru.left(v, ld); --j; }
        if (op != OP_I) {
            rc = ru; --i;
            if (i > 0) ru.seek(v, ld, i - 1, j);
            if ((v.opt & 2) && i > 1 + WALK_PF) prefetch_row<FM>(v, ld, i - 1 - WALK_PF, j > WALK_PF ? j - WALK_PF : 1);
        }
        sink.put(op);
        ++nops;
    }
    res.end_i = bi; res.end_j = bj; res.start_i = i; res.start_j = j;
    res.overlap = best; res.n_ops = nops;
}

template <class FM, class Loader, class Sink>
B2A_HD void walk_local(const PairView& v, Loader ld, Sink& sink, PairResult& res) {
    int M; uint32_t bi, bj;
    find_local_end<FM>(v, ld, M, bi, bj);
    walk_local_from<FM>(v, ld, sink, res, M, bi, bj);
}

// 2-bit op writer: op t of a pair lands in bits 2*(t%16) of word t/16 (traceback order)
struct OpsSink {
    uint32_t* out;      // may be null: ops are counted but not stored
    uint32_t word, fill;
    uint64_t pos;
    B2A_HD explicit OpsSink(uint32_t* o) : out(o), word(0), fill(0), pos(0) {}
    B2A_HD void put(uint32_t op) {
        word |= op << (2u * fill);
        if (++fill == 16u) { if (out) out[pos] = word; ++pos; word = 0; fill = 0; }
    }
    B2A_HD void flush() { if (fill && out) out[pos] = word; }
};

// Word the fill kernels emit for F consecutive steps of one row:
//   sum_t B^(F-1-t) * (P_t - P_{t-1} - g32)  (mod 2^32),  B = 2^K,
// evaluated as  P_{F-1} + (B-1) * S - B^(F-1) * P_{-1} - g32 * (B^F - 1)/(B - 1)  with the Horner sum
// S = sum_{t<F-1} B^(F-2-t) P_t.  short16: P packs two pairs, g32 = gap * 65537, exact per 16-bit half
// because every stored P has both halves in [0, 32767] and every true field lies in [0, B-1].
// wide32: P is the plain int32 H, g32 = gap, exact because the true word is < 2^32.
template <class FM>
B2A_HD uint32_t encode_word(const uint32_t* P /* P[0] = P_{-1}, P[1..F] = P_0..P_{F-1} */, int gap) {
    constexpr int F = FM::F;
    const uint32_t g32 = FM::WBITS == 16 ? (uint32_t)gap * 65537u : (uint32_t)gap;
    if (FM::K == 32) return P[1] - P[0] - g32;
    const uint32_t B = 1u << (FM::K & 31);
    uint32_t S = 0;
    for (int t = 0; t < F - 1; ++t) S = S * B + P[t + 1];
    uint32_t Bpow = 1; for (int t = 0; t < F - 1; ++t) Bpow *= B;          // B^(F-1)
    uint32_t geo = 0; for (int t = 0; t < F; ++t) geo = geo * B + 1u;      // (B^F - 1)/(B - 1)
    return P[F] + (B - 1u) * S - Bpow * P[0] - g32 * geo;
}

} // namespace b2a
