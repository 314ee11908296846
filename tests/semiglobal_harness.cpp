// semiglobal_harness.cpp -- TEST INFRASTRUCTURE.  CPU model of the semi-global short16 record and the semi-global row walk.
//
// The record the semi-global fill (short16_fill_kernel<R, K, false, A8, true>) is specified to write: biased H (+ bias of the
// global plan) of the extended 32R-row problem, row 0 = bias (free leading text), column 0 = bias + i*gap, NW cells without a floor,
// encoded with b2a_format.h's encode_word exactly as hostmodel.cpp encodes the global and local records.  The walker is row_walk.h's
// row_walk_global<K, ..., SEMI = true>, the function short16_traceback_kernel<K, false, true> runs, started at the end cell the
// fill's epilogue is specified to find (the first maximum of the pair's own row m over columns 0..n).
#include <cstdint>
#include <cstring>
#include <vector>
#include "../bioinformatics-algorithms_b200/csrc/b2a_format.h"
#include "../bioinformatics-algorithms_b200/csrc/row_walk.h"

using namespace b2a;

namespace {

std::vector<int32_t> sg_dp(const uint8_t* p, uint32_t m, const uint8_t* t, uint32_t n, int R, int match, int mismatch, int gap,
                           int bias, uint8_t junk) {
    const uint32_t rows = 32u * (uint32_t)R;
    const size_t W = (size_t)n + 1;
    std::vector<int32_t> H((rows + 1) * W);
    for (uint32_t j = 0; j <= n; ++j) H[j] = bias;
    for (uint32_t i = 1; i <= rows; ++i) {
        H[i * W] = bias + (int)i * gap;
        const uint8_t pc = i <= m ? p[i - 1] : junk;
        for (uint32_t j = 1; j <= n; ++j) {
            int v = H[(i - 1) * W + j - 1] + (pc == t[j - 1] ? match : mismatch);
            const int l = H[i * W + j - 1] + gap, u = H[(i - 1) * W + j] + gap;
            if (l > v) v = l;
            if (u > v) v = u;
            H[i * W + j] = v;
        }
    }
    return H;
}

template <int K>
int sg_encode(const uint8_t* pa, const uint8_t* pb, uint32_t m, const uint8_t* ta, const uint8_t* tb, uint32_t n, int R,
              int match, int mismatch, int gap, int bias, uint8_t junk, Chunk* codes) {
    constexpr int F = Geo<K>::F, CS = Geo<K>::CS;
    const uint32_t NC = num_chunks(n, CS);
    const size_t W = (size_t)n + 1;
    const auto HA = sg_dp(pa, m, ta, n, R, match, mismatch, gap, bias, junk);
    const auto HB = sg_dp(pb, m, tb, n, R, match, mismatch, gap, bias, junk);
    for (uint32_t L = 0; L < 32; ++L)
        for (int r = 0; r < R; ++r) {
            const uint32_t i = L * (uint32_t)R + (uint32_t)r + 1;
            auto P = [&](int64_t q) -> uint32_t {               // packed H after step q (frozen outside columns 1..n)
                int64_t j = q - (int64_t)L;
                if (j < 0) j = 0;
                if (j > (int64_t)n) j = n;
                const int32_t a = HA[i * W + (size_t)j], b = HB[i * W + (size_t)j];
                if (a < 0 || a > 32767 || b < 0 || b > 32767) return 0xFFFFFFFFu;
                return (uint32_t)a | ((uint32_t)b << 16);
            };
            for (uint32_t c = 0; c < NC; ++c) {
                uint32_t w[3];
                for (int wi = 0; wi < 3; ++wi) {
                    const int64_t q0 = (int64_t)c * CS + (int64_t)wi * F;
                    uint32_t Pv[F + 1];
                    for (int t = 0; t <= F; ++t) {
                        Pv[t] = P(q0 - 1 + t);
                        if (Pv[t] == 0xFFFFFFFFu) return -2;                         // biased H outside [0, 32767]
                    }
                    for (int t = 0; t < F; ++t) {                                    // the delta lemma holds with the free row 0
                        const int dlo = (int)(Pv[t + 1] & 0xFFFF) - (int)(Pv[t] & 0xFFFF) - gap;
                        const int dhi = (int)(Pv[t + 1] >> 16) - (int)(Pv[t] >> 16) - gap;
                        if (dlo < 0 || dlo > (int)Geo<K>::MASK || dhi < 0 || dhi > (int)Geo<K>::MASK) return -3;
                    }
                    w[wi] = encode_word<Short16<K>>(Pv, gap);
                }
                codes[((size_t)c * 32u + L) * (uint32_t)R + (uint32_t)r] = Chunk{w[0], w[1], w[2], P((int64_t)c * CS + CS - 1)};
            }
        }
    return 0;
}

struct HostMem {
    Chunk chunk(const Chunk* p) const { return *p; }
    uint64_t word8(const uint8_t* p) const { uint64_t w; std::memcpy(&w, p, 8); return w; }
};

// text at byte offset toff (0..7) of an 8-byte aligned buffer with a zero word on each side (the walker's aligned word loads)
struct Text {
    std::vector<uint64_t> buf;
    const uint8_t* t;
    Text(const uint8_t* s, uint32_t n, uint32_t toff) : buf((n + toff + 7u) / 8u + 2u, 0ull) {
        uint8_t* b = reinterpret_cast<uint8_t*>(buf.data()) + 8 + toff;
        if (n) std::memcpy(b, s, n);
        t = b;
    }
};

struct PairPair {
    uint32_t M, N;
    std::vector<uint8_t> PA, PB, TA, TB;
    uint8_t junk;
    PairPair(const uint8_t* pa, uint32_t ma, const uint8_t* ta, uint32_t na, const uint8_t* pb, uint32_t mb, const uint8_t* tb, uint32_t nb)
        : M(ma > mb ? ma : mb), N(na > nb ? na : nb), junk(pa[0]) {
        PA.assign(M, junk); PB.assign(M, junk); TA.assign(N, 'A'); TB.assign(N, 'A');      // padding: junk cells of the other half's shape
        std::memcpy(PA.data(), pa, ma); std::memcpy(PB.data(), pb, mb);
        std::memcpy(TA.data(), ta, na); std::memcpy(TB.data(), tb, nb);
    }
};

// the epilogue's end column: first maximum of the biased row m over columns 0..n of the pair's own shape
uint32_t end_column(const uint8_t* p, uint32_t m, const uint8_t* t, uint32_t n, int match, int mismatch, int gap) {
    const auto H = sg_dp(p, m, t, n, (int)((m + 31u) / 32u), match, mismatch, gap, 0, p[0]);
    const size_t W = (size_t)n + 1;
    uint32_t bj = 0;
    for (uint32_t j = 1; j <= n; ++j) if (H[m * W + j] > H[m * W + bj]) bj = j;
    return bj;
}

template <int K>
int run_rows(const uint8_t* pa, uint32_t ma, const uint8_t* ta, uint32_t na, const uint8_t* pb, uint32_t mb, const uint8_t* tb,
             uint32_t nb, int R, int match, int mismatch, int gap, int bias, uint32_t toff, PairResult* res,
             uint32_t* opsA, uint32_t* opsB, uint32_t* iters) {
    const PairPair pp(pa, ma, ta, na, pb, mb, tb, nb);
    std::vector<Chunk> codes((size_t)R * num_chunks(pp.N, Geo<K>::CS) * 32u);
    const int rc = sg_encode<K>(pp.PA.data(), pp.PB.data(), pp.M, pp.TA.data(), pp.TB.data(), pp.N, R, match, mismatch, gap, bias,
                                pp.junk, codes.data());
    if (rc) return rc;
    for (int half = 0; half < 2; ++half) {
        const uint8_t* p = half ? pb : pa; const uint8_t* t = half ? tb : ta;
        const uint32_t m = half ? mb : ma, n = half ? nb : na;
        const Text tx(t, n, toff);
        RowWalkPair v{codes.data(), p, tx.t, m, n, (uint32_t)R, (uint32_t)short16_rmagic(R), half, match, mismatch, gap, bias, false};
        v.j_end = end_column(p, m, t, n, match, mismatch, gap);
        OpsRunSink sink(half ? opsB : opsA);
        std::memset(&res[half], 0, sizeof(PairResult));
        iters[half] = row_walk_global<K, HostMem, OpsRunSink, true>(v, HostMem{}, sink, res[half]);
        sink.flush();
        res[half].path = 1;
    }
    return 0;
}

// every cell (i, j), i = 1..m, j = 0..n, of one half decoded from the record (rw_seek), unbiased
template <int K>
int decode_rows(const uint8_t* pa, uint32_t ma, const uint8_t* ta, uint32_t na, const uint8_t* pb, uint32_t mb, const uint8_t* tb,
                uint32_t nb, int R, int match, int mismatch, int gap, int bias, int half, int32_t* out) {
    const PairPair pp(pa, ma, ta, na, pb, mb, tb, nb);
    std::vector<Chunk> codes((size_t)R * num_chunks(pp.N, Geo<K>::CS) * 32u);
    const int rc = sg_encode<K>(pp.PA.data(), pp.PB.data(), pp.M, pp.TA.data(), pp.TB.data(), pp.N, R, match, mismatch, gap, bias,
                                pp.junk, codes.data());
    if (rc) return rc;
    const uint32_t m = half ? mb : ma, n = half ? nb : na;
    const RowWalkPair v{codes.data(), nullptr, nullptr, m, n, (uint32_t)R, (uint32_t)short16_rmagic(R), half, match, mismatch, gap, bias, false};
    for (uint32_t i = 1; i <= m; ++i)
        for (uint32_t j = 0; j <= n; ++j) {
            uint64_t X; int H; uint32_t rem;
            rw_seek<K>(v, HostMem{}, i, j, X, H, rem);
            out[(size_t)(i - 1) * (n + 1) + j] = H - bias;
        }
    return 0;
}

} // namespace

extern "C" {

int sg_run_pairpair(int K, int R, int bias, const uint8_t* pa, uint32_t ma, const uint8_t* ta, uint32_t na, const uint8_t* pb,
                    uint32_t mb, const uint8_t* tb, uint32_t nb, int match, int mismatch, int gap, uint32_t toff, PairResult* res,
                    uint32_t* opsA, uint32_t* opsB, uint32_t* iters) {
    switch (K) {
        case 2: return run_rows<2>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, toff, res, opsA, opsB, iters);
        case 4: return run_rows<4>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, toff, res, opsA, opsB, iters);
        case 8: return run_rows<8>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, toff, res, opsA, opsB, iters);
    }
    return -1;
}

int sg_decode(int K, int R, int bias, const uint8_t* pa, uint32_t ma, const uint8_t* ta, uint32_t na, const uint8_t* pb, uint32_t mb,
              const uint8_t* tb, uint32_t nb, int match, int mismatch, int gap, int half, int32_t* out) {
    switch (K) {
        case 2: return decode_rows<2>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, half, out);
        case 4: return decode_rows<4>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, half, out);
        case 8: return decode_rows<8>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, half, out);
    }
    return -1;
}

// the record of one pair-pair of equal shape (m x n), as the semi-global fill writes it (white-box GPU test)
int sg_encode_record(int K, int R, int bias, const uint8_t* pa, const uint8_t* pb, uint32_t m, const uint8_t* ta, const uint8_t* tb,
                     uint32_t n, int match, int mismatch, int gap, uint8_t junk, Chunk* codes) {
    switch (K) {
        case 2: return sg_encode<2>(pa, pb, m, ta, tb, n, R, match, mismatch, gap, bias, junk, codes);
        case 4: return sg_encode<4>(pa, pb, m, ta, tb, n, R, match, mismatch, gap, bias, junk, codes);
        case 8: return sg_encode<8>(pa, pb, m, ta, tb, n, R, match, mismatch, gap, bias, junk, codes);
    }
    return -1;
}

int sg_plan(uint32_t m, uint32_t n, int match, int mismatch, int gap, int* out) {
    Short16Plan pl;
    if (!short16_plan(2, m, n, match, mismatch, gap, pl)) return 0;
    out[0] = pl.K; out[1] = pl.R; out[2] = pl.bias;
    return 1;
}

} // extern "C"
