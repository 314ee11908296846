// row_walker_harness.cpp -- TEST INFRASTRUCTURE.  Runs the NW row walker of csrc/row_walk.h (the function the short16
// traceback kernel runs for global mode) on CPU-built short16 records.  The record comes from hostmodel.cpp's encoder,
// so the walker reads exactly the bytes the fill kernel is specified to write.  Pair-pairs may mix shapes: the record is
// built for max(m) x max(n) with the shorter pattern / text padded, as the fill kernel sweeps it.
#include "hostmodel.cpp"
#include "../bioinformatics-algorithms_b200/csrc/row_walk.h"

namespace {

struct HostMem {
    Chunk chunk(const Chunk* p) const { return *p; }
    uint64_t word8(const uint8_t* p) const { uint64_t w; std::memcpy(&w, p, 8); return w; }
};

// text at byte offset toff (0..7) of an 8-byte aligned buffer with a zero word on each side, so the walker's aligned
// word loads read inside the buffer
struct Text {
    std::vector<uint64_t> buf;
    const uint8_t* t;
    Text(const uint8_t* s, uint32_t n, uint32_t toff) : buf((n + toff + 7u) / 8u + 2u, 0ull) {
        uint8_t* b = reinterpret_cast<uint8_t*>(buf.data()) + 8 + toff;
        if (n) std::memcpy(b, s, n);
        t = b;
    }
};

template <int K>
int run_rows(const uint8_t* pa, uint32_t ma, const uint8_t* ta, uint32_t na, const uint8_t* pb, uint32_t mb, const uint8_t* tb,
             uint32_t nb, int R, int match, int mismatch, int gap, int bias, int hw4, uint32_t toff, PairResult* res,
             uint32_t* opsA, uint32_t* opsB, uint32_t* iters) {
    const uint32_t M = ma > mb ? ma : mb, N = na > nb ? na : nb;
    const uint8_t junk = pa[0];
    std::vector<uint8_t> PA(M, junk), PB(M, junk), TA(N, 'A'), TB(N, 'A');    // padding: junk cells of the other half's shape
    std::memcpy(PA.data(), pa, ma); std::memcpy(PB.data(), pb, mb);
    std::memcpy(TA.data(), ta, na); std::memcpy(TB.data(), tb, nb);
    std::vector<Chunk> codes((size_t)R * num_chunks(N, Geo<K>::CS) * 32u);
    const int rc = encode<K>(0, PA.data(), PB.data(), M, TA.data(), TB.data(), N, R, match, mismatch, gap, bias, junk, codes.data(), nullptr);
    if (rc) return rc;
    for (int half = 0; half < 2; ++half) {
        const Text tx(half ? tb : ta, half ? nb : na, toff);
        const RowWalkPair v{codes.data(), half ? pb : pa, tx.t, half ? mb : ma, half ? nb : na, (uint32_t)R, (uint32_t)short16_rmagic(R),
                            half, match, mismatch, gap, bias, hw4 != 0};
        OpsRunSink sink(half ? opsB : opsA);
        std::memset(&res[half], 0, sizeof(PairResult));
        iters[half] = row_walk_global<K>(v, HostMem{}, sink, res[half]);
        sink.flush();
        res[half].path = 1;
    }
    return 0;
}

} // namespace

extern "C" int rw_run_pairpair(int K, int R, int bias, const uint8_t* pa, uint32_t ma, const uint8_t* ta, uint32_t na,
                               const uint8_t* pb, uint32_t mb, const uint8_t* tb, uint32_t nb, int match, int mismatch, int gap,
                               int hw4, uint32_t toff, PairResult* res, uint32_t* opsA, uint32_t* opsB, uint32_t* iters) {
    switch (K) {
        case 2: return run_rows<2>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, hw4, toff, res, opsA, opsB, iters);
        case 4: return run_rows<4>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, hw4, toff, res, opsA, opsB, iters);
        case 8: return run_rows<8>(pa, ma, ta, na, pb, mb, tb, nb, R, match, mismatch, gap, bias, hw4, toff, res, opsA, opsB, iters);
    }
    return -1;
}
