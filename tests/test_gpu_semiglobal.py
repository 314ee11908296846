"""GPU tests of the semi-global mode (B2A_MODE_SEMIGLOBAL): both kernel families through the C ABI against the semi-global oracle
(tests/semiglobal_oracle.c), pair by pair -- score, end / start cell, overlap, n_ops and the op list.  Run with `pytest -m gpu`."""
import ctypes as C
import random

import numpy as np
import pytest

import oracle_binding as ob
import semiglobal_oracle as sg
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

pkg = load_package()
from bioinformatics_algorithms_b200 import workload  # noqa: E402

SEMI = pkg.SEMIGLOBAL


@pytest.fixture(scope="module")
def eng():
    e = pkg.Engine(0)
    yield e
    e.close()


def rnd(rng, n, alpha=b"ACGT"):
    return bytes(rng.choice(alpha) for _ in range(n))


def tandem(rng, n):
    unit = rnd(rng, rng.randint(1, 4))
    return (unit * (n // len(unit) + 1))[:n]


def read_from(rng, t, m, psub=0.05):
    a = rng.randint(0, max(0, len(t) - m))
    p = bytearray(t[a:a + m])
    for x in range(len(p)):
        if rng.random() < psub:
            p[x] = rng.choice(b"ACGT")
    return bytes(p) or b"A"


def want(p, t, s):
    a = sg.align(p, t, *s)
    return (a.score, a.end_i, a.end_j, a.start_i, a.start_j, a.overlap, len(a.ops)), a.ops


def check(eng, ps, ts, s, expect_path=None):
    res, ops = eng.align_batch(SEMI, ps, ts, *s, want_ops=True)
    for k, (p, t) in enumerate(zip(ps, ts)):
        got = tuple(int(res[f][k]) for f in ("score", "end_i", "end_j", "start_i", "start_j", "overlap", "n_ops"))
        w, wops = want(p, t, s)
        assert (got, ops[k]) == (w, wops), (k, len(p), len(t), s, got, w)
        if expect_path is not None:
            assert int(res["path"][k]) == expect_path, (k, len(p), len(t))
    return res, ops


def config2_pairs(n, seed):
    pat, po, txt, to = workload.config2(n, seed=seed)
    return workload.split(pat, po), workload.split(txt, to)


def test_config2_shape_two_scorings(eng):
    ps, ts = config2_pairs(2048, 481)
    check(eng, ps, ts, (1, -1, -1), expect_path=1)          # K = 2
    check(eng, ps, ts, (2, -3, -4), expect_path=1)          # K = 4


def test_tie_stress_tandem_repeats(eng):
    rng = random.Random(7)
    ps, ts = [], []
    for _ in range(600):
        t = tandem(rng, rng.randint(50, 400))
        ps.append(t[rng.randint(0, 20):][:rng.randint(1, 120)] or b"A"); ts.append(t)
    check(eng, ps, ts, (1, -1, -1))
    check(eng, ps, ts, (1, -4, -2))


def test_ragged_batches_mixed_shape_pair_pairs(eng):
    rng = random.Random(13)
    ps, ts = [], []
    for _ in range(1500):
        t = rnd(rng, rng.randint(1, 600))
        ps.append(read_from(rng, t, rng.randint(1, 200))); ts.append(t)
    for s in ((1, -1, -1), (2, -3, -4), (3, -1, -2)):
        check(eng, ps, ts, s)


@pytest.mark.parametrize("m", [1, 31, 32, 33, 511, 512, 513])
def test_short16_wide32_boundary(eng, m):
    rng = random.Random(m)
    ts = [rnd(rng, m + rng.randint(0, 300)) for _ in range(40)]
    ps = [read_from(rng, t, m) for t in ts]
    check(eng, ps, ts, (1, -1, -1), expect_path=1 if m <= 512 else 2)


def test_reads_with_an_N_take_the_eight_symbol_kernel(eng):
    rng = random.Random(3)
    ps, ts = config2_pairs(1024, 17)
    ps = [p[:40] + b"N" + p[41:] if k % 3 == 0 else p for k, p in enumerate(ps)]
    check(eng, ps, ts, (1, -1, -1), expect_path=1)
    ps = [rnd(rng, 100, b"ACGTNRY") for _ in range(200)]          # up to 7 pattern symbols: still s16x2
    ts = [rnd(rng, 300, b"ACGTNRY") for _ in range(200)]
    check(eng, ps, ts, (2, -3, -4), expect_path=1)


def test_wide32_general_alphabet_and_odd_scorings(eng):
    rng = random.Random(21)
    ps = [rnd(rng, rng.randint(1, 300), bytes(range(65, 85))) for _ in range(150)]    # > 7 pattern symbols
    ts = [rnd(rng, rng.randint(1, 700), bytes(range(65, 85))) for _ in range(150)]
    for s in ((1, -1, -1), (7, -3, -5), (300, -200, -250), (1, -1, 0), (0, -2, -1)):
        check(eng, ps, ts, s)


def test_scorings_around_the_int16_plan(eng):
    """the short16 plan's largest K = 8 scoring that still fits, and one just outside it (served by wide32)"""
    rng = random.Random(5)
    ts = [rnd(rng, 1000) for _ in range(64)]
    ps = [read_from(rng, t, 150) for t in ts]
    from test_semiglobal_walker_cpu import plan
    inside = outside = None
    for match in range(1, 128):
        s = (match, -1, -1)
        if plan(150, 1000, s) is not None:
            inside = s
        elif inside is not None:
            outside = s
            break
    assert inside and outside
    check(eng, ps, ts, inside, expect_path=1)
    check(eng, ps, ts, outside, expect_path=2)


def test_long_pair_on_wide32(eng):
    rng = random.Random(20)
    t = rnd(rng, 20000)
    p = read_from(rng, t[3000:], 15000, psub=0.08)
    check(eng, [p], [t], (1, -1, -1), expect_path=2)
    check(eng, [p], [t], (2, -3, -4), expect_path=2)


def test_fill_record_matches_host_model_bit_for_bit(eng):
    from test_semiglobal_walker_cpu import harness, plan
    lib = pkg.load_library()
    lib.b2a_debug_copy_record.restype = C.c_int64
    lib.b2a_debug_copy_record.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
    hs = harness()
    rng = random.Random(11)
    for (m, n, s) in ((150, 1000, (1, -1, -1)), (20, 20, (1, -1, -1)), (97, 130, (2, -3, -4)), (33, 70, (5, -4, -16))):
        pa, pb = (rnd(rng, m) for _ in range(2))
        ta, tb = (rnd(rng, n) for _ in range(2))
        K, R, bias = plan(m, n, s)
        CS = 3 * (16 // K)
        nchunks = R * ((n + 31 + CS) // CS) * 32
        w = np.zeros(nchunks * 4, dtype=np.uint32)
        syms = sorted(set(pa + pb))
        assert hs.sg_encode_record(K, R, bias, pa, pb, m, ta, tb, n, *s, syms[0], w.ctypes.data_as(C.c_void_p)) == 0
        eng.align_batch(SEMI, [pa, pb], [ta, tb], *s, want_ops=False)
        got = np.zeros(nchunks * 4, dtype=np.uint32)
        assert lib.b2a_debug_copy_record(eng.ctx, got.ctypes.data, got.nbytes, None, 0) == got.nbytes
        g4, w4 = got.reshape(-1, 32, R, 4), w.reshape(-1, 32, R, 4)      # rows beyond m are junk
        for L in range(32):
            for r in range(R):
                if L * R + r < m:
                    assert np.array_equal(g4[:, L, r, :], w4[:, L, r, :]), (m, n, s, L, r)


def test_score_only_equals_full_call(eng):
    rng = random.Random(9)
    ps, ts = config2_pairs(1000, 99)
    ps += [rnd(rng, 700), rnd(rng, 90, bytes(range(65, 80))), b"", b"ACG"]
    ts += [rnd(rng, 1500), rnd(rng, 400, bytes(range(65, 80))), b"ACGT", b""]
    pat, po = pkg.pack(ps); txt, to = pkg.pack(ts)
    for s in ((1, -1, -1), (2, -3, -4)):
        full = eng.align_packed(SEMI, pat, po, txt, to, *s, want_ops=True)
        so = eng.align_packed(SEMI, pat, po, txt, to, *s, score_only=True)
        for f in ("score", "end_i", "end_j"):
            assert np.array_equal(full[f], so[f]), f
    rng = random.Random(30)
    t = rnd(rng, 30000)
    p = read_from(rng, t[5000:], 20000, psub=0.1)
    so = eng.align_packed(SEMI, *pkg.pack([p]), *pkg.pack([t]), 1, -1, -1, score_only=True)
    assert (int(so["score"][0]), int(so["end_i"][0]), int(so["end_j"][0])) == sg.score_only(p, t, 1, -1, -1)


def test_multi_run_equals_single_runs(eng):
    rng = random.Random(4)
    ps, ts = config2_pairs(3000, 8)
    ps += [rnd(rng, 600), rnd(rng, 50, bytes(range(65, 80)))]; ts += [rnd(rng, 800), rnd(rng, 300, bytes(range(65, 80)))]
    pat, po = pkg.pack(ps); txt, to = pkg.pack(ts)
    single = {md: eng.align_packed(md, pat, po, txt, to, 1, -1, -1, want_ops=True) for md in (pkg.GLOBAL, pkg.LOCAL, SEMI)}
    for modes in ((pkg.GLOBAL, SEMI), (pkg.LOCAL, SEMI), (SEMI, pkg.GLOBAL)):
        got = eng.align_packed_multi(list(modes), pat, po, txt, to, 1, -1, -1, want_ops=True)
        for r, md in enumerate(modes):
            assert np.array_equal(got[r], single[md]), (modes, r)
            eng.select_run(r)
            k = len(ps) - 3
            assert pkg.unpack_ops(*eng.copy_ops(len(ps)), k, got[r]["n_ops"][k]) == \
                (sg.align(ps[k], ts[k], 1, -1, -1).ops if md == SEMI else ob.align(md, ps[k], ts[k], 1, -1, -1).ops)


def test_seq2_inputs_equal_byte_inputs(eng):
    ps, ts = config2_pairs(4000, 12)
    ps[5] = ps[5][:10] + b"N" + ps[5][11:]
    pat, po = pkg.pack(ps); txt, to = pkg.pack(ts)
    ref = eng.align_packed_multi([SEMI, pkg.LOCAL], pat, po, txt, to, 1, -1, -1, want_ops=True)
    got = eng.align_seq2_multi([SEMI, pkg.LOCAL], pkg.PackedSeq(pat), po, pkg.PackedSeq(txt), to, 1, -1, -1, want_ops=True)
    for r in range(2):
        assert np.array_equal(got[r], ref[r])


def test_ops_sink_delivers_semi_global_lists(eng):
    rng = random.Random(6)
    ps, ts = config2_pairs(12000, 6)
    ps += [rnd(rng, 700)]; ts += [rnd(rng, 900)]
    pat, po = pkg.pack(ps); txt, to = pkg.pack(ts)
    n = len(ps)
    modes = [SEMI, pkg.GLOBAL]
    eng.set_ops_sink(None)
    ref = eng.align_packed_multi(modes, pat, po, txt, to, 1, -1, -1, want_ops=True)
    off, total = eng.ops_offsets(n)
    sink = [pkg.pinned_empty(total + 5, np.uint32) for _ in range(2)]
    eng.set_option(pkg.OPT_SEG_PAIRS, 4096); eng.set_option(pkg.OPT_SEG_FIRST, 2048)
    try:
        eng.set_ops_sink(sink)
        got = eng.align_packed_multi(modes, pat, po, txt, to, 1, -1, -1, want_ops=True)
    finally:
        eng.set_ops_sink(None)
        eng.set_option(pkg.OPT_SEG_FIRST, 1 << 14); eng.set_option(pkg.OPT_SEG_PAIRS, 1 << 17)
    assert np.array_equal(got[0], ref[0])
    for k in list(range(0, n, 501)) + [n - 1]:
        assert pkg.unpack_ops(sink[0], off, k, got[0]["n_ops"][k]) == sg.align(ps[k], ts[k], 1, -1, -1).ops, k


def test_device_resident_run(eng):
    ps, ts = config2_pairs(5000, 31)
    pat, po = pkg.pack(ps); txt, to = pkg.pack(ts)
    ref = eng.align_packed(SEMI, pat, po, txt, to, 2, -3, -4)
    eng.upload(SEMI, pat, po, txt, to, 2, -3, -4)
    eng.run()
    assert np.array_equal(eng.download(len(ps)), ref)


def test_select_best_and_python_shim(eng):
    r = eng.semiGlobalAlignment(b"ACGTACGA", b"TTTTACGTACGATTTT", 1, -1, -1)
    assert (r.score, r.cigar, r.mdz, int(r.record["start_j"]), int(r.record["end_j"])) == (8, "8M", "8", 4, 12)
    assert (r.alignedPattern, r.alignedReference) == (b"ACGTACGA", b"ACGTACGA")
    p, t = b"ACGTTGCA", b"GGACGATTGCAGG"
    r = eng.semiGlobalAlignment(p, t, 1, -1, -1)
    a = sg.align(p, t, 1, -1, -1)
    assert (r.score, r.cigar, r.mdz) == (a.score, a.cigar, a.mdz)
    res, _ = eng.align_batch(SEMI, [b"AC", b"ACGT", b"ACGT"], [b"TTAC", b"GACGTC", b"ACGTAA"], 1, -1, -1, want_ops=False)
    assert pkg.select_best(SEMI, res) == 1                      # score key, first of the two 4s
    assert pkg.select_best(pkg.GLOBAL, res) == 1


def test_degenerate_shapes(eng):
    ps, ts = [b"", b"ACG", b"A", b"ACGT"], [b"ACGT", b"", b"A", b"T"]
    check(eng, ps, ts, (1, -1, -1))
    check(eng, ps, ts, (2, -3, -4))


def test_error_paths(eng):
    pat, po = pkg.pack([b"ACGT"]); txt, to = pkg.pack([b"ACGTT"])
    with pytest.raises(pkg.B2AError) as ei:
        eng.align_packed(SEMI, pat, po, txt, to, 1, -1, -1, tie_hw4=True)
    assert "rc=-1" in str(ei.value)
    with pytest.raises(pkg.B2AError) as ei:
        eng.align_packed(3, pat, po, txt, to, 1, -1, -1)
    assert "rc=-1" in str(ei.value)
    lib = pkg.load_library()
    prm = pkg.Params(SEMI, 1, -1, -1, 0)
    res = np.zeros(1, dtype=pkg.RESULT_DTYPE)
    a = np.zeros(0, dtype=pkg.ANCHOR_DTYPE)
    p = np.frombuffer(b"ACGTACGT", dtype=np.uint8); t = np.frombuffer(b"ACGTACGT", dtype=np.uint8)
    assert lib.b2a_align_anchored(eng.ctx, C.byref(prm), p.ctypes.data, 8, t.ctypes.data, 8, a.ctypes.data, 0, res.ctypes.data, None, 0) == -1
    e = pkg.Engine(0)
    try:
        e.set_option(pkg.OPT_CKPT_BYTES, 1 << 16)                  # any wide32 pair of this size would go to the checkpointed path
        rng = random.Random(1)
        t = rnd(rng, 3000)
        with pytest.raises(pkg.B2AError) as ei:
            e.align_batch(SEMI, [read_from(rng, t, 1200)], [t], 1, -1, -1)
        assert "rc=-4" in str(ei.value) and "semi-global" in str(ei.value)
        res, ops = e.align_batch(SEMI, [b"ACGT"], [b"TACGTT"], 1, -1, -1)     # the context stays usable
        assert (int(res["score"][0]), ops[0]) == (4, b"MMMM")
    finally:
        e.close()


def test_config2_full_size_one_million_pairs(eng):
    """1 M config-2 pairs: NW <= semi-global <= SW on every pair, n_ops consistent with the end / start cell on every pair, the op
    lists re-score to the score on a seeded sample of 20 000 pairs, and the oracle on 2 000 of them."""
    pat, po, txt, to = workload.config2(1_000_000, seed=481)
    g, sw, se = eng.align_packed_multi([pkg.GLOBAL, pkg.LOCAL], pat, po, txt, to, 1, -1, -1) + \
        [eng.align_packed(SEMI, pat, po, txt, to, 1, -1, -1, want_ops=True)]
    assert np.all(g["score"] <= se["score"]) and np.all(se["score"] <= sw["score"])
    m = (po[1:] - po[:-1]).astype(np.int64)
    span = se["end_j"].astype(np.int64) - se["start_j"].astype(np.int64)
    n_m = m + span - se["n_ops"].astype(np.int64)                  # 'M' columns: m = M + D, span = M + I
    assert np.all(se["end_i"] == m) and np.all(se["start_i"] == 0) and np.all(span >= 0) and np.all(n_m >= 0)
    assert np.all(n_m <= np.minimum(m, span))
    words, off = eng.copy_ops(1_000_000)
    rng = random.Random(481)
    for k in rng.sample(range(1_000_000), 20000):
        ops = pkg.unpack_ops(words, off, k, se["n_ops"][k])
        p, t = bytes(pat[po[k]:po[k + 1]]), bytes(txt[to[k]:to[k + 1]])
        pi, tj, s = 0, int(se["start_j"][k]), 0
        for op in reversed(ops):
            if op == 0x4D:
                s += 1 if p[pi] == t[tj] else -1; pi += 1; tj += 1
            elif op == 0x44:
                s -= 1; pi += 1
            else:
                s -= 1; tj += 1
        assert (s, pi, tj) == (int(se["score"][k]), len(p), int(se["end_j"][k])), k
    for k in rng.sample(range(1_000_000), 2000):
        p, t = bytes(pat[po[k]:po[k + 1]]), bytes(txt[to[k]:to[k + 1]])
        w, wops = want(p, t, (1, -1, -1))
        got = tuple(int(se[f][k]) for f in ("score", "end_i", "end_j", "start_i", "start_j", "overlap", "n_ops"))
        assert (got, pkg.unpack_ops(words, off, k, se["n_ops"][k])) == (w, wops), k
