"""Every case of the kernel instance matrix (tests/kernel_matrix.py) through the C ABI, pair by pair against the plain reference of its
mode: hw2's NW / SW oracle, the semi-global oracle, hw4's NW for B2A_TIE_HW4, hw3's affine DP.  Score, end / start cell, overlap, n_ops,
the op list byte for byte and `path` (which kernel family served the pair, as the routing model predicts).  The record cases also compare
the short16 fill's HBM record with the host model's bit for bit.  Run with `pytest -m gpu`."""
import ctypes as C

import numpy as np
import pytest

import kernel_matrix as km
import oracle_binding as ob
import semiglobal_oracle as sg
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

pkg = load_package()
CASES = km.all_cases()


@pytest.fixture(scope="module")
def eng():
    e = pkg.Engine(0)
    yield e
    e.close()


def want_pair(case, p, t):
    """the reference's (score, end_i, end_j, start_i, start_j, overlap, n_ops) and op list"""
    s = case.scoring
    if case.tie_hw4:
        score, dist, ops = ob.hw4_nw(p, t, *s)
        return (score, len(p), len(t), 0, 0, dist, len(ops)), ops
    a = sg.align(p, t, *s) if case.mode == km.SEMI else ob.align(case.mode, p, t, *s)
    return (a.score, a.end_i, a.end_j, a.start_i, a.start_j, a.overlap, len(a.ops)), a.ops


def run_hw2(eng, case):
    ps, ts = [p for p, _ in case.pairs], [t for _, t in case.pairs]
    pat, po = pkg.pack(ps)
    txt, to = pkg.pack(ts)
    s = case.scoring
    for opt, default in km.CKPT_DEFAULTS.items():
        eng.set_option(opt, case.options.get(opt, default))
    try:
        if case.seq2:
            res = eng.align_seq2_multi([case.mode], pkg.PackedSeq(pat), po, pkg.PackedSeq(txt), to, *s, want_ops=case.want_ops)[0]
        else:
            res = eng.align_packed(case.mode, pat, po, txt, to, *s, want_ops=case.want_ops, score_only=case.score_only, tie_hw4=case.tie_hw4)
    finally:
        for opt, default in km.CKPT_DEFAULTS.items():
            eng.set_option(opt, default)
    ops = None
    if case.want_ops:
        words, off = eng.copy_ops(len(ps))
        ops = [pkg.unpack_ops(words, off, k, res["n_ops"][k]) for k in range(len(ps))]
    return res, ops


def check_record(eng, case):
    """the fill's record of the case's one pair-pair equals the host model's on every real row (rows past m are junk)"""
    lib = pkg.load_library()
    lib.b2a_debug_copy_record.restype = C.c_int64
    lib.b2a_debug_copy_record.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
    (pa, ta), (pb, tb) = case.pairs
    m, n, s = len(pa), len(ta), case.scoring
    K, R, bias = km.plan(case.mode, m, n, s)
    nchunks = R * km.num_chunks(n, 3 * (16 // K)) * 32
    want, want_rb = np.zeros(nchunks * 4, np.uint32), np.zeros(R * 32, np.uint32)
    junk = min(pa + pb)
    if case.mode == km.SEMI:
        from test_semiglobal_walker_cpu import harness
        rc = harness().sg_encode_record(K, R, bias, pa, pb, m, ta, tb, n, *s, junk, want.ctypes.data_as(C.c_void_p))
    else:
        from test_format_model import PairResult
        rc = km._hm().hm_run_pairpair(case.mode, K, R, pa, pb, m, ta, tb, n, *s, bias, junk, (PairResult * 2)(), None, None,
                                      want.ctypes.data_as(C.c_void_p), want_rb.ctypes.data_as(C.c_void_p))
    assert rc == 0, (case.name, rc)
    got, got_rb = np.zeros_like(want), np.zeros_like(want_rb)
    assert lib.b2a_debug_copy_record(eng.ctx, got.ctypes.data, got.nbytes, got_rb.ctypes.data, got_rb.nbytes) == got.nbytes
    real = (np.arange(32)[:, None] * R + np.arange(R)[None, :]) < m              # [lane][row of the lane]
    g4, w4 = got.reshape(-1, 32, R, 4), want.reshape(-1, 32, R, 4)           # [chunk column][lane][row of the lane][word]
    bad = np.argwhere(np.any(g4 != w4, axis=(0, 3)) & real)
    assert len(bad) == 0, (case.name, "record differs at (lane, row)", bad[:5].tolist())
    if case.mode == km.LOCAL:
        grb, wrb = got_rb.reshape(R, 32).T, want_rb.reshape(R, 32).T
        assert np.array_equal(grb[real], wrb[real]), (case.name, "row maxima differ")


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_kernel_matrix_case_vs_reference(eng, case):
    s = case.scoring
    if case.kind == "affine_score":
        got = eng.affine_scores([p for p, _ in case.pairs], [t for _, t in case.pairs], *s)
        for k, (p, t) in enumerate(case.pairs):
            assert int(got[k]) == ob.affine_score(p, t, *s), (case.name, k, len(p), len(t))
        return
    if case.kind == "affine_align":
        sc, ops = eng.affine_align([p for p, _ in case.pairs], [t for _, t in case.pairs], *s)
        for k, (p, t) in enumerate(case.pairs):
            assert (int(sc[k]), ops[k]) == ob.affine_align(p, t, *s), (case.name, k, len(p), len(t))
        return
    _, path = km.route(case)
    res, ops = run_hw2(eng, case)
    for k, (p, t) in enumerate(case.pairs):
        assert int(res["path"][k]) == path[k], (case.name, k, len(p), len(t), int(res["path"][k]), path[k])
        if case.score_only:
            if case.mode == km.LOCAL:
                want = (ob.score_only(km.LOCAL, p, t, *s)[0],)
            elif case.mode == km.SEMI:
                want = sg.score_only(p, t, *s)
            else:
                want = (ob.score_only(km.GLOBAL, p, t, *s)[0], len(p), len(t))
            got = tuple(int(res[f][k]) for f in ("score", "end_i", "end_j")[:len(want)])
            assert got == want, (case.name, k, len(p), len(t), got, want)
            continue
        w, wops = want_pair(case, p, t)
        got = tuple(int(res[f][k]) for f in ("score", "end_i", "end_j", "start_i", "start_j", "overlap", "n_ops"))
        assert (got, ops[k]) == (w, wops), (case.name, k, len(p), len(t), got, w)
    if case.record:
        check_record(eng, case)
