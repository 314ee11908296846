"""CPU tests of the semi-global short16 path: tests/semiglobal_harness.cpp builds the record the semi-global fill is specified to
write and runs row_walk.h's semi-global walk (the function short16_traceback_kernel<K, false, true> runs) from the end cell the
fill's epilogue is specified to find.  Score, end / start cell, overlap, n_ops and the op list must equal the semi-global oracle's;
the record must decode to the oracle's H matrix.  `python tests/test_semiglobal_walker_cpu.py` prints iteration counts on config-2
pairs next to the global walk's.
"""
import ctypes as C
import hashlib
import os
import random
import subprocess
import sys
import tempfile

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "bioinformatics-algorithms_b200"))

import semiglobal_oracle as sg  # noqa: E402
import workload  # noqa: E402
from test_semiglobal_cpu import py_semiglobal  # noqa: E402

CSRC = os.path.join(ROOT, "bioinformatics-algorithms_b200", "csrc")
SCORINGS = [(1, -1, -1), (2, -3, -4), (1, -4, -2), (3, -1, -2), (5, -4, -3)]


class PairResult(C.Structure):
    _fields_ = [("score", C.c_int32), ("end_i", C.c_uint32), ("end_j", C.c_uint32), ("start_i", C.c_uint32),
                ("start_j", C.c_uint32), ("overlap", C.c_int32), ("n_ops", C.c_uint32), ("path", C.c_uint32)]


_lib = None


def harness():
    """tests/semiglobal_harness.cpp compiled into a temporary directory (keyed by the sources' hash)"""
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "semiglobal_harness.cpp"), os.path.join(CSRC, "row_walk.h"), os.path.join(CSRC, "b2a_format.h")]
        h = hashlib.sha256()
        for s in srcs:
            with open(s, "rb") as f:
                h.update(f.read())
        so = os.path.join(tempfile.gettempdir(), f"b2a_semiglobal_harness_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = so + f".{os.getpid()}.tmp"
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", tmp, srcs[0]])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def unpack_ops(words, n_ops):
    return bytes(b"MDI"[(words[t // 16] >> (2 * (t % 16))) & 3] for t in range(n_ops))


def plan(M, N, s):
    out = (C.c_int * 3)()
    return tuple(out) if harness().sg_plan(M, N, s[0], s[1], s[2], out) else None


def walk(pa, ta, pb, tb, s, toff=0):
    """Both halves of one pair-pair through the semi-global walk: [(PairResult, ops, iterations)] * 2, or None if the short16
    record cannot hold the pair-pair's max shape under scoring s."""
    pl = plan(max(len(pa), len(pb)), max(len(ta), len(tb)), s)
    if pl is None:
        return None
    K, R, bias = pl
    res = (PairResult * 2)()
    oa = (C.c_uint32 * ((len(pa) + len(ta)) // 16 + 2))()
    ob_ = (C.c_uint32 * ((len(pb) + len(tb)) // 16 + 2))()
    it = (C.c_uint32 * 2)()
    rc = harness().sg_run_pairpair(K, R, bias, pa, len(pa), ta, len(ta), pb, len(pb), tb, len(tb), s[0], s[1], s[2], toff,
                                   res, oa, ob_, it)
    assert rc == 0, f"harness rc={rc} (K={K} R={R} bias={bias})"
    return [(res[0], unpack_ops(oa, res[0].n_ops), it[0]), (res[1], unpack_ops(ob_, res[1].n_ops), it[1])]


def check(pa, ta, pb, tb, s, toff=0):
    got = walk(pa, ta, pb, tb, s, toff)
    if got is None:
        return False
    for (r, ops, _), (p, t) in zip(got, ((pa, ta), (pb, tb))):
        a = sg.align(p, t, *s)
        assert (r.score, r.end_i, r.end_j, r.start_i, r.start_j, r.overlap, r.n_ops, ops) == \
               (a.score, a.end_i, a.end_j, a.start_i, a.start_j, a.overlap, len(a.ops), a.ops), (p, t, s)
    return True


def config2_pairs(n_pairs, seed=481):
    pat, po, txt, to = workload.config2(n_pairs, seed=seed)
    return ([bytes(pat[po[k]:po[k + 1]]) for k in range(n_pairs)], [bytes(txt[to[k]:to[k + 1]]) for k in range(n_pairs)])


def rnd(rng, n, alpha=b"ACGT"):
    return bytes(rng.choice(alpha) for _ in range(n))


def tandem(rng, n):
    unit = rnd(rng, rng.randint(1, 4))
    return (unit * (n // len(unit) + 1))[:n]


@pytest.mark.parametrize("s", SCORINGS)
def test_walker_equals_oracle_random_and_tandem(s):
    rng = random.Random(11 + s[0] * 7 - s[1])
    done = 0
    for k in range(120):
        m, n = rng.randint(1, 70), rng.randint(1, 160)
        f = tandem if k % 2 else rnd
        pa, ta = f(rng, m), f(rng, n)
        done += check(pa, ta, pa, ta, s, toff=k % 8)
    assert done >= 100


@pytest.mark.parametrize("s", SCORINGS)
def test_walker_mixed_shape_pair_pairs(s):
    rng = random.Random(23 - s[2])
    done = 0
    for k in range(80):
        ma, mb = rng.randint(1, 64), rng.randint(1, 64)
        na, nb = rng.randint(1, 140), rng.randint(1, 140)
        done += check(rnd(rng, ma), rnd(rng, na), tandem(rng, mb), tandem(rng, nb), s, toff=(3 * k) % 8)
    assert done >= 60


@pytest.mark.parametrize("K_scoring", [(1, -1, -1), (2, -3, -4), (5, -40, -60)])
def test_walker_delta_widths(K_scoring):
    """K = 2, 4 and 8 records (delta span 4, 11 and 161)"""
    rng = random.Random(3)
    K = plan(40, 100, K_scoring)[0]
    assert K == {(1, -1, -1): 2, (2, -3, -4): 4, (5, -40, -60): 8}[K_scoring]
    for _ in range(40):
        pa, ta = rnd(rng, rng.randint(1, 40)), rnd(rng, rng.randint(1, 100))
        assert check(pa, ta, pa, ta, K_scoring)


@pytest.mark.parametrize("m", [1, 2, 31, 32, 33, 63, 64, 65, 255, 256, 257, 511, 512])
def test_walker_edge_sizes(m):
    rng = random.Random(m)
    t = rnd(rng, m + 40)
    a = rng.randint(0, 40)
    p = bytearray(t[a:a + m])
    for _ in range(max(1, m // 20)):
        p[rng.randrange(m)] = rng.choice(b"ACGT")
    assert check(bytes(p), t, bytes(p), t, (1, -1, -1))
    assert check(bytes(p), t[:max(1, m // 2)], rnd(rng, m), t, (1, -1, -1))


def test_walker_config2_pairs_with_ties():
    pats, txts = config2_pairs(300)
    for s in [(1, -1, -1), (2, -3, -4)]:
        for k in range(0, 300, 2):
            assert check(pats[k], txts[k], pats[k + 1], txts[k + 1], s, toff=k % 8)
    rng = random.Random(9)
    for _ in range(30):                                         # tandem repeats: many equal maxima in row m
        t = tandem(rng, 300)
        assert check(t[5:155], t, t[17:167], t, (1, -1, -1))


@pytest.mark.parametrize("s", [(1, -1, -1), (2, -3, -4), (1, -4, -2)])
def test_record_decodes_to_oracle_matrix(s):
    rng = random.Random(41)
    lib = harness()
    for k in range(25):
        ma, mb = rng.randint(1, 80), rng.randint(1, 80)
        na, nb = rng.randint(1, 90), rng.randint(1, 90)
        pa, ta, pb, tb = rnd(rng, ma), rnd(rng, na), tandem(rng, mb), tandem(rng, nb)
        pl = plan(max(ma, mb), max(na, nb), s)
        assert pl is not None
        for half, (p, t) in enumerate(((pa, ta), (pb, tb))):
            m, n = len(p), len(t)
            out = (C.c_int32 * (m * (n + 1)))()
            assert lib.sg_decode(pl[0], pl[1], pl[2], pa, ma, ta, na, pb, mb, tb, nb, s[0], s[1], s[2], half, out) == 0
            H = full_matrix(p, t, *s)
            assert [out[(i - 1) * (n + 1) + j] for i in range(1, m + 1) for j in range(n + 1)] == \
                   [H[i][j] for i in range(1, m + 1) for j in range(n + 1)]


def full_matrix(P, T, match, mismatch, gap):
    m, n = len(P), len(T)
    H = [[0] * (n + 1) for _ in range(m + 1)]
    for i in range(1, m + 1):
        H[i][0] = i * gap
        for j in range(1, n + 1):
            H[i][j] = max(H[i - 1][j - 1] + (match if P[i - 1] == T[j - 1] else mismatch), H[i][j - 1] + gap, H[i - 1][j] + gap)
    return H


def test_python_statement_agrees_on_walker_cases():
    rng = random.Random(2)
    for _ in range(50):
        p, t = rnd(rng, rng.randint(1, 20)), rnd(rng, rng.randint(1, 50))
        e = py_semiglobal(p, t, 2, -3, -4)
        a = sg.align(p, t, 2, -3, -4)
        assert (e["score"], e["end_j"], e["start_j"], e["ops"]) == (a.score, a.end_j, a.start_j, a.ops)


if __name__ == "__main__":
    sys.path.insert(0, HERE)
    import test_row_walker_cpu as rwg
    pats, txts = config2_pairs(2000)
    for s in [(1, -1, -1), (2, -3, -4)]:
        semi, glob, warps_s, warps_g = [], [], [], []
        for k in range(0, 2000, 2):
            a = walk(pats[k], txts[k], pats[k + 1], txts[k + 1], s)
            g = rwg.walk(pats[k], txts[k], pats[k + 1], txts[k + 1], s)
            semi += [a[0][2], a[1][2]]
            glob += [g[0][2], g[1][2]]
        for w in range(0, len(semi), 32):
            warps_s.append(max(semi[w:w + 32]))
            warps_g.append(max(glob[w:w + 32]))
        print(f"scoring {s}: iterations per pair  semi-global {sum(semi) / len(semi):.1f}  global {sum(glob) / len(glob):.1f};"
              f"  per warp of 32 walks (max)  semi-global {sum(warps_s) / len(warps_s):.1f}  global {sum(warps_g) / len(warps_g):.1f}")
