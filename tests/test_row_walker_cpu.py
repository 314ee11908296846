"""CPU tests of the NW row walker (csrc/row_walk.h) that short16_traceback_kernel<K, false> runs.

tests/row_walker_harness.cpp builds short16 records with hostmodel.cpp's encoder and runs the walker on them; score,
start / end cell, overlap (hw2's longest exact run, or hw4's distance), n_ops and the op list must equal the oracle's.
`python tests/test_row_walker_cpu.py` prints the walker's iteration counts on config-2 pairs next to the per-cell walk's.
"""
import ctypes as C
import os
import random
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "bioinformatics-algorithms_b200"))

import oracle_binding as ob  # noqa: E402
import workload  # noqa: E402

BUILD = os.path.join(HERE, "_build")
CSRC = os.path.join(ROOT, "bioinformatics-algorithms_b200", "csrc")


class PairResult(C.Structure):
    _fields_ = [("score", C.c_int32), ("end_i", C.c_uint32), ("end_j", C.c_uint32), ("start_i", C.c_uint32),
                ("start_j", C.c_uint32), ("overlap", C.c_int32), ("n_ops", C.c_uint32), ("path", C.c_uint32)]


_lib = None


def harness():
    global _lib
    if _lib is None:
        os.makedirs(BUILD, exist_ok=True)
        so = os.path.join(BUILD, "librowwalker.so")
        srcs = [os.path.join(HERE, "row_walker_harness.cpp"), os.path.join(HERE, "hostmodel.cpp"),
                os.path.join(CSRC, "row_walk.h"), os.path.join(CSRC, "b2a_format.h"), os.path.join(CSRC, "fasta_hw2.h")]
        if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(s) for s in srcs):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-fPIC", "-shared", "-o", so, srcs[0], "-lpthread"])
        _lib = C.CDLL(so)
    return _lib


def unpack_ops(words, n_ops):
    return bytes(b"MDI"[(words[t // 16] >> (2 * (t % 16))) & 3] for t in range(n_ops))


def walk(pa, ta, pb, tb, s, hw4=False, toff=0):
    """Both halves of one pair-pair through the row walker: [(PairResult, ops, iterations)] * 2, or None if the short16
    record cannot hold the pair-pair's max shape under scoring s."""
    lib = harness()
    M, N = max(len(pa), len(pb)), max(len(ta), len(tb))
    plan = (C.c_int * 3)()
    if not lib.hm_plan(0, M, N, s[0], s[1], s[2], plan):
        return None
    K, R, bias = plan[0], plan[1], plan[2]
    res = (PairResult * 2)()
    oa = (C.c_uint32 * ((len(pa) + len(ta)) // 16 + 2))()
    obuf = (C.c_uint32 * ((len(pb) + len(tb)) // 16 + 2))()
    it = (C.c_uint32 * 2)()
    rc = lib.rw_run_pairpair(K, R, bias, pa, len(pa), ta, len(ta), pb, len(pb), tb, len(tb), s[0], s[1], s[2], int(hw4), toff,
                             res, oa, obuf, it)
    assert rc == 0, f"harness rc={rc} (K={K} R={R} bias={bias})"
    return [(res[0], unpack_ops(oa, res[0].n_ops), it[0]), (res[1], unpack_ops(obuf, res[1].n_ops), it[1])]


def check(pa, ta, pb, tb, s, hw4=False, toff=0):
    got = walk(pa, ta, pb, tb, s, hw4, toff)
    if got is None:
        return False
    for (r, ops, _), (p, t) in zip(got, ((pa, ta), (pb, tb))):
        if hw4:
            score, dist, want = ob.hw4_nw(p, t, *s)
            assert (r.score, r.overlap, r.n_ops, ops) == (score, dist, len(want), want), (p, t, s)
            assert (r.end_i, r.end_j, r.start_i, r.start_j) == (len(p), len(t), 0, 0)
        else:
            a = ob.align(ob.GLOBAL, p, t, *s)
            assert (r.score, r.end_i, r.end_j, r.start_i, r.start_j, r.overlap, r.n_ops, ops) == \
                   (a.score, a.end_i, a.end_j, a.start_i, a.start_j, a.overlap, len(a.ops), a.ops), (p, t, s)
    return True


def rnd(rng, n, alpha=b"ACGT"):
    return bytes(rng.choice(alpha) for _ in range(n))


def related(rng, m, n, alpha=b"ACGT"):
    t = rnd(rng, n, alpha)
    k = rng.randint(0, max(0, n - m))
    src = bytearray(t[k:k + m])
    for x in range(len(src)):
        if rng.random() < 0.08:
            src[x] = rng.choice(alpha)
    return (bytes(src) + rnd(rng, m, alpha))[:m], t


SCORINGS = [(1, -1, -1), (2, -3, -4), (5, -4, -16), (1, 0, 0), (3, -2, -1)]
SIZES = [1, 2, 31, 32, 33, 150, 512]


@pytest.mark.parametrize("hw4", [False, True], ids=["hw2", "hw4"])
@pytest.mark.parametrize("s", SCORINGS, ids=lambda s: "%d_%d_%d" % s)
def test_row_walker_edge_sizes_vs_oracle(s, hw4):
    rng = random.Random(hash((s, hw4)) & 0xFFFF)
    done = 0
    for m in SIZES:
        for n in SIZES:
            if m * n > 150 * 512 and (m, n) != (512, 512):
                continue
            kind = rng.random()
            if kind < 0.3:
                u = rnd(rng, rng.randint(1, 3), b"AC")
                pa, ta = (u * 600)[:m], (rnd(rng, 2, b"AC") * 600)[:n]
            elif kind < 0.7:
                pa, ta = related(rng, m, n)
            else:
                pa, ta = rnd(rng, m), rnd(rng, n)
            pb, tb = related(rng, m, n)
            done += check(pa, ta, pb, tb, s, hw4, toff=rng.randint(0, 7))
    assert done >= 20


@pytest.mark.parametrize("hw4", [False, True], ids=["hw2", "hw4"])
@pytest.mark.parametrize("s", SCORINGS, ids=lambda s: "%d_%d_%d" % s)
def test_row_walker_random_and_mixed_shapes_vs_oracle(s, hw4):
    rng = random.Random(7 + SCORINGS.index(s) * 2 + hw4)
    done = 0
    for _ in range(40):
        shapes = [(rng.randint(1, 90), rng.randint(1, 160)) for _ in range(2)]
        if rng.random() < 0.3:
            shapes[1] = shapes[0]
        pairs = []
        for m, n in shapes:
            kind = rng.random()
            if kind < 0.3:     # tie stress
                pairs.append(((rnd(rng, rng.randint(1, 3), b"AC") * 200)[:m], (rnd(rng, rng.randint(1, 3), b"AC") * 200)[:n]))
            elif kind < 0.7:
                pairs.append(related(rng, m, n))
            else:
                pairs.append((rnd(rng, m), rnd(rng, n)))
        (pa, ta), (pb, tb) = pairs
        done += check(pa, ta, pb, tb, s, hw4, toff=rng.randint(0, 7))
    assert done >= 30


def config2_pairs(n_pairs, tie_fraction):
    pat, po, txt, to = workload.config2(n_pairs, seed=1234, tie_fraction=tie_fraction)
    return ([bytes(pat[po[k]:po[k + 1]]) for k in range(n_pairs)], [bytes(txt[to[k]:to[k + 1]]) for k in range(n_pairs)])


@pytest.mark.parametrize("hw4", [False, True], ids=["hw2", "hw4"])
def test_row_walker_config2_ties_vs_oracle(hw4):
    ps, ts = config2_pairs(96, 0.5)
    for k in range(0, len(ps), 2):
        assert check(ps[k], ts[k], ps[k + 1], ts[k + 1], (1, -1, -1), hw4, toff=k % 8)


def iteration_counts(n_pairs=2048, tie_fraction=0.0):
    """Row-walker iterations per pair, and the per-cell walk's loop counts (the run along the last row, then one step per
    cell until row 0 or column 0) derived from the op list, for config-2 pairs; both also as the maximum over each group
    of 32 consecutive pairs (one warp of the traceback kernel)."""
    ps, ts = config2_pairs(n_pairs, tie_fraction)
    new, run_a, steps = [], [], []
    for k in range(0, n_pairs, 2):
        got = walk(ps[k], ts[k], ps[k + 1], ts[k + 1], (1, -1, -1))
        for (r, ops, it), p in zip(got, (ps[k], ps[k + 1])):
            new.append(it)
            lead = len(ops) - len(ops.lstrip(b"I")) if len(p) >= 2 else 0
            tail = 0 if ops[-1:] == b"M" else len(ops) - len(ops.rstrip(ops[-1:]))
            run_a.append(lead)
            steps.append(len(ops) - lead - tail)
    new, run_a, steps = (np.array(x, dtype=np.int64) for x in (new, run_a, steps))
    warp = lambda x: x.reshape(-1, 32).max(axis=1)  # noqa: E731
    return {"pairs": n_pairs,
            "row_walker_iterations_mean": float(new.mean()), "row_walker_iterations_warp_max_mean": float(warp(new).mean()),
            "per_cell_last_row_run_mean": float(run_a.mean()), "per_cell_steps_mean": float(steps.mean()),
            "per_cell_warp_max_mean": float((warp(run_a) + warp(steps)).mean())}


def test_row_walker_iterations_config2():
    c = iteration_counts(256)
    # a staircase of ~150 climbs: about one iteration per row plus the windows that end at a chunk edge
    assert 150 <= c["row_walker_iterations_mean"] < 0.4 * c["per_cell_steps_mean"], c


if __name__ == "__main__":
    import json
    print(json.dumps(iteration_counts(), indent=1))
