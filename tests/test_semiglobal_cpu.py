"""Semi-global mode (B2A_MODE_SEMIGLOBAL) on the CPU: the C oracle against an independent pure-Python statement of the
contract (include/b2align.h), op for op, plus the properties that tie the mode to hw2's global and local modes."""
import random

import pytest

import oracle_binding as ob
import semiglobal_oracle as sg

SCORINGS = [(1, -1, -1), (2, -3, -4), (1, -4, -2), (3, -1, -2), (5, -4, -3)]


def py_semiglobal(P: bytes, T: bytes, match, mismatch, gap):
    """The contract restated: H(0, j) = 0, H(i, 0) = i gap, hw2's cells and tie order d > l > u, end cell = first
    maximum of row m, traceback (i>0, j>0, 'd') -> M, (i>0, 'u') -> D, (j>0, 'l') -> I, stop at row 0."""
    m, n = len(P), len(T)
    H = [[0] * (n + 1) for _ in range(m + 1)]
    d = [[""] * (n + 1) for _ in range(m + 1)]
    for i in range(1, m + 1):
        H[i][0] = i * gap
        d[i][0] = "u"
        for j in range(1, n + 1):
            v, c = H[i - 1][j - 1] + (match if P[i - 1] == T[j - 1] else mismatch), "d"
            if H[i][j - 1] + gap > v:
                v, c = H[i][j - 1] + gap, "l"
            if H[i - 1][j] + gap > v:
                v, c = H[i - 1][j] + gap, "u"
            H[i][j], d[i][j] = v, c
    last = H[m]
    bj = last.index(max(last))
    i, j, ops, cur, best = m, bj, bytearray(), 0, 0
    while i > 0:
        c = d[i][j]
        if j > 0 and c == "d":
            ops.append(ord("M"))
            if P[i - 1] == T[j - 1] and P[i - 1] != ord("-"):
                cur += 1
                best = max(best, cur)
            else:
                cur = 0
            i, j = i - 1, j - 1
        elif c == "u":
            ops.append(ord("D")); cur = 0; i -= 1
        else:
            assert j > 0 and c == "l"
            ops.append(ord("I")); cur = 0; j -= 1
    return dict(score=last[bj], end_i=m, end_j=bj, start_i=0, start_j=j, overlap=best, ops=bytes(ops))


def rescore(ops: bytes, P: bytes, T: bytes, start_j, match, mismatch, gap):
    """score of an op list (traceback order) and the bases it consumes"""
    pi, tj, s = 0, start_j, 0
    for op in reversed(ops):
        if op == ord("M"):
            s += match if P[pi] == T[tj] else mismatch
            pi += 1; tj += 1
        elif op == ord("D"):
            s += gap; pi += 1
        else:
            s += gap; tj += 1
    return s, pi, tj


def rnd(rng, n, alpha=b"ACGT"):
    return bytes(rng.choice(alpha) for _ in range(n))


def tandem(rng, n):
    unit = rnd(rng, rng.randint(1, 4))
    return (unit * (n // len(unit) + 1))[:n]


def cases(seed, count):
    rng = random.Random(seed)
    for k in range(count):
        kind = k % 4
        if kind == 0:
            P, T = rnd(rng, rng.randint(1, 14)), rnd(rng, rng.randint(1, 40))
        elif kind == 1:
            P, T = tandem(rng, rng.randint(1, 16)), tandem(rng, rng.randint(1, 40))
        elif kind == 2:
            alpha = bytes(range(33, 33 + rng.randint(2, 12)))
            P, T = rnd(rng, rng.randint(1, 14), alpha), rnd(rng, rng.randint(1, 40), alpha)
        else:                                                   # a read cut from its window and mutated
            T = rnd(rng, rng.randint(8, 40))
            a = rng.randint(0, len(T) - 4)
            P = bytearray(T[a:a + rng.randint(3, min(16, len(T) - a))])
            for _ in range(rng.randint(0, 2)):
                x = rng.randrange(len(P))
                P[x] = rng.choice(b"ACGT")
            P = bytes(P)
        yield P, T


@pytest.mark.parametrize("scoring", SCORINGS)
def test_oracle_matches_python_statement(scoring):
    for P, T in cases(hash(scoring) & 0xFFFF, 700):
        a = sg.align(P, T, *scoring)
        e = py_semiglobal(P, T, *scoring)
        got = dict(score=a.score, end_i=a.end_i, end_j=a.end_j, start_i=a.start_i, start_j=a.start_j,
                   overlap=a.overlap, ops=a.ops)
        assert got == e, (P, T, scoring)


@pytest.mark.parametrize("scoring", SCORINGS)
def test_score_is_best_global_over_substrings(scoring):
    rng = random.Random(7 + scoring[1])
    for _ in range(150):
        P, T = rnd(rng, rng.randint(1, 8)), rnd(rng, rng.randint(0, 12))
        want = max(ob.align(ob.GLOBAL, P, T[a:b], *scoring).score for a in range(len(T) + 1) for b in range(a, len(T) + 1))
        assert sg.align(P, T, *scoring).score == want, (P, T)


@pytest.mark.parametrize("scoring", SCORINGS)
def test_between_global_and_local_and_rescores(scoring):
    for P, T in cases(100 + scoring[0], 500):
        a = sg.align(P, T, *scoring)
        assert ob.align(ob.GLOBAL, P, T, *scoring).score <= a.score <= ob.align(ob.LOCAL, P, T, *scoring).score
        s, pi, tj = rescore(a.ops, P, T, a.start_j, *scoring)
        assert (s, pi, tj) == (a.score, len(P), a.end_j), (P, T)
        assert a.start_j <= a.end_j
        assert a.ops.count(b"M") + a.ops.count(b"D") == len(P)


@pytest.mark.parametrize("scoring", SCORINGS)
def test_score_only_matches_full(scoring):
    for P, T in cases(300 + scoring[2], 400):
        a = sg.align(P, T, *scoring)
        assert sg.score_only(P, T, *scoring) == (a.score, a.end_i, a.end_j)


def test_score_only_long_pair():
    rng = random.Random(5)
    T = rnd(rng, 3000)
    P = T[1200:1500]
    a = sg.align(P, T, 2, -3, -4)
    assert (a.score, a.end_j, a.start_j) == (600, 1500, 1200)
    assert sg.score_only(P, T, 2, -3, -4) == (600, 300, 1500)


@pytest.mark.parametrize("scoring", SCORINGS)
def test_degenerate_shapes(scoring):
    match, mismatch, gap = scoring
    a = sg.align(b"", b"ACGT", *scoring)
    assert (a.score, a.end_i, a.end_j, a.start_i, a.start_j, a.ops) == (0, 0, 0, 0, 0, b"")
    a = sg.align(b"ACG", b"", *scoring)
    assert (a.score, a.end_i, a.end_j, a.start_i, a.start_j, a.ops) == (3 * gap, 3, 0, 0, 0, b"DDD")
    assert sg.score_only(b"ACG", b"", *scoring) == (3 * gap, 3, 0)
    assert sg.score_only(b"", b"ACG", *scoring) == (0, 0, 0)


def test_ties_take_the_first_maximum():
    # the read fits twice; the walk ends at the leftmost copy's end and starts at its first base
    a = sg.align(b"ACGT", b"TTACGTTTACGTTT", 1, -1, -1)
    assert (a.score, a.end_j, a.start_j, a.cigar) == (4, 6, 2, "4M")
    # an empty stretch of text ties with nothing: every column of row m below 0 leaves j* = 0
    a = sg.align(b"AA", b"CC", 1, -5, -1)
    assert (a.score, a.end_j, a.start_j, a.ops) == (-2, 0, 0, b"DD")
