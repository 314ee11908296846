"""The kernel instance matrix: one table of cases that, together, make every kernel instance of libb2align.so serve a pair.

TEST INFRASTRUCTURE.  tests/test_kernel_matrix_cpu.py checks that the union of `instances(case)` over `CASES` equals the list of kernel
entries compiled into the library (microbench_kernel excepted), so a new instance without a case -- or a case that names an instance
the library no longer has -- fails the suite.  tests/test_gpu_kernel_matrix.py runs every case through the C ABI and compares each pair
with the plain reference of its mode.

`instances(case)` restates the engine's routing (b2a_api.cu) on the host:
  * a pair is a short16 pair iff every run's short16 plan (hm_plan) accepts its shape and the call is not score-only; pairs of one
    shape are zipped into pair-pairs, leftovers of different shapes are zipped in (R, n, m) order, and what is left runs alone;
  * a pair-pair takes the 8-symbol fill (A8) iff one of its patterns holds a byte outside the four most frequent pattern bytes of
    the segment, and goes to wide32 instead if one of its patterns holds more than 7 distinct bytes;
  * wide32 uses ALPHA4 (the int8 PRMT tables) iff the whole batch holds <= 4 distinct pattern bytes and match / mismatch fit int8;
  * score-only launches use the K = 2 wide32 fill;
  * a wide32 pair whose record exceeds B2A_OPT_CKPT_BYTES takes the checkpointed path: a score pass (the KEEPCOL instance when the
    text is longer than 2 << B2A_OPT_CKPT_COLS), local mode's wide32_first_best_row_kernel, then record fills of band groups and
    wide32_ckpt_walk_kernel -- unless the local score is 0, which needs no walk.
Every batch here holds fewer than 16 384 pairs, which the engine never splits: one segment is the whole batch, so "the segment's
pattern bytes" are the batch's.  An instance counts for a case when it does work for one of the case's pairs: the 8-symbol fill is
launched behind every 4-symbol fill, but returns at once unless a flagged pair-pair exists.

Instances are tuples (kernel name, template arguments), e.g. ("short16_fill_kernel", (16, 8, 0, 1, 0)) for
short16_fill_kernel<16, 8, LOCAL = false, A8 = true, SEMI = false>.
"""
import ctypes as C
import random
from dataclasses import dataclass, field
from functools import lru_cache

import oracle_binding as ob

GLOBAL, LOCAL, SEMI = 0, 1, 2
OPT_CKPT_BYTES, OPT_CKPT_GROUP, OPT_CKPT_COLS = 6, 7, 8
CKPT_DEFAULTS = {OPT_CKPT_BYTES: 48 << 30, OPT_CKPT_GROUP: 1 << 30, OPT_CKPT_COLS: 13}
SEG_PAIRS = 16384
WIDE_R, AFFINE_R_SCORE = 4, 8
R_CLASSES = (1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 16)
ACGT = b"ACGT"
PROT = b"ACDEFGHIKLMNPQRSTVWY"


@dataclass
class Case:
    name: str
    kind: str                            # "hw2", "affine_score", "affine_align"
    scoring: tuple
    pairs: list                          # [(pattern bytes, text bytes)]
    mode: int = GLOBAL
    want_ops: bool = True
    score_only: bool = False
    tie_hw4: bool = False
    seq2: bool = False                   # 2-bit packed inputs (b2a_align_batch_multi_seq2)
    options: dict = field(default_factory=dict)
    record: bool = False                 # one pair-pair: also compare the fill's record with the host model


# ---- host models (tests/hostmodel.cpp) ----
@lru_cache(maxsize=None)
def _hm():
    from test_format_model import hostmodel
    return hostmodel()


@lru_cache(maxsize=None)
def plan(mode, m, n, s):
    """(K, R, bias) of the short16 plan, or None when the s16x2 record cannot hold the shape"""
    out = (C.c_int * 3)()
    return tuple(out) if _hm().hm_plan(mode, m, n, s[0], s[1], s[2], out) else None


def k_wide(s):
    return _hm().hm_delta_bits_wide(*s)


def short16_r(m):
    r = (m + 31) // 32
    return r if r <= 8 else (10 if r <= 10 else (12 if r <= 12 else 16))


def num_chunks(n, cs):
    return (n + 31 + cs) // cs


def _top4(pats):
    hist = {}
    for p in pats:
        for b in p:
            hist[b] = hist.get(b, 0) + 1
    top = sorted(hist, key=lambda b: (-hist[b], b))[:4]
    return set(top), len(hist) > 4


def pair_pairs(case):
    """The engine's pair-pair plan of one segment (b2a_api.cu, batch_prepare pass 2): ({R: [(a, b)]}, [wide32 pair indices])"""
    s = case.scoring
    def plan_all(m, n):
        return None if case.score_only else plan(case.mode, m, n, s)
    pps, wide, pending = {}, [], {}
    last = None                                                   # (key, index) of a pair waiting for its same-shape neighbour
    def park(key, idx):
        if key in pending:
            pps.setdefault(short16_r(key[0]), []).append((pending.pop(key), idx))
        else:
            pending[key] = idx
    for q, (p, t) in enumerate(case.pairs):
        key = (len(p), len(t))
        pl = plan_all(*key)
        if pl is None:
            wide.append(q)
            continue
        if last is not None and key == last[0]:
            pps.setdefault(pl[1], []).append((last[1], q))
            last = None
            continue
        if last is not None:
            park(*last)
            last = None
        if key in pending:
            pps.setdefault(pl[1], []).append((pending.pop(key), q))
        else:
            last = (key, q)
    if last is not None:
        park(*last)
    left = sorted((short16_r(m), n, m, idx) for (m, n), idx in pending.items())
    mix_ok = case.mode != LOCAL or (s[2] < 0 and s[1] < 0)
    q = 0
    while q < len(left):
        R, n, m, idx = left[q]
        if mix_ok and q + 1 < len(left) and left[q + 1][0] == R:
            _, n2, m2, idx2 = left[q + 1]
            both = plan_all(max(m, m2), max(n, n2))
            if both is not None and both[1] == R:
                pps.setdefault(R, []).append((min(idx, idx2), max(idx, idx2)))
                q += 2
                continue
        pps.setdefault(R, []).append((idx, idx))
        q += 1
    return pps, wide


def route(case):
    """(set of instances the case makes serve a pair, per-pair `path` the result records must show: 1 short16, 2 wide32)"""
    if case.kind != "hw2":
        return _route_affine(case)
    s = case.scoring
    match, mismatch, gap = s
    local, semi = int(case.mode == LOCAL), int(case.mode == SEMI)
    pats = [p for p, _ in case.pairs]
    inst = {("alphabet_finish_kernel", ())}
    if sum(map(len, pats)):
        inst.add(("alphabet_kernel", ()))
    if case.seq2:
        inst.add(("seq2_expand_kernel", ()))
        if any(b not in ACGT for p, t in case.pairs for b in p + t):
            inst.add(("seq2_patch_kernel", ()))
    path = [0] * len(case.pairs)
    pps, wide = pair_pairs(case)
    top4, too_many = _top4(pats)
    if pps:
        inst |= {("dirty_kernel", ()), ("dirty_compact_kernel", ())}
        K = plan(case.mode, 1, 1, s)[0]
    for R, lst in pps.items():
        for a, b in lst:
            halves = (a,) if a == b else (a, b)
            if too_many and any(x not in top4 for h in halves for x in pats[h]):
                if any(len(set(pats[h])) > 7 for h in halves):
                    wide += list(halves)
                    continue
                inst.add(("short16_fill_kernel", (R, K, local, 1, semi)))
            else:
                inst.add(("short16_fill_kernel", (R, K, local, 0, semi)))
            inst.add(("short16_traceback_kernel", (K, local, semi)))
            for h in halves:
                path[h] = 1
    if not wide:
        return inst, path
    alpha4 = int(len(set(b for p in pats for b in p)) <= 4 and -128 <= match <= 127 and -128 <= mismatch <= 127)
    Kw, store = k_wide(s), not case.score_only
    cs = 2 * (32 // Kw)
    opt = {**CKPT_DEFAULTS, **case.options}
    regular = False
    for q in sorted(set(wide)):
        p, t = case.pairs[q]
        m, n = len(p), len(t)
        path[q] = 2
        nbands = (m + 32 * WIDE_R - 1) // (32 * WIDE_R) if m and n else 0
        if store and nbands * WIDE_R * num_chunks(n, cs) * 32 * 16 > opt[OPT_CKPT_BYTES]:
            assert not semi, "semi-global mode has no checkpointed path"
            keepcol = int(n > (2 << opt[OPT_CKPT_COLS]))
            inst.add(("wide32_fill_kernel", (2, local, 0, alpha4, keepcol, 0)))
            if local:
                inst.add(("wide32_first_best_row_kernel", ()))
                if ob.score_only(LOCAL, p, t, *s)[0] == 0:
                    continue                                      # no positive cell: the empty alignment, no walk
            inst.add(("wide32_fill_kernel", (Kw, local, 1, alpha4, 0, 0)))
            inst.add(("wide32_ckpt_walk_kernel", (Kw, local)))
            continue
        regular = True
        if nbands:
            inst.add(("wide32_fill_kernel", (Kw if store else 2, local, int(store), alpha4, 0, semi)))
    if regular:
        inst.add(("wide32_traceback_kernel", (Kw, local, semi)))
    return inst, path


def _route_affine(case):
    match, mismatch = case.scoring[:2]
    pats = [p for p, _ in case.pairs]
    inst = {("alphabet_finish_kernel", ())}
    if sum(map(len, pats)):
        inst.add(("alphabet_kernel", ()))
    if any(p and t for p, t in case.pairs):
        alpha4 = int(len(set(b for p in pats for b in p)) <= 4 and -128 <= match <= 127 and -128 <= mismatch <= 127)
        trace = case.kind == "affine_align"
        inst.add(("affine32_score_kernel", (alpha4, int(trace), WIDE_R if trace else AFFINE_R_SCORE)))
        if trace:
            inst.add(("affine32_traceback_kernel", ()))
    return inst, None


def instances(case):
    return route(case)[0]


# ---- the cases ----
def rnd(rng, n, alpha=ACGT):
    return bytes(rng.choice(alpha) for _ in range(n))


def mutate(rng, s, alpha=ACGT, psub=0.08, pindel=0.03):
    out = bytearray()
    for ch in s:
        r = rng.random()
        if r < pindel:
            continue
        if r < 2 * pindel:
            out.append(rng.choice(alpha))
        out.append(rng.choice(alpha) if rng.random() < psub else ch)
    return bytes(out)


def related(rng, m, n, alpha=ACGT):
    """a text of length n and an m-byte pattern that shares stretches of it (the usual read-against-window shape)"""
    t = rnd(rng, n, alpha)
    p = (mutate(rng, t, alpha) + rnd(rng, m, alpha))[:m]
    return p, t


def tandem(rng, m, n):
    unit = rnd(rng, rng.randint(1, 4))
    t = (unit * (n // len(unit) + 2))[:n]
    p = (unit * (m // len(unit) + 4))[rng.randint(0, 3):][:m]
    return p, t


def with_rare(rng, p, rare=b"NRY"):
    """p with one or two bytes replaced by symbols outside ACGT (the 8-symbol fill's pair-pairs)"""
    b = bytearray(p)
    for _ in range(1 if len(b) < 8 else 2):
        b[rng.randrange(len(b))] = rng.choice(rare)
    return bytes(b)


SHORT16_SCORINGS = {2: (1, -1, -1), 4: (2, -3, -4), 8: (5, -4, -16)}
CHUNK_STEPS = {2: 24, 4: 12, 8: 6}


def short16_class_m():
    """both ends of every rows-per-lane class: 1, 32, 33, 64, ..., 225, 256, 257, 320, 321, 384, 385, 512"""
    out, lo = [], 1
    for R in R_CLASSES:
        out += [lo, 32 * R]
        lo = 32 * R + 1
    return out


def short16_cases():
    cases = []
    for K, s in SHORT16_SCORINGS.items():
        CS = CHUNK_STEPS[K]
        ns = (1, CS - 1, CS, CS + 1, 127, 128, 129)
        for mode in (GLOBAL, LOCAL, SEMI):
            rng = random.Random(1000 * K + mode)
            pairs = []

            def pair(m, n, variant):
                p, t = tandem(rng, m, n) if len(pairs) % 4 == 0 else related(rng, m, n)
                return (with_rare(rng, p) if variant else p, t)
            for variant in (0, 1):                                 # pair-pairs of one shape: 4-symbol, then 8-symbol
                for m in short16_class_m():
                    for n in ns:
                        pairs += [pair(m, n, variant), pair(m, n, variant)]
            for k, (m, n) in enumerate((m, n) for m in short16_class_m() for n in ns):
                pairs.append(pair(m, n, k % 2))                    # one leftover per shape: zipped with a neighbour of another shape
            for R in R_CLASSES:                                    # one more per class: an odd count leaves a singleton
                pairs.append(pair(32 * R - 5, 50, R % 2))
            pairs.append((rnd(rng, 150, b"ACGTNRYK"), rnd(rng, 300)))   # 8 distinct pattern bytes: wide32 serves its pair-pair
            pairs.append((rnd(rng, 150, b"ACGTNRYK"), rnd(rng, 300)))
            cases.append(Case(f"short16_K{K}_mode{mode}", "hw2", s, pairs, mode=mode))
    return cases


def boundary_cases():
    """The largest n the short16 plan accepts for every (R, K, global / semi-global), and n + 1: an all-match and an all-mismatch pair at
    both.  An off-by-one in the int16 bias shows here."""
    cases = []
    for K, s in SHORT16_SCORINGS.items():
        for mode in (GLOBAL, SEMI):
            pairs = []
            for R in R_CLASSES:
                m = 32 * R
                lo, hi = 1, 30001                                  # plan(lo) holds, plan(hi) does not (the record caps n at 30 000)
                assert plan(mode, m, lo, s) and not plan(mode, m, hi, s)
                while hi - lo > 1:
                    mid = (lo + hi) // 2
                    lo, hi = (mid, hi) if plan(mode, m, mid, s) else (lo, mid)
                for n in (lo, lo + 1):
                    pairs += [(b"A" * m, b"A" * n), (b"A" * m, b"C" * n)]
            cases.append(Case(f"plan_boundary_K{K}_mode{mode}", "hw2", s, pairs, mode=mode))
    return cases


def record_cases():
    """One pair-pair per batch for every (R, K, mode), over ACGT and with 'N' / 'R' in the patterns: the fill's record is compared with the
    host model's bit for bit."""
    cases = []
    for K, s in SHORT16_SCORINGS.items():
        n = 3 * CHUNK_STEPS[K] + 7
        for mode in (GLOBAL, LOCAL, SEMI):
            for R in R_CLASSES:
                m = 32 * R - 7 if R > 1 else 25
                for variant in (0, 1):
                    rng = random.Random(K * 100000 + mode * 10000 + R * 10 + variant)
                    pairs = [related(rng, m, n) for _ in range(2)]
                    if variant:
                        pairs = [(with_rare(rng, p, b"NR"), t) for p, t in pairs]
                    cases.append(Case(f"record_K{K}_mode{mode}_R{R}_a{4 + 4 * variant}", "hw2", s, pairs, mode=mode, record=True))
    return cases


WIDE_M = (1, 127, 128, 129, 255, 256, 257, 513)
WIDE_N = (1, 2, 3, 4, 5, 31, 32, 33, 64, 65)
WIDE_SCORINGS = {2: (1, -1, -1), 4: (2, -3, -4), 8: (5, -4, -16), 16: (100, -100, -200), 32: (1, -1, 1), 33: (-1, -2, -1)}


def wide_cases():
    """wide32 at the edges of its tile (n < 4), its 32-column blocks and its 128-row bands: every K, mode, ALPHA4 on / off, record and
    score-only, and hw4's tie order.  K = 2 / 4 / 8 reach wide32 through m > 512 or n beyond the plan (ALPHA4 on), or through patterns
    with more than 7 distinct bytes (ALPHA4 off)."""
    cases = []
    for tag, s in WIDE_SCORINGS.items():
        for alpha4 in (1, 0):
            alpha = ACGT if alpha4 else PROT
            rng = random.Random(tag * 10 + alpha4)
            pairs = [related(rng, m, n, alpha) for m in WIDE_M for n in WIDE_N]
            if tag in (2, 4, 8):                                   # n beyond the short16 plan
                n_out = {2: 30001, 4: 8200, 8: 2100}[tag]
                pairs += [related(rng, 128, n_out, alpha), related(rng, 40, n_out, alpha)]
            variants = [(mode, False, False) for mode in (GLOBAL, LOCAL, SEMI)] + \
                       [(mode, True, False) for mode in (GLOBAL, LOCAL, SEMI)] + [(GLOBAL, False, True)]
            for mode, so, hw4 in variants:
                cases.append(Case(f"wide_K{tag}_a{alpha4}_mode{mode}{'_score_only' if so else ''}{'_hw4' if hw4 else ''}", "hw2", s,
                                  pairs, mode=mode, want_ops=not so, score_only=so, tie_hw4=hw4))
    return cases


def ckpt_cases():
    """Every wide32 pair on the checkpointed path (B2A_OPT_CKPT_BYTES = 0), one band per re-filled group, tiles of 32 or 128 columns:
    all five K, both modes, ALPHA4 on and off."""
    cases = []
    for tag, s in WIDE_SCORINGS.items():
        for mode in (GLOBAL, LOCAL):
            for alpha4 in (1, 0):
                alpha = ACGT if alpha4 else PROT
                for cols, group in ((5, 1), (7, 600_000)):
                    rng = random.Random(tag * 1000 + mode * 100 + alpha4 * 10 + cols)
                    shapes = ((513, 300), (600, 700), (300, 64), (129, 257), (700, 40))
                    pairs = [related(rng, m, n, alpha) for m, n in shapes]
                    if tag in (2, 4, 8) and alpha4:                 # m > 512 only: shorter ACGT pairs stay on short16
                        pairs = [(p + rnd(rng, 513 - len(p)) if len(p) < 513 else p, t) for p, t in pairs]
                    pairs.append(tandem(rng, 640, 520))
                    cases.append(Case(f"ckpt_K{tag}_mode{mode}_a{alpha4}_cols{cols}", "hw2", s, pairs, mode=mode,
                                      options={OPT_CKPT_BYTES: 0, OPT_CKPT_GROUP: group, OPT_CKPT_COLS: cols}))
    return cases


def affine_cases():
    cases = []
    for alpha4, alpha in ((1, ACGT), (0, PROT)):
        rng = random.Random(77 + alpha4)
        ns = (1, 2, 3, 4, 5, 31, 32, 33)
        pairs = [related(rng, m, n, alpha) for m in (255, 256, 257, 511, 512, 513) for n in ns]
        cases.append(Case(f"affine_score_a{alpha4}", "affine_score", (5, -4, -16, -4), pairs))
        pairs = [related(rng, m, n, alpha) for m in (127, 128, 129) for n in ns + (200,)]
        cases.append(Case(f"affine_align_a{alpha4}", "affine_align", (5, -4, -16, -4), pairs))
    return cases


def seq2_cases():
    rng = random.Random(5)
    pairs = [related(rng, 150, 400) for _ in range(64)]
    pairs = [(with_rare(rng, p, b"N") if k % 5 == 0 else p, t) for k, (p, t) in enumerate(pairs)]
    return [Case("seq2_global", "hw2", (1, -1, -1), pairs, mode=GLOBAL, seq2=True)]


@lru_cache(maxsize=None)
def all_cases():
    cases = short16_cases() + boundary_cases() + record_cases() + wide_cases() + ckpt_cases() + affine_cases() + seq2_cases()
    assert all(len(c.pairs) < SEG_PAIRS for c in cases)
    assert len({c.name for c in cases}) == len(cases)
    return cases
