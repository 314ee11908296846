"""bioinformatics-algorithms_b200 -- B200-native pairwise alignment engine (Python harness side).

Thin ctypes binding over the C ABI in include/b2align.h (libb2align.so, built in-tree by
`make -C bioinformatics-algorithms_b200`).  The product is the shared library + the `hw2`
drop-in binary; this module exists for tests, bench.py and scripting.  It mirrors the
reference's function seam (hw2.cpp:118, :192) with one-pair shims and exposes the batch call
that replaces the loop hw2.cpp:328-338.

There is no CPU fallback: importing works without a GPU (so symbols can be inspected), but
creating an Engine raises if the library or a CUDA device is missing.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2A_LIB") or os.path.join(HERE, "libb2align.so")      # B2A_LIB: experiment builds (scripts/)
HW2_BIN = os.path.join(HERE, "bin", "hw2")
HW3_BIN = os.path.join(HERE, "bin", "hw3")
HW4_BIN = os.path.join(HERE, "bin", "hw4")

GLOBAL, LOCAL = 0, 1
SEMIGLOBAL = 2          # the whole pattern against its best-fitting substring of the text (include/b2align.h)
SCORE_ONLY = 2
TIE_HW4 = 4
OPT_LANES, OPT_SEG_PAIRS, OPT_SEG_BYTES, OPT_SEG_FIRST, OPT_CKPT_BYTES, OPT_CKPT_GROUP, OPT_CKPT_COLS = 1, 2, 3, 5, 6, 7, 8
WANT_OPS = 1

RESULT_DTYPE = np.dtype([("score", "<i4"), ("end_i", "<u4"), ("end_j", "<u4"), ("start_i", "<u4"),
                         ("start_j", "<u4"), ("overlap", "<i4"), ("n_ops", "<u4"), ("path", "<u4")])

EXPORTS = ["b2a_device_count", "b2a_create", "b2a_destroy", "b2a_last_error", "b2a_host_alloc", "b2a_host_free",
           "b2a_host_register", "b2a_host_unregister", "b2a_align_batch", "b2a_align_batch_multi", "b2a_select_run",
           "b2a_seq2_pack", "b2a_seq2_unpack", "b2a_align_batch_multi_seq2", "b2a_find_anchors", "b2a_align_anchored", "b2a_set_ops_sink", "b2a_affine_score_batch", "b2a_affine_align_batch", "b2a_affine_fetch_ops", "b2a_affine_star_scores", "b2a_fetch_ops", "b2a_copy_ops", "b2a_batch_upload", "b2a_batch_run",
           "b2a_batch_download", "b2a_batch_times", "b2a_set_option", "b2a_batch_stats", "b2a_render_cigar", "b2a_render_mdz", "b2a_select_best",
           "b2a_upgma_newick", "b2a_center_star_phylip",
           "b2a_microbench_int16x2", "b2a_debug_copy_record"]


class Params(C.Structure):
    _fields_ = [("mode", C.c_int32), ("match", C.c_int32), ("mismatch", C.c_int32), ("gap", C.c_int32),
                ("flags", C.c_uint32)]


class Seq2(C.Structure):
    """b2a_seq2 (include/b2align.h): a concatenated byte buffer as 2-bit codes + an exception list."""
    _fields_ = [("codes", C.c_void_p), ("n_bytes", C.c_uint64), ("alphabet", C.c_uint8 * 4), ("reserved", C.c_uint32),
                ("exc_pos", C.c_void_p), ("exc_byte", C.c_void_p), ("n_exc", C.c_uint64)]


class B2AError(RuntimeError):
    pass


_lib = None


def load_library():
    """dlopen libb2align.so (raises loudly if the CUDA extension was not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B2AError(f"{LIB_PATH} is missing: build it with `make -C {HERE}` (no CPU fallback exists)")
        lib = C.CDLL(LIB_PATH)
        lib.b2a_create.restype = C.c_void_p
        lib.b2a_create.argtypes = [C.c_int]
        lib.b2a_destroy.argtypes = [C.c_void_p]
        lib.b2a_last_error.restype = C.c_char_p
        lib.b2a_last_error.argtypes = [C.c_void_p]
        lib.b2a_host_alloc.restype = C.c_void_p
        lib.b2a_host_alloc.argtypes = [C.c_size_t]
        lib.b2a_host_free.argtypes = [C.c_void_p]
        P = C.c_void_p
        lib.b2a_align_batch.argtypes = [P, C.POINTER(Params), P, P, P, P, C.c_uint64, P]
        lib.b2a_align_batch_multi.argtypes = [P, C.POINTER(Params), C.c_uint32, P, P, P, P, C.c_uint64, P]
        lib.b2a_select_run.argtypes = [P, C.c_uint32]
        lib.b2a_seq2_pack.restype = C.c_int64
        lib.b2a_seq2_pack.argtypes = [P, C.c_uint64, P, P, P, P, C.c_uint64]
        lib.b2a_seq2_unpack.argtypes = [C.POINTER(Seq2), C.c_uint64, C.c_uint64, P]
        lib.b2a_set_ops_sink.argtypes = [P, P, C.c_uint32, C.c_uint64]
        lib.b2a_find_anchors.restype = C.c_int64
        lib.b2a_find_anchors.argtypes = [P, C.c_uint64, P, C.c_uint64, C.c_uint32, C.c_uint32, P, C.c_uint64]
        lib.b2a_align_anchored.restype = C.c_int64
        lib.b2a_align_anchored.argtypes = [P, C.POINTER(Params), P, C.c_uint64, P, C.c_uint64, P, C.c_uint64, P, P, C.c_uint64]
        lib.b2a_align_batch_multi_seq2.argtypes = [P, C.POINTER(Params), C.c_uint32, C.POINTER(Seq2), P, C.POINTER(Seq2), P, C.c_uint64, P]
        lib.b2a_host_register.argtypes = [P, C.c_size_t]
        lib.b2a_host_unregister.argtypes = [P]
        lib.b2a_batch_upload.argtypes = [P, C.POINTER(Params), P, P, P, P, C.c_uint64]
        lib.b2a_batch_run.argtypes = [P, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        lib.b2a_batch_download.argtypes = [P, P]
        lib.b2a_batch_times.argtypes = [P] + [C.POINTER(C.c_float)] * 3
        lib.b2a_set_option.argtypes = [P, C.c_int, C.c_int64]
        lib.b2a_batch_stats.argtypes = [P] + [C.POINTER(C.c_uint64)] * 5
        lib.b2a_fetch_ops.restype = C.c_int64
        lib.b2a_fetch_ops.argtypes = [P, C.c_uint64, P, C.c_uint64]
        lib.b2a_copy_ops.restype = C.c_int64
        lib.b2a_copy_ops.argtypes = [P, P, C.c_uint64, P]
        lib.b2a_render_cigar.restype = C.c_int64
        lib.b2a_render_cigar.argtypes = [C.c_char_p, C.c_uint64, P, C.c_uint64]
        lib.b2a_render_mdz.restype = C.c_int64
        lib.b2a_render_mdz.argtypes = [C.c_char_p, C.c_uint64, C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32, P, C.c_uint64]
        lib.b2a_select_best.restype = C.c_int64
        lib.b2a_select_best.argtypes = [C.c_int32, P, C.c_uint64]
        lib.b2a_center_star_phylip.restype = C.c_int64
        lib.b2a_center_star_phylip.argtypes = [C.c_uint32, C.c_uint32, P, P, P, P, P, P, C.c_uint64]
        lib.b2a_upgma_newick.restype = C.c_int64
        lib.b2a_upgma_newick.argtypes = [P, C.c_uint32, P, P, C.c_uint64]
        lib.b2a_microbench_int16x2.argtypes = [P, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]
        lib.b2a_affine_score_batch.argtypes = [P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, P, P, P, P, C.c_uint64, P]
        lib.b2a_affine_align_batch.argtypes = [P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, P, P, P, P, C.c_uint64, P, P]
        lib.b2a_affine_fetch_ops.restype = C.c_int64
        lib.b2a_affine_fetch_ops.argtypes = [P, C.c_uint64, P, C.c_uint64]
        lib.b2a_affine_star_scores.argtypes = [P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, P, P, C.c_uint32,
                                               C.c_uint32, C.c_uint32, P, P, P]
        _lib = lib
    return _lib


def pack(seqs):
    """list of bytes -> (uint8 bytes, uint64 offsets[n+1]) in the layout b2a_align_batch takes."""
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    if len(seqs):
        np.cumsum([len(s) for s in seqs], out=off[1:])
    data = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy() if len(seqs) else np.zeros(0, np.uint8)
    return data, off


class PackedSeq:
    """Owner of the arrays a b2a_seq2 points to (b2a_seq2_pack); .c is the struct the C ABI takes."""

    def __init__(self, data, alphabet=b"ACGT", pinned=False):
        lib = load_library()
        data = np.ascontiguousarray(data, dtype=np.uint8)
        assert len(alphabet) == 4
        alpha = (C.c_uint8 * 4)(*alphabet)
        n = data.size
        alloc = pinned_empty if pinned else (lambda k, dt: np.empty(max(k, 1), dtype=dt))
        self.codes = alloc((n + 3) // 4, np.uint8)
        cap = n // 128 + 4096                                  # usually enough: one pass.  Otherwise the call says how many there are
        while True:
            self.exc_pos = alloc(cap, np.uint64)
            self.exc_byte = alloc(cap, np.uint8)
            n_exc = lib.b2a_seq2_pack(data.ctypes.data, n, alpha, self.codes.ctypes.data, self.exc_pos.ctypes.data,
                                      self.exc_byte.ctypes.data, cap)
            if n_exc < 0:
                raise B2AError("b2a_seq2_pack failed")
            if n_exc <= cap:
                break
            cap = int(n_exc)
        self.n_bytes, self.n_exc = n, int(n_exc)
        self.c = Seq2(self.codes.ctypes.data, n, alpha, 0, self.exc_pos.ctypes.data, self.exc_byte.ctypes.data, n_exc)

    @property
    def nbytes(self):
        """bytes that cross PCIe for the whole buffer"""
        return (self.n_bytes + 3) // 4 + 9 * self.n_exc

    def unpack(self, first=0, count=None):
        count = self.n_bytes - first if count is None else count
        out = np.empty(max(count, 1), dtype=np.uint8)
        if load_library().b2a_seq2_unpack(C.byref(self.c), first, count, out.ctypes.data) != 0:
            raise B2AError("b2a_seq2_unpack failed")
        return out[:count]


ANCHOR_DTYPE = np.dtype([("i", "<u4"), ("j", "<u4"), ("len", "<u4")])


def find_anchors(pattern, text, k=16, spacing=256):
    """b2a_find_anchors: chain of unique exact k-mer matches, ascending in both sequences (numpy record array i, j, len)."""
    lib = load_library()
    p = np.frombuffer(pattern, dtype=np.uint8) if isinstance(pattern, (bytes, bytearray)) else np.ascontiguousarray(pattern, dtype=np.uint8)
    t = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else np.ascontiguousarray(text, dtype=np.uint8)
    cap = max(1, p.size // max(spacing, k, 1) + 2)
    out = np.zeros(cap, dtype=ANCHOR_DTYPE)
    got = lib.b2a_find_anchors(p.ctypes.data, p.size, t.ctypes.data, t.size, k, spacing, out.ctypes.data, cap)
    if got < 0 or got > cap:
        raise B2AError(f"b2a_find_anchors failed ({got})")
    return out[:got]


def pinned_empty(n, dtype):
    """numpy array over cudaHostAlloc'ed memory (freed when the array's base object dies)."""
    lib = load_library()
    dt = np.dtype(dtype)
    nbytes = max(int(n) * dt.itemsize, 1)
    ptr = lib.b2a_host_alloc(nbytes)
    if not ptr:
        raise B2AError("b2a_host_alloc failed")

    class _Owner:
        def __init__(self, p):
            self.p = p

        def __del__(self):
            try:
                lib.b2a_host_free(self.p)
            except Exception:
                pass
    buf = (C.c_uint8 * nbytes).from_address(ptr)
    buf._owner = _Owner(ptr)
    return np.frombuffer(buf, dtype=dt, count=int(n))


def host_register(arr):
    """Pin an existing numpy buffer (e.g. over POSIX shared memory) for asynchronous device copies."""
    if load_library().b2a_host_register(arr.ctypes.data, arr.nbytes) != 0:
        raise B2AError("b2a_host_register failed")


def host_unregister(arr):
    load_library().b2a_host_unregister(arr.ctypes.data)


def unpack_ops(words, off, k, n_ops):
    """2-bit device ops of pair k -> b'MDI...' in traceback order."""
    w = words[int(off[k]): int(off[k]) + (int(n_ops) + 15) // 16]
    if n_ops == 0:
        return b""
    codes = (np.repeat(w, 16) >> np.tile(np.arange(0, 32, 2, dtype=np.uint32), len(w))) & 3
    return np.frombuffer(b"MDI?", dtype=np.uint8)[codes[:int(n_ops)]].tobytes()


def render_cigar(ops: bytes) -> str:
    lib = load_library()
    cap = 24 * (len(ops) + 2)
    buf = C.create_string_buffer(cap)
    n = lib.b2a_render_cigar(ops, len(ops), buf, cap)
    if n < 0:
        raise B2AError("b2a_render_cigar failed")
    return buf.raw[:n].decode("latin-1")


def render_mdz(ops: bytes, pattern: bytes, text: bytes, start_i: int, start_j: int) -> str:
    lib = load_library()
    cap = 24 * (len(ops) + 2)
    buf = C.create_string_buffer(cap)
    n = lib.b2a_render_mdz(ops, len(ops), pattern, text, start_i, start_j, buf, cap)
    if n < 0:
        raise B2AError("b2a_render_mdz failed")
    return buf.raw[:n].decode("latin-1")


def aligned_strings(ops: bytes, pattern: bytes, text: bytes, start_i: int, start_j: int):
    """alignedPattern / alignedReference of struct AlignmentResult (hw2.cpp:17-23) from the op list."""
    ap, ar = bytearray(), bytearray()
    i, j = start_i, start_j
    for op in reversed(ops):
        if op == 0x4D:      # M
            ap.append(pattern[i]); ar.append(text[j]); i += 1; j += 1
        elif op == 0x44:    # D
            ap.append(pattern[i]); ar.append(0x2D); i += 1
        else:               # I
            ap.append(0x2D); ar.append(text[j]); j += 1
    return bytes(ap), bytes(ar)


class AlignmentResult:
    """Mirror of the reference's struct AlignmentResult (hw2.cpp:17-23)."""
    __slots__ = ("score", "alignedPattern", "alignedReference", "cigar", "mdz", "record", "ops")


class Engine:
    """One context on one GPU (b2a_create / b2a_destroy)."""

    def __init__(self, device=0):
        self.lib = load_library()
        self.ctx = self.lib.b2a_create(int(device))
        if not self.ctx:
            raise B2AError(f"b2a_create({device}) failed: no usable sm_100 CUDA device (there is no CPU fallback)")

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.b2a_destroy(self.ctx)
            self.ctx = None

    __del__ = close

    def _check(self, rc, what):
        if rc < 0:
            raise B2AError(f"{what} failed (rc={rc}): {self.lib.b2a_last_error(self.ctx).decode()}")
        return rc

    # -- the batch call that replaces hw2.cpp:328-338 --
    def align_packed(self, mode, pat, pat_off, txt, txt_off, match, mismatch, gap, want_ops=False, results=None,
                     score_only=False, tie_hw4=False):
        n = len(pat_off) - 1
        if results is None:
            results = np.empty(n, dtype=RESULT_DTYPE)
        prm = Params(mode, match, mismatch, gap, (WANT_OPS if want_ops else 0) | (SCORE_ONLY if score_only else 0) | (TIE_HW4 if tie_hw4 else 0))
        self._check(self.lib.b2a_align_batch(self.ctx, C.byref(prm), pat.ctypes.data, pat_off.ctypes.data,
                                             txt.ctypes.data, txt_off.ctypes.data, n, results.ctypes.data), "b2a_align_batch")
        return results

    def align_packed_multi(self, modes, pat, pat_off, txt, txt_off, match, mismatch, gap, want_ops=False, results=None):
        """Several runs (modes) over ONE upload of the pairs (b2a_align_batch_multi): returns one result array per mode."""
        n = len(pat_off) - 1
        if results is None:
            results = [np.empty(n, dtype=RESULT_DTYPE) for _ in modes]
        prms = (Params * len(modes))(*[Params(m, match, mismatch, gap, WANT_OPS if want_ops else 0) for m in modes])
        ptrs = (C.c_void_p * len(modes))(*[r.ctypes.data for r in results])
        self._check(self.lib.b2a_align_batch_multi(self.ctx, prms, len(modes), pat.ctypes.data, pat_off.ctypes.data,
                                                   txt.ctypes.data, txt_off.ctypes.data, n, ptrs), "b2a_align_batch_multi")
        return results

    def align_seq2_multi(self, modes, pat2, pat_off, txt2, txt_off, match, mismatch, gap, want_ops=False, results=None):
        """align_packed_multi over compact inputs (PackedSeq, b2a_align_batch_multi_seq2): a quarter of the upload, the same results."""
        n = len(pat_off) - 1
        if results is None:
            results = [np.empty(n, dtype=RESULT_DTYPE) for _ in modes]
        prms = (Params * len(modes))(*[Params(m, match, mismatch, gap, WANT_OPS if want_ops else 0) for m in modes])
        ptrs = (C.c_void_p * len(modes))(*[r.ctypes.data for r in results])
        self._check(self.lib.b2a_align_batch_multi_seq2(self.ctx, prms, len(modes), C.byref(pat2.c), pat_off.ctypes.data,
                                                        C.byref(txt2.c), txt_off.ctypes.data, n, ptrs), "b2a_align_batch_multi_seq2")
        return results

    def align_anchored(self, pattern, text, anchors, match, mismatch, gap, tie_hw4=False):
        """b2a_align_anchored: global alignment through the given exact-match anchors -> (result record, ops bytes in traceback order)."""
        p = np.frombuffer(pattern, dtype=np.uint8) if isinstance(pattern, (bytes, bytearray)) else np.ascontiguousarray(pattern, dtype=np.uint8)
        t = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else np.ascontiguousarray(text, dtype=np.uint8)
        a = np.ascontiguousarray(anchors, dtype=ANCHOR_DTYPE)
        prm = Params(GLOBAL, match, mismatch, gap, TIE_HW4 if tie_hw4 else 0)
        res = np.zeros(1, dtype=RESULT_DTYPE)
        cap = p.size + t.size + 1
        buf = C.create_string_buffer(cap)
        n = self._check(self.lib.b2a_align_anchored(self.ctx, C.byref(prm), p.ctypes.data, p.size, t.ctypes.data, t.size,
                                                    a.ctypes.data, len(a), res.ctypes.data, buf, cap), "b2a_align_anchored")
        return res[0], buf.raw[:n]

    def set_ops_sink(self, buffers):
        """b2a_set_ops_sink: uint32 arrays (one per run, pinned for asynchronous copies) that receive the op words of the next batch calls
        segment by segment; None switches it off.  The arrays must stay alive while the sink is set."""
        if not buffers:
            self._sink = None
            return self._check(self.lib.b2a_set_ops_sink(self.ctx, None, 0, 0), "b2a_set_ops_sink")
        self._sink = list(buffers)
        ptrs = (C.c_void_p * len(buffers))(*[b.ctypes.data for b in buffers])
        self._check(self.lib.b2a_set_ops_sink(self.ctx, ptrs, len(buffers), min(b.size for b in buffers)), "b2a_set_ops_sink")

    def ops_offsets(self, n_pairs):
        """per-pair word offsets of the last batch's op lists (n_pairs + 1 entries) and the total word count"""
        off = np.empty(n_pairs + 1, dtype=np.uint64)
        total = self._check(self.lib.b2a_copy_ops(self.ctx, None, 0, off.ctypes.data), "b2a_copy_ops")
        return off, total

    def select_run(self, run):
        self._check(self.lib.b2a_select_run(self.ctx, int(run)), "b2a_select_run")

    def align_batch(self, mode, patterns, texts, match, mismatch, gap, want_ops=True, tie_hw4=False):
        """lists of bytes -> (results recarray, list of op byte-strings in traceback order or None)."""
        assert len(patterns) == len(texts)
        pat, po = pack(patterns)
        txt, to = pack(texts)
        res = self.align_packed(mode, pat, po, txt, to, match, mismatch, gap, want_ops, tie_hw4=tie_hw4)
        ops = None
        if want_ops:
            words, off = self.copy_ops(len(patterns))
            ops = [unpack_ops(words, off, k, res["n_ops"][k]) for k in range(len(patterns))]
        return res, ops

    def copy_ops(self, n_pairs):
        total = self._check(self.lib.b2a_copy_ops(self.ctx, None, 0, None), "b2a_copy_ops")
        words = np.empty(max(total, 1), dtype=np.uint32)
        off = np.empty(n_pairs + 1, dtype=np.uint64)
        self._check(self.lib.b2a_copy_ops(self.ctx, words.ctypes.data, total, off.ctypes.data), "b2a_copy_ops")
        return words, off

    def fetch_ops(self, pair, n_ops):
        buf = C.create_string_buffer(int(n_ops) + 1)
        n = self._check(self.lib.b2a_fetch_ops(self.ctx, pair, buf, int(n_ops)), "b2a_fetch_ops")
        return buf.raw[:n]

    # -- device-resident variant, for kernel-only timing --
    def upload(self, mode, pat, pat_off, txt, txt_off, match, mismatch, gap, want_ops=False, score_only=False):
        prm = Params(mode, match, mismatch, gap, (WANT_OPS if want_ops else 0) | (SCORE_ONLY if score_only else 0))
        self._check(self.lib.b2a_batch_upload(self.ctx, C.byref(prm), pat.ctypes.data, pat_off.ctypes.data,
                                              txt.ctypes.data, txt_off.ctypes.data, len(pat_off) - 1), "b2a_batch_upload")

    def run(self):
        f, t = C.c_float(), C.c_float()
        self._check(self.lib.b2a_batch_run(self.ctx, C.byref(f), C.byref(t)), "b2a_batch_run")
        return f.value, t.value

    def times(self):
        """(fill_ms, traceback_ms, total_ms) of the last run()"""
        v = [C.c_float() for _ in range(3)]
        self.lib.b2a_batch_times(self.ctx, *[C.byref(x) for x in v])
        return tuple(x.value for x in v)

    def set_option(self, option, value):
        self._check(self.lib.b2a_set_option(self.ctx, int(option), int(value)), "b2a_set_option")

    def download(self, n_pairs, results=None):
        if results is None:
            results = np.empty(n_pairs, dtype=RESULT_DTYPE)
        self._check(self.lib.b2a_batch_download(self.ctx, results.ctypes.data), "b2a_batch_download")
        return results

    # -- hw3's distance stage (hw3.cpp:23-98, :231-251): score-only affine global alignment --
    def affine_scores(self, patterns, texts, match, mismatch, gap_open, gap_extend):
        """lists of bytes -> int32 scores, pair k = affine_alignment(patterns[k], texts[k], ..., &score)"""
        assert len(patterns) == len(texts)
        pat, po = pack(patterns)
        txt, to = pack(texts)
        out = np.zeros(len(patterns), dtype=np.int32)
        self._check(self.lib.b2a_affine_score_batch(self.ctx, match, mismatch, gap_open, gap_extend, pat.ctypes.data,
                                                    po.ctypes.data, txt.ctypes.data, to.ctypes.data, len(patterns),
                                                    out.ctypes.data), "b2a_affine_score_batch")
        return out

    def affine_align(self, patterns, texts, match, mismatch, gap_open, gap_extend):
        """hw3's affine_alignment WITH traceback (hw3.cpp:23-135): (int32 scores, list of op byte-strings in traceback order)"""
        assert len(patterns) == len(texts)
        pat, po = pack(patterns)
        txt, to = pack(texts)
        n = len(patterns)
        sc = np.zeros(max(n, 1), dtype=np.int32)
        nops = np.zeros(max(n, 1), dtype=np.uint32)
        self._check(self.lib.b2a_affine_align_batch(self.ctx, match, mismatch, gap_open, gap_extend, pat.ctypes.data, po.ctypes.data,
                                                    txt.ctypes.data, to.ctypes.data, n, sc.ctypes.data, nops.ctypes.data),
                    "b2a_affine_align_batch")
        ops = []
        for k in range(n):
            buf = C.create_string_buffer(int(nops[k]) + 1)
            got = self._check(self.lib.b2a_affine_fetch_ops(self.ctx, k, buf, int(nops[k])), "b2a_affine_fetch_ops")
            ops.append(buf.raw[:got])
        return sc[:n], ops

    def affine_star_scores(self, seqs, match, mismatch, gap_open, gap_extend, pair_first=0, pair_count=None):
        """All-vs-all (i < j) scores of one sequence set, the star sums and the centre index (hw3.cpp:231-251)."""
        data, off = pack(seqs)
        n = len(seqs)
        total = n * (n - 1) // 2
        if pair_count is None:
            pair_count = total - pair_first
        ps = np.zeros(max(pair_count, 1), dtype=np.int32)
        sums = np.zeros(max(n, 1), dtype=np.int32)
        center = C.c_int64(-1)
        self._check(self.lib.b2a_affine_star_scores(self.ctx, match, mismatch, gap_open, gap_extend, data.ctypes.data,
                                                    off.ctypes.data, n, pair_first, pair_count, ps.ctypes.data,
                                                    sums.ctypes.data, C.byref(center)), "b2a_affine_star_scores")
        return ps[:pair_count], sums[:n], center.value

    def stats(self):
        v = [C.c_uint64() for _ in range(5)]
        self.lib.b2a_batch_stats(self.ctx, *[C.byref(x) for x in v])
        return dict(zip(("launches", "cells", "fill_bytes", "h2d_bytes", "d2h_bytes"), (x.value for x in v)))

    def microbench(self, kind=0):
        g, mhz = C.c_double(), C.c_float()
        self._check(self.lib.b2a_microbench_int16x2(self.ctx, kind, C.byref(g), C.byref(mhz)), "b2a_microbench_int16x2")
        return g.value, mhz.value

    # -- one-pair shims with the reference's own names and argument order (hw2.cpp:118, :192) --
    def _one(self, mode, pattern, reference, matchScore, mismatchScore, gapPenalty):
        res, ops = self.align_batch(mode, [pattern], [reference], matchScore, mismatchScore, gapPenalty, True)
        r = AlignmentResult()
        r.record, r.ops, r.score = res[0], ops[0], int(res["score"][0])
        si, sj = int(res["start_i"][0]), int(res["start_j"][0])
        r.alignedPattern, r.alignedReference = aligned_strings(ops[0], pattern, reference, si, sj)
        r.cigar = render_cigar(ops[0])
        r.mdz = render_mdz(ops[0], pattern, reference, si, sj)
        return r

    def globalAlignmentNeedlemanWunsch(self, patterns, references, matchScore, mismatchScore, gapPenalty):
        return self._one(GLOBAL, patterns, references, matchScore, mismatchScore, gapPenalty)

    def localAlignmentSmithWaterman(self, patterns, references, matchScore, mismatchScore, gapPenalty):
        return self._one(LOCAL, patterns, references, matchScore, mismatchScore, gapPenalty)

    def semiGlobalAlignment(self, pattern, reference, matchScore, mismatchScore, gapPenalty):
        """Semi-global mode (not in the reference): the whole pattern against the substring of the reference that suits it best;
        record.end_j / record.start_j give where it sits (alignedReference covers reference[start_j:end_j])."""
        return self._one(SEMIGLOBAL, pattern, reference, matchScore, mismatchScore, gapPenalty)


def center_star_phylip(names, seqs, centre, ops):
    """hw3's output file (hw3.cpp:253-357) from the op lists of affine_alignment(seqs[centre], seqs[i]); ops[centre] is ignored."""
    lib = load_library()
    n = len(seqs)
    enc = [x if isinstance(x, bytes) else x.encode() for x in names]
    ops = [o if o is not None else b"" for o in ops]
    name_arr = (C.c_char_p * n)(*enc)
    seq_arr = (C.c_char_p * n)(*seqs)
    ops_arr = (C.c_char_p * n)(*ops)
    slen = np.array([len(s) for s in seqs], dtype=np.uint64)
    olen = np.array([len(o) for o in ops], dtype=np.uint64)
    cap = 64 + n * (sum(len(s) for s in seqs) * 12 // 10 + 64)
    buf = C.create_string_buffer(cap)
    k = lib.b2a_center_star_phylip(n, centre, name_arr, seq_arr, slen.ctypes.data, ops_arr, olen.ctypes.data, buf, cap)
    if k < 0:
        raise B2AError("b2a_center_star_phylip failed")
    return buf.raw[:k].decode("latin-1")


def upgma_newick(pair_dist, names):
    """hw4's tree line (without the newline) from the i < j row-major pair distances (hw4.cpp:154-228)."""
    lib = load_library()
    d = np.ascontiguousarray(pair_dist, dtype=np.int32)
    n = len(names)
    arr = (C.c_char_p * max(n, 1))(*[x if isinstance(x, bytes) else x.encode() for x in names])
    cap = 64 + sum(len(x) + 64 for x in names)
    buf = C.create_string_buffer(cap)
    k = lib.b2a_upgma_newick(d.ctypes.data, n, arr, buf, cap)
    if k < 0:
        raise B2AError("b2a_upgma_newick failed")
    return buf.raw[:k].decode("latin-1")


def select_best(mode, results):
    lib = load_library()
    res = np.ascontiguousarray(results)
    return int(lib.b2a_select_best(mode, res.ctypes.data, len(res)))
