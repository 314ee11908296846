"""ctypes binding to tests/semiglobal_oracle.c -- the CPU statement of the semi-global mode.

TEST INFRASTRUCTURE ONLY.  The library is compiled with the system C compiler on first use into a
temporary directory (keyed by the source's hash), so a read-only checkout works too.  CIGAR and MD:Z
come from the pinned hw2 oracle (tests/oracle_binding.py).
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import oracle_binding as ob

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "semiglobal_oracle.c")
SEMIGLOBAL = 2

_lib = None


def lib():
    global _lib
    if _lib is None:
        with open(SRC, "rb") as f:
            tag = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"b2a_semiglobal_oracle_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            tmp = so + f".{os.getpid()}.tmp"
            subprocess.check_call(["cc", "-O2", "-shared", "-fPIC", "-o", tmp, SRC])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.orc_semiglobal.restype = C.c_int
        _lib.orc_semiglobal_score.restype = C.c_int
    return _lib


def align(pattern: bytes, text: bytes, match: int, mismatch: int, gap: int) -> ob.Alignment:
    """One pair, semi-global: score, end/start cell, overlap, ops (traceback order), CIGAR, MD:Z."""
    L, O = lib(), ob.lib()
    m, n = len(pattern), len(text)
    res = ob.OrcResult()
    ops = C.create_string_buffer(m + n + 1)
    rc = L.orc_semiglobal(pattern, C.c_uint32(m), text, C.c_uint32(n), C.c_int(match), C.c_int(mismatch), C.c_int(gap),
                          C.byref(res), ops)
    if rc != 0:
        raise RuntimeError(f"orc_semiglobal rc={rc}")
    a = ob.Alignment()
    a.score, a.end_i, a.end_j = res.score, res.end_i, res.end_j
    a.start_i, a.start_j, a.overlap = res.start_i, res.start_j, res.overlap
    a.ops = ops.raw[:res.n_ops]
    cap = 16 * (m + n) + 64
    buf = C.create_string_buffer(cap)
    w = O.orc_cigar(a.ops, C.c_uint32(res.n_ops), buf, C.c_size_t(cap))
    a.cigar = buf.raw[:w].decode("latin-1")
    w = O.orc_mdz(a.ops, C.c_uint32(res.n_ops), pattern, text, C.c_uint32(res.start_i), C.c_uint32(res.start_j),
                  buf, C.c_size_t(cap))
    a.mdz = buf.raw[:w].decode("latin-1")
    return a


def score_only(pattern: bytes, text: bytes, match, mismatch, gap):
    """(score, end_i, end_j) in linear memory."""
    res = ob.OrcResult()
    rc = lib().orc_semiglobal_score(pattern, C.c_uint32(len(pattern)), text, C.c_uint32(len(text)),
                                    C.c_int(match), C.c_int(mismatch), C.c_int(gap), C.byref(res))
    if rc != 0:
        raise RuntimeError(f"orc_semiglobal_score rc={rc}")
    return res.score, res.end_i, res.end_j
