"""CPU reference of lattice-char-index-utterance (tests/char_utterance_ref.cc) through ctypes.

Test infrastructure, like oracle/ora.py, whose lattice and option structures it shares: the
reference is compiled once per process into a temporary directory, so the tests write nothing
into the tree.
"""
import ctypes as C
import os
import subprocess
import tempfile
import threading

from oracle import ora

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_LOCK = threading.Lock()
CHAR_UTTERANCE, BRUTE_CHAR_UTTERANCE = 0, 1


def lib():
    global _LIB
    with _LOCK:
        if _LIB is None:
            out = os.path.join(tempfile.mkdtemp(prefix="klu_charutt_"), "libklu_charutt_ref.so")
            cxx = os.environ.get("CXX", "g++")
            subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-o", out,
                            os.path.join(_HERE, "char_utterance_ref.cc")], check=True)
            L = C.CDLL(out)
            L.charutt_run.restype = C.c_void_p
            L.charutt_run.argtypes = [C.c_int, C.POINTER(ora.OraLat), C.POINTER(ora.OraOpts)]
            L.ora_error.restype = C.c_char_p
            L.ora_error.argtypes = [C.c_void_p]
            L.ora_nrows.restype = C.c_int64
            L.ora_nrows.argtypes = [C.c_void_p, C.c_int]
            L.ora_get_d.argtypes = [C.c_void_p, C.c_void_p]
            L.ora_get_str.restype = C.c_char_p
            L.ora_get_str.argtypes = [C.c_void_p, C.c_int64]
            L.ora_free.argtypes = [C.c_void_p]
            _LIB = L
    return _LIB


def _run(tool, lat, wspace, other_groups, **o):
    import numpy as np
    label_group = {0: 0}
    for w in wspace:
        label_group[w] = 1
    inc = [ora.INT_MAX]
    for gi, grp in enumerate(other_groups):
        for lab in grp:
            label_group[lab] = gi + 2
        inc.append(gi + 2)
    L = lib()
    ol, k1 = ora.make_lat(lat)
    oo, k2 = ora.make_opts(label_group=label_group, inc_groups=inc, del_groups=[1], **o)
    h = L.charutt_run(tool, C.byref(ol), C.byref(oo))
    try:
        err = L.ora_error(h).decode()
        if err:
            raise RuntimeError("char utterance reference: " + err)
        d = np.zeros(L.ora_nrows(h, 4), np.float64)
        L.ora_get_d(h, d.ctypes.data_as(C.c_void_p) if d.size else None)
        s = [L.ora_get_str(h, i).decode() for i in range(L.ora_nrows(h, 7))]
        return list(zip(s, d.tolist()))
    finally:
        L.ora_free(h)


def char_utterance(lat, wspace, other_groups=(), **o):
    """Rows (string, logp), logp = log P(the pseudo-word occurs at least once in the line), the
    nbest best by (logp desc, string asc): run search + first-occurrence DP."""
    return _run(CHAR_UTTERANCE, lat, wspace, other_groups, **o)


def brute_char_utterance(lat, wspace, other_groups=(), **o):
    """The same rows from the list of all paths (tiny lattices)."""
    return _run(BRUTE_CHAR_UTTERANCE, lat, wspace, other_groups, **o)
