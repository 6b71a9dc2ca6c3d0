"""ctypes binding of tests/ms_checker.c, the CPU checkers of the matching statistics.  The shared object is compiled
on first use into the temporary directory, so a read-only tree works too."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ms_checker.c")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        with open(_SRC, "rb") as f:
            tag = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "sab200_ms_checker_%s_%d.so" % (tag, os.getuid()))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-std=c99", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        vp, u64 = C.c_void_p, C.c_uint64
        L.checker_ms_naive.argtypes = [vp, u64, vp, vp, u64, vp, vp, vp]
        L.checker_ms_naive.restype = C.c_int
        L.checker_ms_bisect.argtypes = [vp, u64, vp, vp, vp, u64, vp, vp, vp]
        L.checker_ms_bisect.restype = C.c_int
        _LIB = L
    return _LIB


def _u8(a):
    a = np.frombuffer(bytes(a), dtype=np.uint8) if not isinstance(a, np.ndarray) else a
    return np.ascontiguousarray(a, dtype=np.uint8)


def _run(fn, s, qs, offs, *pre):
    t, q = _u8(s), _u8(qs)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    total = int(offs[-1])
    out = [np.zeros(total, dtype=np.uint32) for _ in range(3)]
    args = [t.ctypes.data, t.size] + [a.ctypes.data for a in pre] + [q.ctypes.data, offs.ctypes.data, offs.size - 1]
    assert fn(*args, *[o.ctypes.data for o in out]) == 0
    return tuple(out)


def naive(s, qs, offs):
    """(len, lo, hi) by the definition, over every text position (no suffix array)"""
    return _run(lib().checker_ms_naive, s, qs, offs)


def bisect(s, sa, qs, offs):
    """(len, lo, hi) by a lower-bound search of every query suffix over `sa` (n+1 entries)"""
    return _run(lib().checker_ms_bisect, s, qs, offs, np.ascontiguousarray(sa, dtype=np.uint32))
