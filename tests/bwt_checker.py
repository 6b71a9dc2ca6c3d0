"""ctypes binding of tests/bwt_checker.c, the CPU checkers of the Burrows-Wheeler transform.  The shared object is
compiled on first use into the temporary directory, so a read-only tree works too."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "bwt_checker.c")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        with open(_SRC, "rb") as f:
            tag = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "sab200_bwt_checker_%s_%d.so" % (tag, os.getuid()))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-std=c99", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.checker_bwt.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
        L.checker_bwt.restype = C.c_int
        L.checker_inverse_bwt.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
        L.checker_inverse_bwt.restype = C.c_int
        _LIB = L
    return _LIB


def _u8(a):
    a = np.frombuffer(bytes(a), dtype=np.uint8) if not isinstance(a, np.ndarray) else a
    return np.ascontiguousarray(a, dtype=np.uint8)


def bwt(s, sa):
    """(transform, primary index) of `s` by the definition, from its suffix array `sa` (n+1 entries, sa[0] = n)."""
    t = _u8(s)
    sa = np.ascontiguousarray(sa, dtype=np.uint32)
    assert sa.size == t.size + 1
    out = np.empty(t.size, dtype=np.uint8)
    p = C.c_uint64()
    assert lib().checker_bwt(t.ctypes.data, t.size, sa.ctypes.data, out.ctypes.data, C.byref(p)) == 0
    return out, int(p.value)


def inverse_bwt(u, primary):
    """The text of (u, primary) by the LF walk, or None when (u, primary) is the transform of no text."""
    t = _u8(u)
    out = np.empty(t.size, dtype=np.uint8)
    rc = lib().checker_inverse_bwt(t.ctypes.data, t.size, int(primary), out.ctypes.data)
    assert rc in (0, -1), rc
    return out if rc == 0 else None
