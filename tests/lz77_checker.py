"""ctypes binding of tests/lz77_checker.c, the CPU checkers of the LZ77 factorization.  The shared object is compiled on
first use into the temporary directory, so a read-only tree works too."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lz77_checker.c")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        with open(_SRC, "rb") as f:
            tag = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "sab200_lz77_checker_%s_%d.so" % (tag, os.getuid()))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-std=c99", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        vp, u64 = C.c_void_p, C.c_uint64
        L.checker_lz77_brute.argtypes = [vp, u64, vp, vp, C.POINTER(u64)]
        L.checker_lz77_brute.restype = C.c_int
        L.checker_lz77_sa.argtypes = [vp, u64, vp, vp, vp, C.POINTER(u64)]
        L.checker_lz77_sa.restype = C.c_int
        L.checker_lz77_verify.argtypes = [vp, u64, vp, vp, u64]
        L.checker_lz77_verify.restype = C.c_int64
        L.checker_lz77_decode.argtypes = [vp, vp, u64, u64, vp]
        L.checker_lz77_decode.restype = C.c_int
        _LIB = L
    return _LIB


def _u8(a):
    a = np.frombuffer(bytes(a), dtype=np.uint8) if not isinstance(a, np.ndarray) else a
    return np.ascontiguousarray(a, dtype=np.uint8)


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def _buf(n):
    return np.empty(max(n, 1), dtype=np.uint32)


def lz77_brute(s):
    """(pos, len) of the greedy parse by brute force; pos is the byte for literals and 0 for copies (no source)."""
    t = _u8(s)
    pos, ln, z = _buf(t.size), _buf(t.size), C.c_uint64()
    assert lib().checker_lz77_brute(t.ctypes.data, t.size, pos.ctypes.data, ln.ctypes.data, C.byref(z)) == 0
    return pos[:z.value].copy(), ln[:z.value].copy()


def lz77(s, sa):
    """(pos, len) by the definition of include/sab200.h over the suffix array `sa` (n+1 entries, sa[0] = n)."""
    t = _u8(s)
    sa = _u32(sa)
    assert sa.size == t.size + 1
    pos, ln, z = _buf(t.size), _buf(t.size), C.c_uint64()
    assert lib().checker_lz77_sa(t.ctypes.data, t.size, sa.ctypes.data, pos.ctypes.data, ln.ctypes.data, C.byref(z)) == 0
    return pos[:z.value].copy(), ln[:z.value].copy()


def verify(s, pos, ln):
    """0 when (pos, len) is a greedy parse of s, else 1 + the index of the first bad factor."""
    t, pos, ln = _u8(s), _u32(pos), _u32(ln)
    return int(lib().checker_lz77_verify(t.ctypes.data, t.size, pos.ctypes.data, ln.ctypes.data, pos.size))


def decode(pos, ln, n):
    """The n bytes of the parse, or None when it breaks a rule."""
    pos, ln = _u32(pos), _u32(ln)
    out = np.empty(n, dtype=np.uint8)
    rc = lib().checker_lz77_decode(pos.ctypes.data, ln.ctypes.data, pos.size, n, out.ctypes.data)
    return out if rc == 0 else None
