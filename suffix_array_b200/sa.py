"""Host-side mirror of the reference's `SuffixArray` (/root/reference/src/sa.rs:14-374) over the
C ABI of libsab200.so.  Same method names, argument meaning and error behaviour, so the parity
tests read like the reference's own tests (src/tests.rs).  Every method that computes -- new/set,
from_parts, enable_buckets, contains, search_all, search_lcp and their *_batch forms -- runs on
the GPU through include/sab200.h; there is no CPU fallback.

Differences forced by the host language: `search_all` returns a numpy view of the suffix array
(the reference returns `&[u32]`), `search_lcp` returns a Python `range` (reference: `Range<usize>`),
`from_parts` returns None instead of `Option::None`.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import MAX_LENGTH, BKT_LEN, SabError


def _as_text(s):
    if isinstance(s, np.ndarray):
        if s.dtype != np.uint8:
            raise TypeError("text must be bytes-like or a uint8 array")
        return np.ascontiguousarray(s)
    return np.frombuffer(bytes(s), dtype=np.uint8)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def _pack_patterns(pats):
    """list of bytes-like -> (uint8 concatenation, uint64 offsets[np+1])"""
    lens = np.fromiter((len(p) for p in pats), dtype=np.uint64, count=len(pats))
    offs = np.zeros(len(pats) + 1, dtype=np.uint64)
    np.cumsum(lens, out=offs[1:])
    flat = np.frombuffer(b"".join(bytes(p) for p in pats), dtype=np.uint8)
    return flat, offs


def _batch_input(pats, offs):
    """(concatenation, offsets) as given, or packed from a list of bytes-like -> (flat, offs, number of patterns)"""
    flat, offs = (pats, offs) if offs is not None else _pack_patterns(pats)
    flat = np.ascontiguousarray(flat, dtype=np.uint8)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    return flat, offs, offs.size - 1


def saca(s, sa, ngpus=1):
    """src/saca.rs:9-15.  Asserts mirror the reference's (`:10-11`), with the new MAX_LENGTH."""
    assert s.size <= MAX_LENGTH
    assert s.size + 1 == sa.size
    L = _lib.require_gpu()
    _lib.check(L.sab200_saca(_ptr(s), s.size, sa.ctypes.data_as(C.c_void_p), ngpus), "sab200_saca")


def bwt(s):
    """Burrows-Wheeler transform of `s` (include/sab200.h): -> (uint8 array of n bytes, primary index).  The last
    column of the n+1 sorted rotations of s$ without the row of '$'; bwt(b"banana") gives (b"annbaa", 4).  The suffix
    array is built and used on the GPU; only the n bytes come back."""
    t = _as_text(s)
    assert t.size <= MAX_LENGTH
    out = np.empty(t.size, dtype=np.uint8)
    p = C.c_uint64()
    L = _lib.require_gpu()
    _lib.check(L.sab200_bwt(_ptr(t), t.size, _ptr(out), C.byref(p)), "sab200_bwt")
    return out, int(p.value)


def inverse_bwt(u, primary):
    """The text whose transform is (u, primary), as a uint8 array.  Raises ValueError when `primary` is outside
    [1, n] (0 for the empty transform) or `u` is the transform of no text."""
    t = _as_text(u)
    primary = int(primary)
    if t.size > MAX_LENGTH or not 0 <= primary < 2 ** 64:
        raise ValueError("bad transform length or primary index")
    out = np.empty(t.size, dtype=np.uint8)
    L = _lib.require_gpu()
    rc = L.sab200_inverse_bwt(_ptr(t), t.size, primary, _ptr(out))
    if rc == -1:
        raise ValueError(L.sab200_last_error().decode("utf-8", "replace"))
    _lib.check(rc, "sab200_inverse_bwt")
    return out


def lz77(s):
    """Greedy LZ77 factorization of `s` (include/sab200.h): -> (pos, len), uint32 arrays of the z factors.  Factor t
    is a literal (pos = the byte) when len = 0, else a copy of len bytes from the earlier position pos (the source may
    overlap the factor).  lz77(b"banana") gives pos [98, 97, 110, 1], len [0, 0, 0, 3].  Suffix array, LPF and parse
    are computed on the GPU; only the factors come back."""
    t = _as_text(s)
    assert t.size <= MAX_LENGTH
    pos = np.empty(t.size, dtype=np.uint32)  # cap = n always suffices; untouched pages are never committed
    ln = np.empty(t.size, dtype=np.uint32)
    z = C.c_uint64()
    L = _lib.require_gpu()
    _lib.check(L.sab200_lz77(_ptr(t), t.size, _ptr(pos), _ptr(ln), t.size, C.byref(z)), "sab200_lz77")
    return pos[:z.value].copy(), ln[:z.value].copy()


def lz77_decode(pos, len, n):
    """The n bytes of the parse (pos, len), greedy or not, as a uint8 array.  Raises ValueError when the factors do not
    parse n bytes: lengths max(1, len) not summing to n, a literal above 255, a copy whose source is not before it."""
    p = np.ascontiguousarray(pos, dtype=np.uint32)
    ln = np.ascontiguousarray(len, dtype=np.uint32)
    n = int(n)
    if p.shape != ln.shape or p.ndim != 1:
        raise ValueError("pos and len must be 1-D arrays of the same length")
    if not 0 <= n <= MAX_LENGTH:
        raise ValueError("n = %d outside [0, MAX_LENGTH]" % n)
    out = np.empty(n, dtype=np.uint8)
    L = _lib.require_gpu()
    rc = L.sab200_lz77_decode(_ptr(p), _ptr(ln), p.size, n, _ptr(out))
    if rc == -1:
        raise ValueError(L.sab200_last_error().decode("utf-8", "replace"))
    _lib.check(rc, "sab200_lz77_decode")
    return out


class SuffixArray:
    """Suffix array for a byte string (src/sa.rs:14-19): text `s`, `sa` of n+1 u32, optional buckets."""

    def __init__(self, s, _sa=None):
        self.s = _as_text(s)
        self.bkt = None
        self._index = None
        self._ngpus = 1
        if _sa is None:
            self.sa = np.zeros(self.s.size + 1, dtype=np.uint32)  # src/sa.rs:24
            saca(self.s, self.sa)                                  # src/sa.rs:25
        else:
            self.sa = _sa

    # ---- construction (src/sa.rs:23-33)
    @classmethod
    def new(cls, s):
        return cls(s)

    @classmethod
    def new_with_buckets(cls, s, ngpus=1):
        """new() + enable_buckets() (src/sa.rs:23-27, 89-119) in ONE library call: the bucket table falls out of the
        construction's sorted keys (sab200_saca_buckets; SURVEY.md 8f N2).  ngpus > 1 shards the construction."""
        t = _as_text(s)
        assert t.size <= MAX_LENGTH
        sa = np.zeros(t.size + 1, dtype=np.uint32)
        bkt = np.empty(BKT_LEN, dtype=np.uint32)
        L = _lib.require_gpu()
        _lib.check(L.sab200_saca_buckets(_ptr(t), t.size, sa.ctypes.data_as(C.c_void_p), bkt.ctypes.data_as(C.c_void_p), ngpus),
                   "sab200_saca_buckets")
        self = cls(t, _sa=sa)
        self.bkt = bkt
        return self

    def set(self, s):
        """src/sa.rs:30-33, literally: rebuilds `sa` for the new text but -- as in the reference --
        neither replaces the stored text nor clears the bucket table (SURVEY.md Q4)."""
        t = _as_text(s)
        self.sa = np.resize(self.sa, t.size + 1)
        saca(t, self.sa)
        self._drop_index()

    def fit(self):
        """src/sa.rs:36-38 (shrink_to_fit): numpy arrays carry no slack; nothing to do."""

    def len(self):
        return int(self.s.size)

    def __len__(self):
        return self.len()

    def is_empty(self):
        return self.len() == 0

    def into_parts(self):
        """src/sa.rs:51-53"""
        self._drop_index()
        return self.s, self.sa

    @classmethod
    def from_parts(cls, s, sa):
        """src/sa.rs:57-64: None unless `sa` is the suffix array of `s` (GPU linear-time check)."""
        t = _as_text(s)
        a = np.ascontiguousarray(sa, dtype=np.uint32)
        L = _lib.require_gpu()
        rc = L.sab200_check(_ptr(t), t.size, a.ctypes.data_as(C.c_void_p), a.size)
        if rc < 0:
            _lib.check(rc, "sab200_check")
        return cls(t, _sa=a) if rc == 1 else None

    @classmethod
    def unchecked_from_parts(cls, s, sa):
        """src/sa.rs:68-70"""
        return cls(_as_text(s), _sa=np.ascontiguousarray(sa, dtype=np.uint32))

    # ---- buckets (src/sa.rs:89-119)
    def enable_buckets(self):
        if self.bkt is not None:  # src/sa.rs:90-92
            return
        L = _lib.require_gpu()
        bkt = np.empty(BKT_LEN, dtype=np.uint32)
        _lib.check(L.sab200_enable_buckets(_ptr(self.s), self.s.size, bkt.ctypes.data_as(C.c_void_p)),
                   "sab200_enable_buckets")
        self.bkt = bkt
        self._drop_index()

    # ---- LCP array (no reference counterpart: README.md:18-23; SURVEY.md 8f N4)
    def lcp_array(self):
        """lcp[0] = 0, lcp[j] = length of the common prefix of the suffixes sa[j-1] and sa[j] (utils::lcp,
        src/utils.rs:2-7), computed on the GPU (chunked Kasai)."""
        L = _lib.require_gpu()
        out = np.empty(self.sa.size, dtype=np.uint32)
        _lib.check(L.sab200_lcp_array(_ptr(self.s), self.s.size, self.sa.ctypes.data_as(C.c_void_p), self.sa.size,
                                      out.ctypes.data_as(C.c_void_p)), "sab200_lcp_array")
        return out

    # ---- resident index for the query kernels
    def use_gpus(self, ngpus):
        """Replicates the index on `ngpus` GPUs; batched queries are sharded across them."""
        if ngpus != self._ngpus:
            self._drop_index()
            self._ngpus = int(ngpus)

    def _drop_index(self):
        if self._index is not None:
            _lib.lib().sab200_index_destroy(self._index)
            self._index = None

    def _get_index(self):
        if self._index is None:
            L = _lib.require_gpu()
            h = L.sab200_index_create(_ptr(self.s), self.s.size, self.sa.ctypes.data_as(C.c_void_p), self.sa.size,
                                      self.bkt.ctypes.data_as(C.c_void_p) if self.bkt is not None else None,
                                      self._ngpus)
            if not h:
                raise SabError("sab200_index_create failed: " + L.sab200_last_error().decode("utf-8", "replace"))
            self._index = h
        return self._index

    def __del__(self):
        try:
            self._drop_index()
        except Exception:
            pass

    # ---- batched queries (the GPU side door next to the per-pattern methods)
    def search_all_batch(self, pats, offs=None):
        """-> (lo, hi) uint32 arrays; the reference's slice for pattern q is sa[lo[q]:hi[q]]."""
        flat, offs, np_ = _batch_input(pats, offs)
        lo = np.empty(np_, dtype=np.uint32)
        hi = np.empty(np_, dtype=np.uint32)
        _lib.check(_lib.lib().sab200_search_all_batch(self._get_index(), _ptr(flat), _ptr(offs), np_, _ptr(lo), _ptr(hi)),
                   "sab200_search_all_batch")
        return lo, hi

    def contains_batch(self, pats, offs=None):
        flat, offs, np_ = _batch_input(pats, offs)
        out = np.empty(np_, dtype=np.uint8)
        _lib.check(_lib.lib().sab200_contains_batch(self._get_index(), _ptr(flat), _ptr(offs), np_, _ptr(out)),
                   "sab200_contains_batch")
        return out.astype(bool)

    def search_lcp_batch(self, pats, offs=None):
        flat, offs, np_ = _batch_input(pats, offs)
        st = np.empty(np_, dtype=np.uint32)
        en = np.empty(np_, dtype=np.uint32)
        _lib.check(_lib.lib().sab200_search_lcp_batch(self._get_index(), _ptr(flat), _ptr(offs), np_, _ptr(st), _ptr(en)),
                   "sab200_search_lcp_batch")
        return st, en

    # ---- matching statistics (no reference counterpart; include/sab200.h)
    def matching_statistics_batch(self, queries, offs=None):
        """-> (len, lo, hi) uint32 arrays with one entry per byte of the concatenated queries.  At position i of a
        query Q, len[i] is the longest prefix of the rest of Q that occurs in the text, and sa[lo[i]:hi[i]] are the
        positions where it occurs ([0, n+1) when len[i] = 0).  The first call on an index builds its extension
        (integrity check, inverse suffix array, LCP array); a suffix array that is not the text's raises ValueError."""
        flat, offs, nq = _batch_input(queries, offs)
        total = int(offs[-1]) if nq > 0 else 0
        out = [np.empty(total, dtype=np.uint32) for _ in range(3)]
        L = _lib.lib()
        rc = L.sab200_matching_statistics_batch(self._get_index(), _ptr(flat), _ptr(offs), max(nq, 0), *[_ptr(o) for o in out])
        if rc == -1:
            raise ValueError(L.sab200_last_error().decode("utf-8", "replace"))
        _lib.check(rc, "sab200_matching_statistics_batch")
        return tuple(out)

    def matching_statistics(self, query):
        """matching_statistics_batch of the single query"""
        return self.matching_statistics_batch([query])

    # ---- per-pattern queries (src/sa.rs:164-253)
    def contains(self, pat):
        return bool(self.contains_batch([pat])[0])

    def search_all(self, pat):
        lo, hi = self.search_all_batch([pat])
        return self.sa[int(lo[0]):int(hi[0])]

    def search_lcp(self, pat):
        st, en = self.search_lcp_batch([pat])
        return range(int(st[0]), int(en[0]))

    # ---- pack serialisation (feature "pack": src/sa.rs:256-361 over src/packed_sa.rs)
    def dump_bytes(self):
        """src/sa.rs:275-278 -> bytes (bincode header + BitPacker4x blocks, packed on the GPU)."""
        L = _lib.require_gpu()
        cap = int(L.sab200_pack_bound(self.sa.size))
        out = np.empty(cap, dtype=np.uint8)
        n = C.c_uint64()
        _lib.check(L.sab200_pack(self.sa.ctypes.data_as(C.c_void_p), self.sa.size, out.ctypes.data_as(C.c_void_p), cap,
                                 C.byref(n)), "sab200_pack")
        return out[:n.value].tobytes()

    def dump(self, file):
        """src/sa.rs:257-260: writes to a binary file object."""
        file.write(self.dump_bytes())

    def dump_file(self, name):
        """src/sa.rs:264-271"""
        with open(name, "wb") as f:
            self.dump(f)

    @classmethod
    def unchecked_load_bytes(cls, s, data):
        """src/sa.rs:338-346: no integrity check.  Malformed input raises ValueError (io::Error in the reference)."""
        L = _lib.require_gpu()
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        if buf.size < 16:
            raise ValueError("truncated packed suffix array")
        length = int(np.frombuffer(buf[4:8].tobytes(), dtype="<u4")[0])
        sa = np.empty(max(length, 1), dtype=np.uint32)
        n = C.c_uint64()
        rc = L.sab200_unpack(buf.ctypes.data_as(C.c_void_p), buf.size, sa.ctypes.data_as(C.c_void_p), sa.size, C.byref(n))
        if rc == -1:
            raise ValueError(L.sab200_last_error().decode("utf-8", "replace"))
        _lib.check(rc, "sab200_unpack")
        return cls.unchecked_from_parts(s, sa[:n.value])

    @classmethod
    def load_bytes(cls, s, data):
        """src/sa.rs:349-361: ValueError("inconsistent suffix array") where the reference returns InvalidData."""
        obj = cls.unchecked_load_bytes(s, data)
        if cls.from_parts(obj.s, obj.sa) is None:
            raise ValueError("inconsistent suffix array")
        return obj

    @classmethod
    def unchecked_load(cls, s, file):
        return cls.unchecked_load_bytes(s, file.read())

    @classmethod
    def load(cls, s, file):
        """src/sa.rs:293-305"""
        return cls.load_bytes(s, file.read())

    @classmethod
    def unchecked_load_file(cls, s, name):
        with open(name, "rb") as f:
            return cls.unchecked_load(s, f)

    @classmethod
    def load_file(cls, s, name):
        """src/sa.rs:323-335"""
        with open(name, "rb") as f:
            return cls.load(s, f)

    # ---- conversions (src/sa.rs:364-374)
    def __array__(self, dtype=None, copy=None):
        return self.sa if dtype is None else self.sa.astype(dtype)

    def as_ref(self):
        return self.s
