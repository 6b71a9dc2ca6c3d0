"""ctypes loader of libsab200.so (the CUDA engine, built for sm_100a).

There is no CPU path: if the shared library is missing, or no CUDA device is visible, loading
fails loudly -- nothing in this package falls back to the oracle or to numpy.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SAB200_LIB: developer override to A/B-test a variant build of the same CUDA engine
LIB_PATH = os.environ.get("SAB200_LIB") or os.path.join(_HERE, "libsab200.so")
MAX_LENGTH = 0xFFFFFFFE  # include/sab200.h SAB200_MAX_LENGTH (replaces src/saca.rs:6)
BKT_LEN = 256 * 257 + 1
MAX_ROUNDS = 64

_lib = None


class SabError(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [
        ("n", C.c_uint64),
        ("sigma", C.c_uint32),
        ("bits_per_symbol", C.c_uint32),
        ("symbols_per_key", C.c_uint32),
        ("rounds", C.c_uint32),
        ("active", C.c_uint64 * MAX_ROUNDS),
        ("passes", C.c_uint32 * MAX_ROUNDS),
        ("radix_pass_launches", C.c_uint64),
        ("radix_pass_records", C.c_uint64),
        ("radix_pass_bytes", C.c_uint64),
        ("radix_pass_ms", C.c_double),
        ("hist_ms", C.c_double),
        ("pack_ms", C.c_double),
        ("rank_ms", C.c_double),
        ("gather_ms", C.c_double),
        ("total_ms", C.c_double),
        ("h2d_ms", C.c_double),
        ("d2h_ms", C.c_double),
        ("kernel_launches", C.c_uint64),
        ("group_sort_ms", C.c_double),
        ("group_sort_records", C.c_uint64),
        ("group_big_records", C.c_uint64),
    ]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if hasattr(v, "__len__") else v
        r = d["rounds"] + 1
        d["active"] = d["active"][:r]
        d["passes"] = d["passes"][:r]
        return d


PHASES = 16


class DistStats(C.Structure):
    """include/sab200.h sab200_dist_stats"""
    _fields_ = [
        ("nranks", C.c_uint32), ("rank", C.c_uint32), ("rounds", C.c_uint32), ("lazy_isa", C.c_uint32),
        ("rank_layout", C.c_uint32), ("rebalanced", C.c_uint32), ("p2p_rounds", C.c_uint32), ("fused_exchange", C.c_uint32),
        ("slice_len", C.c_uint64), ("sa_off", C.c_uint64), ("all_to_all_bytes", C.c_uint64), ("collectives", C.c_uint64),
        ("resolved_empty", C.c_uint64),
        ("active", C.c_uint64 * MAX_ROUNDS),
        ("phase_ms", C.c_double * PHASES),
        ("total_ms", C.c_double),
        ("wall_ms", C.c_double),
        ("host_setup_ms", C.c_double),
        ("host_finish_ms", C.c_double),
    ]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if hasattr(v, "__len__") else v
        d["active"] = d["active"][:d["rounds"] + 1]
        return d


def build(verbose=False):
    """Compiles the CUDA engine in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    import subprocess
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc"), "all"],
                          stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


def lib():
    """The loaded CDLL with argtypes set.  Raises SabError when the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SabError("libsab200.so is missing (%s): build it with `python -c 'import __graft_entry__ as g; "
                       "g.build()'` or `make -C suffix_array_b200/csrc`; there is no CPU fallback" % LIB_PATH)
    _lib = _bind(C.CDLL(LIB_PATH))
    return _lib


def _bind(L):
    """Sets the prototypes of include/sab200.h on a loaded library."""
    vp, u64, i32 = C.c_void_p, C.c_uint64, C.c_int32
    L.sab200_saca.argtypes = [vp, u64, vp, i32]
    L.sab200_saca.restype = i32
    L.sab200_saca_device.argtypes = [vp, u64, vp, i32]
    L.sab200_saca_device.restype = i32
    L.sab200_get_stats.argtypes = [C.POINTER(Stats)]
    L.sab200_get_stats.restype = i32
    L.sab200_set_profiling.argtypes = [i32]
    L.sab200_set_profiling.restype = None
    L.sab200_last_error.argtypes = []
    L.sab200_last_error.restype = C.c_char_p
    L.sab200_device_count.argtypes = []
    L.sab200_device_count.restype = i32
    L.sab200_version.argtypes = []
    L.sab200_version.restype = C.c_char_p
    L.sab200_shutdown.argtypes = []
    L.sab200_shutdown.restype = None
    _opt = {
        "sab200_enable_buckets": ([vp, u64, vp], i32),
        "sab200_saca_buckets": ([vp, u64, vp, vp, i32], i32),
        "sab200_check": ([vp, u64, vp, u64], i32),
        "sab200_lcp_array": ([vp, u64, vp, u64, vp], i32),
        "sab200_bwt": ([vp, u64, vp, C.POINTER(u64)], i32),
        "sab200_inverse_bwt": ([vp, u64, u64, vp], i32),
        "sab200_bwt_device": ([vp, u64, vp, C.POINTER(u64), i32], i32),
        "sab200_inverse_bwt_device": ([vp, u64, u64, vp, i32], i32),
        "sab200_lz77": ([vp, u64, vp, vp, u64, C.POINTER(u64)], i32),
        "sab200_lz77_decode": ([vp, vp, u64, u64, vp], i32),
        "sab200_lz77_device": ([vp, u64, vp, vp, u64, C.POINTER(u64), i32], i32),
        "sab200_lz77_decode_device": ([vp, vp, u64, u64, vp, i32], i32),
        "sab200_index_create": ([vp, u64, vp, u64, vp, i32], vp),
        "sab200_index_destroy": ([vp], None),
        "sab200_search_all_batch": ([vp, vp, vp, u64, vp, vp], i32),
        "sab200_contains_batch": ([vp, vp, vp, u64, vp], i32),
        "sab200_search_lcp_batch": ([vp, vp, vp, u64, vp, vp], i32),
        "sab200_search_all_batch_device": ([vp, vp, vp, u64, vp, vp], i32),
        "sab200_matching_statistics_batch": ([vp, vp, vp, u64, vp, vp, vp], i32),
        "sab200_matching_statistics_batch_device": ([vp, vp, vp, u64, vp, vp, vp], i32),
        "sab200_index_directory": ([vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)], u64),
        "sab200_index_probes": ([vp, i32], u64),
        "sab200_pack_bound": ([u64], u64),
        "sab200_pack": ([vp, u64, vp, u64, C.POINTER(u64)], i32),
        "sab200_unpack": ([vp, u64, vp, u64, C.POINTER(u64)], i32),
        "sab200_comm_unique_id": ([vp], i32),
        "sab200_comm_create_nccl": ([C.c_char_p, i32, i32, i32], vp),
        "sab200_comm_create_callbacks": ([vp, i32, i32, i32], vp),
        "sab200_comm_destroy": ([vp], None),
        "sab200_saca_sharded": ([vp, vp, u64, u64, i32, vp, u64, i32, C.POINTER(u64), C.POINTER(u64), C.POINTER(vp)], i32),
        "sab200_copy_from_device": ([vp, vp, u64, i32], i32),
        "sab200_sort_pairs_device": ([vp, vp, vp, vp, u64, i32, i32], i32),
        "sab200_group_sort_device": ([vp, vp, vp, vp, u64, i32, i32, i32, C.POINTER(u64)], i32),
        "sab200_comm_stats": ([vp, C.POINTER(DistStats)], i32),
        "sab200_multi_stats": ([i32, C.POINTER(DistStats)], i32),
    }
    for name, (args, res) in _opt.items():
        f = getattr(L, name)
        f.argtypes = args
        f.restype = res
    return L


def require_gpu():
    L = lib()
    if L.sab200_device_count() < 1:
        raise SabError("no CUDA device visible: suffix_array_b200 is a GPU engine and has no CPU fallback")
    return L


def check(rc, what):
    if rc != 0:
        raise SabError("%s failed (rc=%d): %s" % (what, rc, lib().sab200_last_error().decode("utf-8", "replace")))


def last_stats():
    s = Stats()
    check(lib().sab200_get_stats(C.byref(s)), "sab200_get_stats")
    return s.as_dict()
