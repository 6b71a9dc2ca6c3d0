"""suffix_array_b200 -- B200-native suffix-array construction and batched search, a drop-in for
the hot path of the Rust crate hucsmn/suffix_array (src/saca.rs, and the bucket/search methods of
src/sa.rs).  The CUDA engine (csrc/, sm_100a) sits behind the C ABI of include/sab200.h; this
package is the thin host mirror of the reference's `SuffixArray` interface.
"""
from ._lib import MAX_LENGTH, BKT_LEN, SabError, build, last_stats, lib, require_gpu
from .sa import SuffixArray, bwt, inverse_bwt, lz77, lz77_decode, saca

__all__ = ["SuffixArray", "saca", "bwt", "inverse_bwt", "lz77", "lz77_decode", "MAX_LENGTH", "BKT_LEN", "SabError", "build", "last_stats", "lib", "require_gpu"]
