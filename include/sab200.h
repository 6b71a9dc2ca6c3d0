/*
 * sab200.h -- C ABI of the B200-native suffix-array engine (libsab200.so).
 *
 * This is the drop-in boundary for the hot path of the Rust crate hucsmn/suffix_array v0.5.0:
 * every entry point names the reference interface it replaces (file:line under /root/reference).
 * Plain pointers and sizes only; the caller owns every host buffer; the library owns only device
 * memory, streams and events, and keeps no host pointer after a call returns.  There is no CPU
 * fallback: without a CUDA device every compute entry point returns SAB200_ERR_CUDA.
 *
 * Return codes: 0 ok; -1 bad arguments; -2 host/device out of memory; -3 CUDA error;
 * -4 NCCL error; -5 internal error.  sab200_last_error() describes the last failure of the
 * calling thread's most recent call (process-wide string, best effort).
 */
#ifndef SAB200_H
#define SAB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAB200_OK 0
#define SAB200_ERR_ARGS (-1)
#define SAB200_ERR_OOM (-2)
#define SAB200_ERR_CUDA (-3)
#define SAB200_ERR_NCCL (-4)
#define SAB200_ERR_INTERNAL (-5)

/* Replaces `pub const MAX_LENGTH` (src/saca.rs:6, re-exported src/lib.rs:53).  The reference's
 * i32::MAX came from divsufsort's signed indices; the u32 suffix array and the u32 bucket prefix
 * sums (src/sa.rs:112-116) allow n + 1 <= u32::MAX. */
#define SAB200_MAX_LENGTH 0xFFFFFFFEull

/* Length of the bucket table of enable_buckets (src/sa.rs:95): 256 * 257 + 1. */
#define SAB200_BKT_LEN 65793u

#define SAB200_MAX_ROUNDS 64

/* Counters of the last construction on the calling process (for the roofline report). */
typedef struct sab200_stats {
    uint64_t n;
    uint32_t sigma;
    uint32_t bits_per_symbol;
    uint32_t symbols_per_key;
    uint32_t rounds;
    uint64_t active[SAB200_MAX_ROUNDS];
    uint32_t passes[SAB200_MAX_ROUNDS];
    uint64_t radix_pass_launches;
    uint64_t radix_pass_records;
    uint64_t radix_pass_bytes;   /* sum of 2*(K+V)*m over the radix-pass launches */
    double radix_pass_ms;        /* sum of their CUDA-event durations (profiling on) */
    double hist_ms;
    double pack_ms;
    double rank_ms;
    double gather_ms;
    double total_ms;
    double h2d_ms, d2h_ms;
    uint64_t kernel_launches;
    double group_sort_ms;          /* in-group sorts of the rounds (group_sort_kernel + scatter-back) */
    uint64_t group_sort_records;   /* records that went through group_sort_kernel */
    uint64_t group_big_records;    /* ... of which in groups too large for it (radix-sorted) */
} sab200_stats;

/* ---- construction -------------------------------------------------------------------------
 * Replaces saca::saca (src/saca.rs:9-15), the only callee of SuffixArray::new / set
 * (src/sa.rs:25,32): fills all n+1 entries of `sa`, sa[0] = n (src/saca.rs:13), sa[1..] = the
 * suffix starts in increasing suffix order (what cdivsufsort::sort_in_place wrote, src/saca.rs:14).
 * `s` (n bytes) and `sa` (n+1 entries) are HOST buffers owned by the caller (src/sa.rs:24).
 * ngpus = 1: one GPU.  ngpus = 2..16 (at most sab200_device_count()): the text is block-sharded over the
 * first ngpus devices of this process -- one host thread and one stream per GPU, an NCCL communicator
 * created inside the library (ncclCommInitAll, cached between calls) -- and built by the distributed
 * sample sort + prefix doubling described under "multi-GPU" below; every GPU uploads its own shard and
 * downloads its own slice of the suffix array over its own PCIe link.  Returns SAB200_ERR_NCCL when NCCL
 * is not installed or a collective fails.  ngpus = 0 means "all visible devices".
 * The reference panics when n > MAX_LENGTH (src/saca.rs:10); this returns SAB200_ERR_ARGS. */
int32_t sab200_saca(const uint8_t* s, uint64_t n, uint32_t* sa, int32_t ngpus);

/* SuffixArray::new followed by enable_buckets (src/sa.rs:23-27, 89-119) in one call: the bucket table falls out
 * of the construction's sorted initial keys (65 793 binary searches: no pass over the text, no second upload;
 * SURVEY.md 8f N2).  `bkt` receives SAB200_BKT_LEN entries, bit-identical to sab200_enable_buckets. */
int32_t sab200_saca_buckets(const uint8_t* s, uint64_t n, uint32_t* sa, uint32_t* bkt, int32_t ngpus);

/* Same computation with DEVICE buffers already resident on `device` (no copies): d_s holds n
 * bytes, d_sa receives n+1 entries.  Used to time the device pipeline without PCIe. */
int32_t sab200_saca_device(const uint8_t* d_s, uint64_t n, uint32_t* d_sa, int32_t device);

/* ---- bucket index -------------------------------------------------------------------------
 * Replaces the body of SuffixArray::enable_buckets (src/sa.rs:89-119): writes the SAB200_BKT_LEN
 * inclusive right-boundaries of the 2-byte-prefix buckets, layout
 * [$; (0,$),(0,0)..(0,255); ...; (255,$)..(255,255)] (src/sa.rs:94), slot(c0,$) = c0*257+1,
 * slot(c0,c1) = c0*257+c1+2 (src/sa.rs:103,107), u32 wrap-around sums (src/sa.rs:112-116).
 * Reads the text only, like the reference.  `s`, `bkt` are host buffers. */
int32_t sab200_enable_buckets(const uint8_t* s, uint64_t n, uint32_t* bkt);

/* ---- integrity -----------------------------------------------------------------------------
 * Replaces SuffixArray::check_integrity behind from_parts (src/sa.rs:57-84) with a linear-time
 * equivalent (permutation via the inverse array, then neighbour order through the first byte and
 * the ranks of the tails).  Returns 1 (valid), 0 (not the suffix array of s; also when
 * sa_len != n+1, src/sa.rs:73-75, or an entry exceeds n, where the reference would panic), <0 error. */
int32_t sab200_check(const uint8_t* s, uint64_t n, const uint32_t* sa, uint64_t sa_len);

/* ---- LCP array -----------------------------------------------------------------------------
 * No reference counterpart (README.md:18-23 declines the enhanced suffix array; SURVEY.md 8f N4): lcp[0] = 0
 * and lcp[j] = utils::lcp(&s[sa[j-1]..], &s[sa[j]..]) (src/utils.rs:2-7) for j = 1..n.  `sa` must be the suffix
 * array of `s` (n + 1 entries); host buffers.  Kasai's recurrence in chunks of consecutive text positions: the
 * first position of a chunk compares from scratch, the others extend the previous length minus one. */
int32_t sab200_lcp_array(const uint8_t* s, uint64_t n, const uint32_t* sa, uint64_t sa_len, uint32_t* lcp);

/* ---- Burrows-Wheeler transform ----------------------------------------------------------------
 * libdivsufsort's divbwt / inverse_bw_transform, which the reference does not expose.  Over the n+1 rows of the
 * suffix array sab200_saca builds (sa[0] = n): the last column is L[j] = s[sa[j]-1] where sa[j] > 0, and L[p] = '$' at
 * the single row p with sa[p] = 0, the PRIMARY INDEX (1 <= p <= n for n >= 1).  The transform is L without row p:
 * n bytes, bwt[0] = s[n-1].  The empty text gives an empty transform and p = 0.  Example: "banana" -> ("annbaa", 4).
 * This is the layout libdivsufsort documents for divbwt; libdivsufsort is not in the tree, so byte parity with it is
 * pinned only by this definition (like the pack bytes above).
 *
 * sab200_bwt builds the suffix array on the GPU as sab200_saca does (its statistics stay readable through
 * sab200_get_stats), gathers L there, and moves only the n bytes of the transform back.  It takes no device memory
 * beyond what sab200_saca takes.
 * sab200_inverse_bwt returns the text of (bwt, primary).  A primary outside [1, n] (outside {0} when n = 0), or a bwt
 * that is the transform of no text, returns SAB200_ERR_ARGS with sab200_last_error saying which; `s` is then left
 * unwritten.  Device memory: about 25 bytes per byte of text.
 * Host buffers, pageable or pinned; one GPU. */
int32_t sab200_bwt(const uint8_t* s, uint64_t n, uint8_t* bwt, uint64_t* primary);
int32_t sab200_inverse_bwt(const uint8_t* bwt, uint64_t n, uint64_t primary, uint8_t* s);
/* The same with DEVICE buffers already resident on `device` (n bytes each), to time the device work without PCIe. */
int32_t sab200_bwt_device(const uint8_t* d_s, uint64_t n, uint8_t* d_bwt, uint64_t* primary, int32_t device);
int32_t sab200_inverse_bwt_device(const uint8_t* d_bwt, uint64_t n, uint64_t primary, uint8_t* d_s, int32_t device);

/* ---- Lempel-Ziv (LZ77) factorization ------------------------------------------------------------
 * No reference counterpart.  For a text s of n bytes, LPF[i] is the largest l with s[i .. i+l) = s[p .. p+l) for some
 * p < i (the two may overlap: p + l > i is allowed), 0 when s[i] does not occur before i.  The greedy factorization
 * has the starts b_0 = 0, b_{t+1} = b_t + max(1, LPF[b_t]), and z factors in all (b_z = n).  Factor t is
 * (pos[t], len[t]) with len[t] = LPF[b_t]; pos[t] = s[b_t] when len[t] = 0 (a literal), else the SOURCE, fixed so that
 * the output is deterministic: over the suffix array of sab200_saca (row 0, the empty suffix, is never chosen), with
 * j the row of suffix b_t, PSV / NSV are the nearest rows before / after j whose suffix starts before b_t, and the source
 * is whichever of sa[PSV], sa[NSV] shares the longer prefix with suffix b_t, sa[PSV] on a tie.  (LPF[i] is the longer
 * of these two common prefixes, Crochemore-Ilie.)  Examples:
 *   "banana" -> (b,0) (a,0) (n,0) (1,3), z = 4;   "aaaa" -> (a,0) (0,3), z = 2;   the empty text -> z = 0.
 *
 * sab200_lz77 builds the suffix array on the GPU as sab200_saca does (its statistics stay readable through
 * sab200_get_stats), then the inverse suffix array, the LCP array (comparing text only where the permuted LCP array is
 * irreducible: O(n log n) bytes, also on runs such as all-'a' text), LPF and sources at every position, the parse and the
 * compaction, all in the construction's workspace once the construction is done: device memory is what sab200_saca
 * takes (the construction workspace, the text and n + 1 suffix-array words: about 37 bytes per byte of text), and the
 * 8z bytes of output are carved from that workspace.  *z always receives the factor count; when cap < z the call returns SAB200_ERR_ARGS and writes no
 * factor.  cap = n always suffices.
 * sab200_lz77_decode returns the n bytes of any valid parse, greedy or not.  It returns SAB200_ERR_ARGS, with
 * sab200_last_error saying which rule failed, and leaves s unwritten, when the lengths max(1, len[t]) do not sum to n,
 * a literal has pos > 255, a copy has pos >= b_t, z > n, or n > SAB200_MAX_LENGTH.  Device memory: the input, the
 * output and 4(z + n) bytes.
 * Host buffers, pageable or pinned; one GPU. */
int32_t sab200_lz77(const uint8_t* s, uint64_t n, uint32_t* pos, uint32_t* len, uint64_t cap, uint64_t* z);
int32_t sab200_lz77_decode(const uint32_t* pos, const uint32_t* len, uint64_t z, uint64_t n, uint8_t* s);
/* The same with DEVICE buffers already resident on `device`, to time the device work without PCIe. */
int32_t sab200_lz77_device(const uint8_t* d_s, uint64_t n, uint32_t* d_pos, uint32_t* d_len, uint64_t cap,
                           uint64_t* z, int32_t device);
int32_t sab200_lz77_decode_device(const uint32_t* d_pos, const uint32_t* d_len, uint64_t z, uint64_t n,
                                  uint8_t* d_s, int32_t device);

/* ---- batched queries -----------------------------------------------------------------------
 * A resident copy of (text, SA, optional bucket table) on `ngpus` GPUs (replicated; queries are
 * sharded across the replicas, no collective).  bkt_or_null = NULL means "buckets not enabled"
 * (get_bucket then returns the whole array, src/sa.rs:141-143).  Host buffers; copied, not kept.
 * sa_len must be n + 1 (NULL is returned otherwise): the safe mirrors can hold a stale array after the
 * reference's set() quirk (src/sa.rs:30-33 keeps the old text), and a short one must not be over-read.
 * Entries of `sa` larger than n (only reachable through unchecked_from_parts) are treated as the empty
 * suffix by the kernels instead of indexing outside the text.
 * Device memory per replica: n + 4(n + 1) bytes, the bucket table, and the library-private prefix directory of at
 * most 2^27 + 1 u32 entries (one sweep over the suffix array at creation; see sab200_index_directory below). */
typedef struct sab200_index sab200_index;
sab200_index* sab200_index_create(const uint8_t* s, uint64_t n, const uint32_t* sa, uint64_t sa_len,
                                  const uint32_t* bkt_or_null, int32_t ngpus);
void sab200_index_destroy(sab200_index* ix);

/* Patterns are concatenated in `pats`; pattern q is pats[offs[q] .. offs[q+1]) (np+1 offsets).
 *
 * search_all (src/sa.rs:173-204): lo[q], hi[q] are GLOBAL suffix-array indices such that the slice
 * the reference returns is &sa[lo[q]..hi[q]] (SA order).  An empty pattern yields [0, n+1).
 * contains  (src/sa.rs:164-170): out[q] = 1/0.
 * search_lcp (src/sa.rs:207-253): [start[q], end[q]) is the text range the reference returns. */
int32_t sab200_search_all_batch(sab200_index* ix, const uint8_t* pats, const uint64_t* offs, uint64_t np,
                                uint32_t* lo, uint32_t* hi);
int32_t sab200_contains_batch(sab200_index* ix, const uint8_t* pats, const uint64_t* offs, uint64_t np, uint8_t* out);
int32_t sab200_search_lcp_batch(sab200_index* ix, const uint8_t* pats, const uint64_t* offs, uint64_t np,
                                uint32_t* start, uint32_t* end);
/* search_all with DEVICE pattern / result buffers on the GPU of replica 0 (kernel-only timing);
 * d_pats must be followed by at least 8 readable bytes. */
int32_t sab200_search_all_batch_device(sab200_index* ix, const uint8_t* d_pats, const uint64_t* d_offs, uint64_t np,
                                       uint32_t* d_lo, uint32_t* d_hi);

/* ---- matching statistics ---------------------------------------------------------------------
 * No reference counterpart.  Queries are passed like patterns: query q is qs[offs[q] .. offs[q+1]) (nq+1 offsets,
 * non-decreasing, else SAB200_ERR_ARGS; at most 2^31-1 queries).  For every byte position i of a query Q of m bytes
 * (i local to the query):
 *   len[i]          the largest l <= m - i such that Q[i .. i+l) is a substring of s (l = 0 allowed): a match never
 *                   runs past the end of its own query.  If i + len[i] < m, Q[i .. i+len[i]+1) does not occur in s.
 *   [lo[i], hi[i])  the GLOBAL suffix-array indices j in [0, n] whose suffix starts with Q[i .. i+len[i]): for
 *                   len[i] >= 1 exactly what sab200_search_all_batch returns for that pattern (hi - lo occurrences at
 *                   sa[lo .. hi)); [0, n+1) for len[i] = 0.
 * The outputs are indexed by the absolute byte offset in qs: each holds offs[nq] entries (entries before offs[0] are
 * not written).  With several replicas every replica receives the whole concatenation and walks an equal share of
 * the positions.  Host buffers, pageable or pinned.
 * The first call on an index extends it on every replica with the inverse suffix array, the LCP array and block
 * minima over it: 8(n+2) + about n/64 bytes per replica, at the cost of one integrity check and one LCP build per
 * replica.  A suffix array that is not the text's (reachable through unchecked_from_parts) returns SAB200_ERR_ARGS
 * and keeps no extension; an extension that does not fit returns SAB200_ERR_OOM.  The index stays usable either way. */
int32_t sab200_matching_statistics_batch(sab200_index* ix, const uint8_t* qs, const uint64_t* offs, uint64_t nq,
                                         uint32_t* len, uint32_t* lo, uint32_t* hi);
/* the same with DEVICE buffers on the GPU of replica 0 (kernel-only timing); d_qs is indexed by the absolute offsets
 * and must be followed by at least 8 readable bytes */
int32_t sab200_matching_statistics_batch_device(sab200_index* ix, const uint8_t* d_qs, const uint64_t* d_offs, uint64_t nq,
                                                uint32_t* d_len, uint32_t* d_lo, uint32_t* d_hi);

/* Introspection of a resident index (bench and tests).  sab200_index_create also builds a PREFIX DIRECTORY over the
 * resident text and suffix array (csrc/sab_search.cuh: number of suffixes below every code of `depth` leading symbols
 * in base `sigma`), from which search_all / contains start their bisection instead of from the whole two-byte
 * bucket; the answers are unchanged.  SAB_SEARCH_DIR=0 in the environment leaves it out.
 * sab200_index_directory: number of entries (0 = none), base and depth of replica 0.
 * sab200_index_probes: switches the counting of suffix comparisons in search_all on / off (one atomic per pattern:
 * not for timed runs) and returns the count accumulated so far over all replicas. */
uint64_t sab200_index_directory(sab200_index* ix, uint32_t* sigma, uint32_t* depth);
uint64_t sab200_index_probes(sab200_index* ix, int32_t count_on);

/* ---- pack serialisation --------------------------------------------------------------------
 * Replaces PackedSuffixArray::from_sa + dump_bytes and load_bytes + into_sa (src/packed_sa.rs:17-88,
 * 99-124; behind SuffixArray::dump* / load*, src/sa.rs:256-361, feature "pack"): bincode little-endian
 * header (magic "SA4x", length, data length) + BitPacker4x blocks of 128 values at
 * bits = 32 - clz(length - 1), trailing zero bytes of the last block dropped.  Host buffers.
 * sab200_pack_bound(len) bytes always suffice for sab200_pack.  The reference's two latent faults on
 * load (SURVEY.md Q9/Q10: length 1; fully trimmed last block) are guarded, not reproduced.  Byte parity
 * with the bitpacking/bincode crates is unpinned (they are not in the reference tree; its test only
 * checks the round trip, src/tests.rs:63-76). */
uint64_t sab200_pack_bound(uint64_t sa_len);
int32_t sab200_pack(const uint32_t* sa, uint64_t sa_len, uint8_t* out, uint64_t out_cap, uint64_t* out_len);
int32_t sab200_unpack(const uint8_t* bytes, uint64_t nbytes, uint32_t* sa, uint64_t sa_cap, uint64_t* sa_len);

/* ---- multi-GPU construction, one rank per GPU ------------------------------------------------
 * The sharded form of the same saca() (src/saca.rs:9-15) for callers that already run one process (or
 * thread) per GPU: rank g of P holds text positions [g*B, min((g+1)*B, n)), B = max(1, ceil(n / P)), followed
 * by up to SAB200_SHARD_HALO bytes of the next shard, and receives a contiguous slice of the suffix array.
 * The exchange steps (key all-to-all of the sample sort, rank requests / answers / updates of every doubling
 * round) are NCCL collectives enqueued by the library on its own stream.
 *
 *   one process per GPU:  rank 0 calls sab200_comm_unique_id, the host language broadcasts the 128 bytes,
 *                         every rank calls sab200_comm_create_nccl(id, rank, nranks, device).
 *   custom transport:     sab200_comm_create_callbacks -- the caller supplies the three collectives (the
 *                         CPU tests run the whole driver over gloo this way).  Buffers handed to a callback
 *                         are device pointers of the rank's GPU; the library stream is idle during the call.
 */
#define SAB200_SHARD_HALO 64u
#define SAB200_MAX_RANKS 16
typedef struct sab200_comm sab200_comm;
typedef struct sab200_comm_callbacks {
    void* user;
    /* recv[r*bytes .. (r+1)*bytes) = rank r's send[0 .. bytes) */
    int32_t (*all_gather)(void* user, const void* send, void* recv, uint64_t bytes);
    /* in-place sum of count u64 values over all ranks */
    int32_t (*all_reduce_sum_u64)(void* user, uint64_t* buf, uint64_t count);
    /* send[send_off[d] .. +send_bytes[d]) goes to rank d; recv[recv_off[s] .. +recv_bytes[s]) comes from rank s */
    int32_t (*all_to_all_v)(void* user, const void* send, const uint64_t* send_bytes, const uint64_t* send_off,
                            void* recv, const uint64_t* recv_bytes, const uint64_t* recv_off);
} sab200_comm_callbacks;

int32_t sab200_comm_unique_id(uint8_t id[128]);
sab200_comm* sab200_comm_create_nccl(const uint8_t id[128], int32_t rank, int32_t nranks, int32_t device);
sab200_comm* sab200_comm_create_callbacks(const sab200_comm_callbacks* cb, int32_t rank, int32_t nranks, int32_t device);
void sab200_comm_destroy(sab200_comm* comm);

/* Collective: every rank of `comm` calls it with its own shard of the same text of n bytes.
 *   shard / shard_len   this rank's positions + halo: at least min(count + 64, n - lo) bytes (count = own positions);
 *                       device memory of the rank's GPU when shard_on_device != 0, else host memory
 *   out / out_cap       receives the slice (u32 suffix starts); may be NULL.  Device or host like the shard.
 *   slice_len, sa_off   the slice holds suffix-array positions [sa_off, sa_off + slice_len); the sentinel
 *                       sa[0] = n (src/saca.rs:13) is implied: rank 0's slice starts at position 1
 *   d_slice             if not NULL: the slice inside the library's device arena (valid until the next call)
 * Returns SAB200_ERR_ARGS when out_cap < slice_len (slice_len is still reported). */
int32_t sab200_saca_sharded(sab200_comm* comm, const uint8_t* shard, uint64_t shard_len, uint64_t n, int32_t shard_on_device,
                            uint32_t* out, uint64_t out_cap, int32_t out_on_device, uint64_t* slice_len, uint64_t* sa_off,
                            const uint32_t** d_slice);

#define SAB200_PHASES 16
/* phase_ms index: 0 alphabet, 1 pack + splitters, 2 partition by destination, 3 key exchange, 4 local sort,
 * 5 ranks + SA skeleton, 6 ranks to owners, 7 rebalance, 8 round requests/answers, 9 lazy look-ups,
 * 10 round sorts, 11 re-rank, 12 rank updates, 13 new SA entries to their slices, 14 H2D, 15 D2H */
typedef struct sab200_dist_stats {
    uint32_t nranks, rank, rounds, lazy_isa, rank_layout /* 0 block, 1 block-cyclic */, rebalanced;
    uint32_t p2p_rounds, fused_exchange; /* rounds without an exchange step (peer loads / stores); key exchange fused into the partition */
    uint64_t slice_len, sa_off, all_to_all_bytes, collectives, resolved_empty;
    uint64_t active[SAB200_MAX_ROUNDS]; /* active suffixes over all ranks entering round r (0 = after the initial sort) */
    double phase_ms[SAB200_PHASES];     /* CUDA events on the rank's stream */
    double total_ms;                    /* first to last event of the construction on the rank's stream */
    double wall_ms;                     /* host clock around the whole call on this rank */
    double host_setup_ms;               /* ... of which before the first event (context, arena) */
    double host_finish_ms;              /* ... and after the last one (output copy excluded) */
} sab200_dist_stats;
/* Building block, exported for tests and tools: stable LSD radix sort of `count` (u64 key, u32 payload) records by
 * key bits [0, key_bits) over a double buffer of DEVICE memory on `device`.  Returns 0 / 1 = the buffer pair
 * (d_k0, d_v0) / (d_k1, d_v1) that holds the result, < 0 on error. */
int32_t sab200_sort_pairs_device(uint64_t* d_k0, uint64_t* d_k1, uint32_t* d_v0, uint32_t* d_v1, uint64_t count,
                                 int32_t key_bits, int32_t device);
/* Building block, exported for tests and tools: the in-group sort of a doubling round (csrc/sab_group_sort.cuh).
 * The `count` records of (d_k0, d_v0) are grouped by the high 32 bits of their keys (equal high words are
 * contiguous; `ascending` != 0: the groups also arrive in ascending order) and are ordered by the full key inside
 * every group; records with equal keys end up in unspecified order.  Device memory on `device`.  Returns the buffer
 * pair holding the result (always 1), < 0 on error; *nbig_out = records that took the radix-sort path. */
int32_t sab200_group_sort_device(uint64_t* d_k0, uint64_t* d_k1, uint32_t* d_v0, uint32_t* d_v1, uint64_t count,
                                 int32_t key_bits, int32_t ascending, int32_t device, uint64_t* nbig_out);
/* Copies `bytes` from the library's device arena on `device` (a d_slice pointer) into host memory. */
int32_t sab200_copy_from_device(void* dst, const void* d_src, uint64_t bytes, int32_t device);
/* counters of the last sharded construction on `comm` */
int32_t sab200_comm_stats(sab200_comm* comm, sab200_dist_stats* out);
/* counters of rank `rank` of the last sab200_saca(..., ngpus > 1) of this process */
int32_t sab200_multi_stats(int32_t rank, sab200_dist_stats* out);

/* ---- introspection ------------------------------------------------------------------------ */
int32_t sab200_get_stats(sab200_stats* out);
void sab200_set_profiling(int32_t on); /* per-launch CUDA events for the stats above */
const char* sab200_last_error(void);
int32_t sab200_device_count(void);     /* number of CUDA devices visible; 0 if none */
const char* sab200_version(void);
void sab200_shutdown(void);            /* releases device memory, streams and events */

#ifdef __cplusplus
}
#endif
#endif /* SAB200_H */
