// sab_radix.cuh -- hand-written LSD radix sort (8-bit digits) for (key, u32 payload) records.
//
//   radix_hist_kernel   one sweep over the keys -> 256-bin histograms of every digit place
//   radix_scan_kernel   exclusive scans of those histograms + "this pass is a no-op" flags
//   onesweep_kernel     one stable partition pass: tile histogram published early, records ranked per
//                       warp with ballots, tile prefixes chained by a two-level decoupled look-back
//                       (one lane per bin; tile partials + group words), records staged in sorted
//                       order through shared memory, coalesced write-out.
//
// Algorithmic traffic (SURVEY.md 8d): histogram K*m bytes; each pass 2*(K+V)*m bytes.
// Nothing here is a dense contraction; the bound is HBM bandwidth, tensor cores are not used.
#pragma once
#include "sab_common.cuh"

#define SAB_RADIX_BITS 8
#define SAB_RADIX_BINS 256
#define SAB_MAX_PASSES 8
#ifndef SAB_ONESWEEP_MIN_BLOCKS
#define SAB_ONESWEEP_MIN_BLOCKS 3
#endif

// look-back word: [63:36] epoch (28 bits) | [35:34] flag | [33:0] count
#define SAB_LB_VALUE_MASK ((1ull << 34) - 1ull)
#define SAB_LB_FLAG_PARTIAL (1ull << 34)
#define SAB_LB_FLAG_INCLUSIVE (2ull << 34)
#define SAB_LB_FLAG_MASK (3ull << 34)
#define SAB_LB_EPOCH_SHIFT 36
#define SAB_LB_EPOCH_MAX ((1u << 28) - 1u)

template <typename KeyT>
struct KeyTraits;
template <>
struct KeyTraits<u32> {
    static __device__ __forceinline__ u32 digit(u32 k, int shift) { return (k >> shift) & 0xffu; }
    static __device__ __forceinline__ u32 max_key() { return 0xffffffffu; }
};
template <>
struct KeyTraits<u64> {
    static __device__ __forceinline__ u32 digit(u64 k, int shift) { return (u32)(k >> shift) & 0xffu; }
    static __device__ __forceinline__ u64 max_key() { return ~0ull; }
};

// ------------------------------------------------------------------ histogram of all digit places
#define SAB_HIST_THREADS 512
#define SAB_HIST_ITEMS 8

template <typename KeyT>
__global__ void __launch_bounds__(SAB_HIST_THREADS)
radix_hist_kernel(const KeyT* __restrict__ keys, u64 n, int begin_bit, int npass, u64* __restrict__ ghist) {
    SAB_SHARED_ARRAY(u32, s_hist, SAB_MAX_PASSES * SAB_RADIX_BINS);
    for (int i = threadIdx.x; i < SAB_MAX_PASSES * SAB_RADIX_BINS; i += SAB_HIST_THREADS) s_hist[i] = 0;
    __syncthreads();
    const u64 tile = (u64)SAB_HIST_THREADS * SAB_HIST_ITEMS;
    const u64 ntiles = (n + tile - 1) / tile;
    for (u64 t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const u64 base = t * tile;
        KeyT k[SAB_HIST_ITEMS];
#pragma unroll
        for (int j = 0; j < SAB_HIST_ITEMS; ++j) {
            const u64 idx = base + (u64)j * SAB_HIST_THREADS + threadIdx.x;
            k[j] = idx < n ? keys[idx] : (KeyT)0;
        }
#pragma unroll
        for (int j = 0; j < SAB_HIST_ITEMS; ++j) {
            const u64 idx = base + (u64)j * SAB_HIST_THREADS + threadIdx.x;
            if (idx < n) {
                for (int p = 0; p < npass; ++p)
                    atomicAdd(&s_hist[p * SAB_RADIX_BINS + KeyTraits<KeyT>::digit(k[j], begin_bit + p * SAB_RADIX_BITS)], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < npass * SAB_RADIX_BINS; i += SAB_HIST_THREADS) {
        const u32 c = s_hist[i];
        if (c) atomicAdd((unsigned long long*)&ghist[i], (unsigned long long)c);
    }
}

// one block of 256 threads: gbase[p][d] = exclusive prefix of ghist[p][*]; skip[p] = 1 when every key
// has the same digit at place p (the pass would be the identity permutation).
__global__ void __launch_bounds__(SAB_RADIX_BINS)
radix_scan_kernel(const u64* __restrict__ ghist, u64 n, int npass, u64* __restrict__ gbase, u32* __restrict__ skip) {
    SAB_SHARED_ARRAY(u64, s_wsum, 8);
    SAB_SHARED_VAR(u32, s_full);
    const u32 d = threadIdx.x, lane = lane_id(), w = warp_id();
    for (int p = 0; p < npass; ++p) {
        if (d == 0) s_full = 0;
        __syncthreads();
        const u64 c = ghist[p * SAB_RADIX_BINS + d];
        if (c == n) s_full = 1;
        u64 incl = c;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const u64 o = __shfl_up_sync(SAB_FULL, incl, s);
            if ((int)lane >= s) incl += o;
        }
        if (lane == 31) s_wsum[w] = incl;
        __syncthreads();
        u64 woff = 0;
        for (u32 i = 0; i < w; ++i) woff += s_wsum[i];
        gbase[p * SAB_RADIX_BINS + d] = woff + incl - c;
        if (d == 0) skip[p] = s_full;
        __syncthreads();
    }
}

// Lanes of the warp holding the same 8-bit digit.  Eight ballots beat the hardware MATCH.ANY
// instruction here: profiling showed ~45 % of the pass stalled on MATCH results (profiles/r01_variants.md §2).
__device__ __forceinline__ u32 match_digit(u32 d) {
    u32 peers = SAB_FULL;
#pragma unroll
    for (int bit = 0; bit < SAB_RADIX_BITS; ++bit) {
        const bool p = (d >> bit) & 1u;
        const u32 m = __ballot_sync(SAB_FULL, p);
        peers &= p ? m : ~m;
    }
    return peers;
}

// tiles per look-back group (two-level status words); the single-level look-back over tiles measured
// slower, profiles/r01_variants.md §3b
#define SAB_LB_GROUP 8
#ifndef SAB_LB_DEPTH
#define SAB_LB_DEPTH 4
#endif

// ------------------------------------------------------------------ one onesweep pass
template <typename KeyT, bool HAS_VAL, bool IOTA_VAL, int THREADS, int ITEMS>
struct OnesweepCfg {
    static constexpr int WARPS = THREADS / 32;
    static constexpr int TILE = THREADS * ITEMS;
    static constexpr size_t KEY_BYTES = (size_t)TILE * sizeof(KeyT);
    static constexpr size_t VAL_BYTES = HAS_VAL ? (size_t)TILE * sizeof(u32) : 0;
    static constexpr size_t WHIST_BYTES = (size_t)WARPS * SAB_RADIX_BINS * sizeof(u32);
    static constexpr size_t SMEM = KEY_BYTES + VAL_BYTES + WHIST_BYTES + SAB_RADIX_BINS * sizeof(u32);
};

// Digit extractors.  The padding key of a partial tile (all ones) must map to the last bin in use.
template <typename KeyT>
struct ShiftDigit {  // radix digit: bits [shift, shift+8)
    int shift;
    __device__ __forceinline__ u32 operator()(KeyT k) const { return (u32)(k >> shift) & 0xffu; }
};
#define SAB_MAX_RANKS 16
struct SplitterDigit {  // destination rank of a key: number of splitters <= key (multi-GPU sample sort)
    u64 s[SAB_MAX_RANKS - 1];
    int np;
    __device__ __forceinline__ u32 operator()(u64 k) const {
        u32 d = 0;
        for (int i = 0; i < np; ++i) d += (s[i] <= k) ? 1u : 0u;  // np is uniform: 1 compare on 2 GPUs, 7 on 8
        return d;
    }
};
// Which GPU owns rank[q] (multi-GPU), and at which slot of its local array.
//   block  (cyc = 0): GPU g owns positions [g*B, (g+1)*B), the last GPU also the tail; slot = q - g*B
//   cyclic (cyc = 1): blocks of B = 2^shift positions are dealt round-robin: owner = (q >> shift) mod P,
//                     slot = ((q >> shift) / P) << shift | (q mod B) -- any region of the text is spread over
//                     all GPUs, so the requests of a round do not pile up on the owners of one region
struct RankLayout {
    u32 B, pmax, cyc, shift;
    __host__ __device__ __forceinline__ u32 owner(u64 q) const {
        if (cyc) return (u32)((q >> shift) % (pmax + 1u));
        const u32 o = (u32)(q / B);
        return o < pmax ? o : pmax;
    }
    __host__ __device__ __forceinline__ u64 slot(u64 q, u32 o) const {
        if (cyc) return (((q >> shift) / (pmax + 1u)) << shift) | (q & (u64)(B - 1u));
        return q - (u64)o * B;
    }
};
static inline int sab_rank_layout(u32 B, int P, int cyc_shift, RankLayout* L) {
    if (P < 1 || P > 16 || B == 0) return -1;
    L->B = B;
    L->pmax = (u32)P - 1u;
    L->cyc = cyc_shift >= 0 ? 1u : 0u;
    L->shift = cyc_shift >= 0 ? (u32)cyc_shift : 0u;
    if (L->cyc && (cyc_shift > 31 || B != (1u << cyc_shift))) return -1;
    return 0;
}
struct OwnerDigit {  // owner rank of text position key + add
    u32 add;
    RankLayout lay;
    __device__ __forceinline__ u32 operator()(u32 k) const {
        if (k == 0xffffffffu) return lay.pmax + 1u;  // dropped record / tile padding: behind the last rank
        return lay.owner((u64)k + add);
    }
};

struct SliceDigit {  // rank whose suffix-array slice [start[g], start[g+1]) holds SA position k (multi-GPU)
    u32 start[SAB_MAX_RANKS];  // start[0] is not compared: everything below start[1] belongs to rank 0
    u32 pmax;
    __device__ __forceinline__ u32 operator()(u32 k) const {
        if (k == 0xffffffffu) return pmax + 1u;  // dropped record / tile padding: behind the last rank
        u32 d = 0;
#pragma unroll
        for (int i = 1; i < SAB_MAX_RANKS; ++i) d += ((u32)i <= pmax && start[i] <= k) ? 1u : 0u;
        return d;
    }
};

// PEER passes (multi-GPU key exchange fused into the partition): bin d is written to the receive
// buffers of GPU d -- device addresses mapped into this process (symmetric memory), stores travel
// over NVLink -- at record offset gbase[d] inside them.
struct PeerOut {
    u64 k[SAB_MAX_RANKS];  // key buffer of every destination
    u64 v[SAB_MAX_RANKS];  // payload buffer of every destination
};

// vals_in may be null when IOTA_VAL (payload = iota_base + position of the record in the input).
template <typename KeyT, typename DigitOp, bool HAS_VAL, bool IOTA_VAL, bool PEER, int THREADS, int ITEMS>
__global__ void __launch_bounds__(THREADS, SAB_ONESWEEP_MIN_BLOCKS)
onesweep_kernel(const KeyT* __restrict__ keys_in, KeyT* __restrict__ keys_out, const u32* __restrict__ vals_in,
                u32* __restrict__ vals_out, u64 n, DigitOp dop, const u64* __restrict__ gbase,
                u64* __restrict__ lookback, u32* __restrict__ ticket, u32 ticket_base, u32 epoch, PeerOut po, u32 iota_base) {
    typedef OnesweepCfg<KeyT, HAS_VAL, IOTA_VAL, THREADS, ITEMS> Cfg;
    static_assert(THREADS >= SAB_RADIX_BINS && THREADS % 32 == 0, "one look-back lane per bin");
    constexpr int WARPS = Cfg::WARPS, TILE = Cfg::TILE, WTILE = 32 * ITEMS;
    SAB_DYN_SMEM(smem);
    KeyT* s_keys = (KeyT*)smem;
    u32* s_vals = (u32*)(smem + Cfg::KEY_BYTES);
    u32* s_goff = (u32*)(smem + Cfg::KEY_BYTES + Cfg::VAL_BYTES);          // [256] global record index - local start (mod 2^32)
    u32* s_whist = s_goff + SAB_RADIX_BINS;                                  // [WARPS][256]
    SAB_SHARED_VAR(u32, s_tile);
    SAB_SHARED_ARRAY(u32, s_wsum, 8);
    SAB_SHARED_ARRAY(u64, s_pk, SAB_MAX_RANKS);
    SAB_SHARED_ARRAY(u64, s_pv, SAB_MAX_RANKS);

    const u32 tid = threadIdx.x, lane = lane_id(), w = warp_id();
    if (PEER && tid < SAB_MAX_RANKS) {
        s_pk[tid] = po.k[tid];
        s_pv[tid] = po.v[tid];
    }
    if (tid == 0) s_tile = atomicAdd(ticket, 1u) - ticket_base;
    for (int i = tid; i < WARPS * SAB_RADIX_BINS; i += THREADS) s_whist[i] = 0;
    __syncthreads();
    const u32 tile = s_tile;
    const u64 tile_base = (u64)tile * TILE;
    const u64 remaining = n - tile_base;
    const u32 valid = remaining < (u64)TILE ? (u32)remaining : (u32)TILE;
    const bool full = valid == (u32)TILE;  // block-uniform: all tiles but the last take the unguarded paths

    // ---- load (warp-striped: item k of lane l is record w*WTILE + k*32 + l of the tile)
    KeyT keys[ITEMS];
    u32 vals[ITEMS];
    const u32 wofs = w * WTILE + lane;
    const KeyT* kin = keys_in + tile_base + wofs;
    const u32* vin = IOTA_VAL ? nullptr : vals_in + tile_base + wofs;
    if (full) {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) keys[k] = kin[k * 32];
        if (HAS_VAL) {
#pragma unroll
            for (int k = 0; k < ITEMS; ++k) vals[k] = IOTA_VAL ? iota_base + (u32)(tile_base + wofs + k * 32) : vin[k * 32];
        }
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) keys[k] = (wofs + k * 32 < valid) ? kin[k * 32] : KeyTraits<KeyT>::max_key();
        if (HAS_VAL) {
#pragma unroll
            for (int k = 0; k < ITEMS; ++k) {
                if (IOTA_VAL) vals[k] = iota_base + (u32)(tile_base + wofs + k * 32);
                else vals[k] = (wofs + k * 32 < valid) ? vin[k * 32] : 0u;
            }
        }
    }

    // ---- tile histogram first (plain shared-memory atomics, order irrelevant), so the tile's partial is
    // published a whole ranking phase before its successors look back: they never find it missing.
    u32* wh = s_whist + w * SAB_RADIX_BINS;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) atomicAdd(&wh[dop(keys[k])], 1u);
    __syncthreads();
    u32 my_count = 0;
    u64* lb = lookback + (u64)tile * SAB_RADIX_BINS + tid;
    const u64 etag = (u64)epoch << SAB_LB_EPOCH_SHIFT;
    const u32 grp = tile / SAB_LB_GROUP, gr = tile % SAB_LB_GROUP;
    // group status words live behind the tile status words of this launch
    u64* lb2 = lookback + ((n + (u64)TILE - 1) / (u64)TILE + grp) * SAB_RADIX_BINS + tid;
    if (tid < SAB_RADIX_BINS) {
        u32 run = 0;
#pragma unroll
        for (int ww = 0; ww < WARPS; ++ww) {
            const u32 c = s_whist[ww * SAB_RADIX_BINS + tid];
            s_whist[ww * SAB_RADIX_BINS + tid] = run;
            run += c;
        }
        my_count = run;
        // Two-level status: tile partials (never upgraded) + one word per group of SAB_LB_GROUP tiles, owned by
        // the group's last tile: PARTIAL = sum of the group's tile counts (published here, early), later
        // INCLUSIVE = prefix through the end of the group.  A look-back is then the tile's in-group
        // predecessors (one batch of independent loads) plus a walk over GROUPS, 8x shorter than over tiles.
        st_relaxed_u64(lb, etag | SAB_LB_FLAG_PARTIAL | (u64)my_count);
        if (gr == SAB_LB_GROUP - 1) {
            u64 agg = 0;
            bool ok;
            do {
                u64 v[SAB_LB_GROUP - 1];
#pragma unroll
                for (int j = 0; j < SAB_LB_GROUP - 1; ++j) v[j] = ld_relaxed_u64(lb - (u64)(j + 1) * SAB_RADIX_BINS);
                ok = true;
                agg = 0;
#pragma unroll
                for (int j = 0; j < SAB_LB_GROUP - 1; ++j) {
                    ok = ok && (v[j] >> SAB_LB_EPOCH_SHIFT) == (u64)epoch && (v[j] & SAB_LB_FLAG_MASK) != 0;
                    agg += v[j] & SAB_LB_VALUE_MASK;
                }
                if (!ok) SAB_SPIN_PAUSE();
            } while (!ok);
            st_relaxed_u64(lb2, etag | (grp == 0 ? SAB_LB_FLAG_INCLUSIVE : SAB_LB_FLAG_PARTIAL) | (agg + (u64)my_count));
        }
    }
    // block-exclusive scan of the 256 bin counts; the bin start is folded into the per-warp offsets, so
    // the ranking atomics below return final shared-memory slots
    u32 my_start = 0;
    {
        u32 incl = warp_incl_sum(my_count);
        if (tid < SAB_RADIX_BINS && lane == 31) s_wsum[w] = incl;
        __syncthreads();
        if (tid < SAB_RADIX_BINS) {
            u32 woff = 0;
            for (u32 i = 0; i < w; ++i) woff += s_wsum[i];
            my_start = woff + incl - my_count;
#pragma unroll
            for (int ww = 0; ww < WARPS; ++ww) s_whist[ww * SAB_RADIX_BINS + tid] += my_start;
        }
    }
    __syncthreads();
    // ---- rank inside the warp (stable in (k, lane) order): slot of the record in the sorted tile
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const u32 d = dop(keys[k]);
        const u32 peers = match_digit(d);
        const u32 leader = (u32)(__ffs((int)peers) - 1);
        // Atomics of one warp on one address retire in program order, so item k+1 sees item k's update.
        u32 old = 0;
        if (lane == leader) old = atomicAdd(&wh[d], (u32)__popc(peers));
        old = __shfl_sync(SAB_FULL, old, (int)leader);
        const u32 pos = old + (u32)__popc(peers & lanemask_lt());
        // staged as soon as ranked; a scatter loop after the look-back measured slower, r02_ab_radix_variants.txt _unf
        s_keys[pos] = keys[k];
        if (HAS_VAL) s_vals[pos] = vals[k];
    }
    // ---- two-level look-back, one lane per bin: in-group tile partials and the first batch of group words
    // are requested together, so the common case is a single L2 round trip
    if (tid < SAB_RADIX_BINS) {
        u64 excl = 0;
        if (tile > 0) {
            u64 v1[SAB_LB_GROUP - 1];
#pragma unroll
            for (int j = 0; j < SAB_LB_GROUP - 1; ++j)
                v1[j] = ((u32)j < gr) ? ld_relaxed_u64(lb - (u64)(j + 1) * SAB_RADIX_BINS) : 0ull;
            i64 t = (i64)grp - 1;
            bool done = grp == 0;
            const u64* g0 = lb2 - (u64)grp * SAB_RADIX_BINS;  // word of group 0, this bin
            u64 v2[SAB_LB_DEPTH];
#pragma unroll
            for (int j = 0; j < SAB_LB_DEPTH; ++j) v2[j] = (t - j >= 0) ? ld_relaxed_u64(g0 + (u64)(t - j) * SAB_RADIX_BINS) : 0ull;
            for (;;) {
                bool ok = true;
                u64 sum = 0;
#pragma unroll
                for (int j = 0; j < SAB_LB_GROUP - 1; ++j) {
                    if ((u32)j < gr) {
                        ok = ok && (v1[j] >> SAB_LB_EPOCH_SHIFT) == (u64)epoch && (v1[j] & SAB_LB_FLAG_MASK) != 0;
                        sum += v1[j] & SAB_LB_VALUE_MASK;
                    }
                }
                if (ok) {
                    excl = sum;
                    break;
                }
                SAB_SPIN_PAUSE();
#pragma unroll
                for (int j = 0; j < SAB_LB_GROUP - 1; ++j)
                    v1[j] = ((u32)j < gr) ? ld_relaxed_u64(lb - (u64)(j + 1) * SAB_RADIX_BINS) : 0ull;
            }
            while (!done) {
#pragma unroll
                for (int j = 0; j < SAB_LB_DEPTH; ++j) {
                    if (done) break;
                    const u64 f = v2[j] & SAB_LB_FLAG_MASK;
                    if ((v2[j] >> SAB_LB_EPOCH_SHIFT) != (u64)epoch || f == 0) break;  // not published yet: reload from here
                    excl += v2[j] & SAB_LB_VALUE_MASK;
                    --t;
                    if (f == SAB_LB_FLAG_INCLUSIVE) done = true;
                }
                if (!done) {
                    SAB_SPIN_PAUSE();
#pragma unroll
                    for (int j = 0; j < SAB_LB_DEPTH; ++j)
                        v2[j] = (t - j >= 0) ? ld_relaxed_u64(g0 + (u64)(t - j) * SAB_RADIX_BINS) : 0ull;
                }
            }
            if (gr == SAB_LB_GROUP - 1 && grp > 0) st_relaxed_u64(lb2, etag | SAB_LB_FLAG_INCLUSIVE | (excl + (u64)my_count));
        }
        // record indices are < 2^32 (N <= 2^32 - 1): keep the per-bin offset as a wrapping u32
        s_goff[tid] = (u32)(gbase[tid] + excl) - my_start;
    }
    __syncthreads();

    // ---- coalesced write-out: consecutive shared slots of one bin are consecutive in global memory
    if (full) {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u32 p = tid + k * THREADS;
            const KeyT key = s_keys[p];
            const u32 d = dop(key);
            const u32 dst = s_goff[d] + p;
            if (PEER) {
                ((KeyT*)(uintptr_t)s_pk[d & (SAB_MAX_RANKS - 1)])[dst] = key;
                if (HAS_VAL) ((u32*)(uintptr_t)s_pv[d & (SAB_MAX_RANKS - 1)])[dst] = s_vals[p];
            } else {
                keys_out[dst] = key;
                if (HAS_VAL) vals_out[dst] = s_vals[p];
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const u32 p = tid + k * THREADS;
            if (p < valid) {
                const KeyT key = s_keys[p];
                const u32 d = dop(key);
                const u32 dst = s_goff[d] + p;
                if (PEER) {
                    ((KeyT*)(uintptr_t)s_pk[d & (SAB_MAX_RANKS - 1)])[dst] = key;
                    if (HAS_VAL) ((u32*)(uintptr_t)s_pv[d & (SAB_MAX_RANKS - 1)])[dst] = s_vals[p];
                } else {
                    keys_out[dst] = key;
                    if (HAS_VAL) vals_out[dst] = s_vals[p];
                }
            }
        }
    }
}

__global__ void iota_kernel(u32* __restrict__ out, u64 n) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (u32)i;
}
