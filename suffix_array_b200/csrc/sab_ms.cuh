// sab_ms.cuh -- matching statistics of batched queries against a resident index (include/sab200.h):
//   lcp_block_min_kernel   one level of the block-minimum hierarchy over the LCP array (index extension)
//   ms_offs_check_kernel   flags decreasing query offsets (device entry point)
//   ms_kernel              one warp walks SAB_MS_CHUNK consecutive query positions
//
// For position i of a query Q (m bytes), len[i] is the longest prefix of Q[i..] that occurs in the text and [lo, hi)
// the suffix-array range of the suffixes that start with it.  A warp carries (len, t) along its chunk, where
// Q[i .. i+len) = s[t .. t+len).  At i+1 the first b0 = len-1 bytes are known to occur at t+1, so every suffix that
// can extend the match lies in the LCP interval of length b0 around isa[t+1]: the bisection for Q[i+1..] runs inside
// it and compares from byte b0.  The intervals come from the LCP array and its block minima (fan-out 256): a scan of
// the block that holds the rank, a climb until a block minimum falls below the length, a descent into that block --
// at most 2 x 256 entries per level, 32 per warp read, whatever the interval's size.
//
// Work bound (not measured): by Kasai's telescoping, sum over a chunk of (len[i+1] - len[i] + 1) is at most
// C + (longest match in the chunk), and that sum bounds the bytes the carried steps compare beyond their known b0
// (times log2 |J| probes of the bisection, of which the min(lcp_lo, lcp_hi) skip leaves O(log |J|) probes per
// position that compare no new bytes).  A query that lies inside the text is therefore linear in its length per
// chunk, plus one from-scratch search per chunk whose compare is as long as the match at the chunk's first position:
// m^2 / (2C) bytes in all for a query that occurs whole, which is why C is large.
#pragma once
#include "sab_search.cuh"

#define SAB_MS_CHUNK 1024       // positions per warp
#define SAB_MS_THREADS 256
#define SAB_MS_LEVELS 4         // the LCP array and up to three levels of block minima (n + 1 <= 2^32 entries)

// one warp per block of 256 entries: out[w] = min(in[256 w .. 256 w + 255])
__global__ void __launch_bounds__(256) lcp_block_min_kernel(const u32* __restrict__ in, u64 count, u32* __restrict__ out, u64 out_count) {
    const u64 w = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= out_count) return;  // whole warps
    const u32 lane = lane_id();
    u32 v = 0xffffffffu;
    for (u32 t = 0; t < 8; ++t) {
        const u64 j = w * 256 + t * 32 + lane;
        const u32 x = j < count ? in[j] : 0xffffffffu;
        v = x < v ? x : v;
    }
    for (int o = 16; o; o >>= 1) {
        const u32 x = __shfl_xor_sync(SAB_FULL, v, o);
        v = x < v ? x : v;
    }
    if (lane == 0) out[w] = v;
}

__global__ void __launch_bounds__(256) ms_offs_check_kernel(const u64* __restrict__ offs, u64 nq, u32* __restrict__ flag) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < nq && offs[q + 1] < offs[q]) flag[0] = 1;
}

struct MsArgs {
    SearchArgs s;             // text, n, sa, prefix directory; queries at absolute offsets (pats, offs, np = queries)
    const u32* isa;           // n + 1
    const u32* lvl[SAB_MS_LEVELS];  // lvl[0] = LCP array (n + 1), lvl[k] = minima of the blocks of 256 of lvl[k-1]
    u64 cnt[SAB_MS_LEVELS];   // entries of each level
    u32 top;                  // last level: cnt[top] <= 256
    u32 fresh_below;          // T >= 1: a carried length minus one below T takes a from-scratch search
    u64 p0, p1;               // absolute query positions of this launch; p0 starts a chunk
    u32 *len, *lo, *hi;       // indexed by absolute position
};

#define SAB_MS_NONE (~0ull)

// last j in [lo, hi] with v[j] < l (SAB_MS_NONE if none); hi >= lo
__device__ __forceinline__ u64 ms_last_below(const u32* __restrict__ v, u64 lo, u64 hi, u64 l, u32 lane) {
    for (u64 top = hi + 1;;) {
        const u64 span = top - lo;
        const bool ok = lane < span && (u64)v[top - 1 - lane] < l;
        const u32 bal = __ballot_sync(SAB_FULL, ok);
        if (bal) return top - (u64)__ffs((int)bal);
        if (span <= 32) return SAB_MS_NONE;
        top -= 32;
    }
}

// first j in [lo, hi] with v[j] < l (SAB_MS_NONE if none); hi >= lo
__device__ __forceinline__ u64 ms_first_below(const u32* __restrict__ v, u64 lo, u64 hi, u64 l, u32 lane) {
    for (u64 b = lo;; b += 32) {
        const bool ok = b + lane <= hi && (u64)v[b + lane] < l;
        const u32 bal = __ballot_sync(SAB_FULL, ok);
        if (bal) return b + (u64)(__ffs((int)bal) - 1);
        if (hi - b < 32) return SAB_MS_NONE;
    }
}

// LCP interval [a, b) of length l >= 1 around rank r (the suffix at r has at least l bytes): a = largest j <= r with
// lcp[j] < l (lcp[0] = 0, so it exists), b = smallest j > r with lcp[j] < l, or n + 1.
// Levels: any type with the lvl / cnt / top members of MsArgs, a block-minimum hierarchy over lvl[0].  Over another
// array ms_left returns 0 when no entry of [0, r] is below l.
template <typename Levels>
__device__ __forceinline__ u64 ms_left(const Levels& a, u64 r, u64 l, u32 lane) {
    u64 j = ms_last_below(a.lvl[0], r & ~255ull, r, l, lane);
    if (j != SAB_MS_NONE) return j;
    u32 k = 1;
    for (u64 e = r >> 8; k <= a.top; ++k, e >>= 8) {  // e: the block of level k-1 that holds r, an entry of level k
        if ((e & 255) && (j = ms_last_below(a.lvl[k], e & ~255ull, e - 1, l, lane)) != SAB_MS_NONE) break;
    }
    if (k > a.top) return 0;  // not reached: lcp[0] = 0
    for (; k > 0; --k) {
        const u64 s = j << 8, e = s + 255 < a.cnt[k - 1] ? s + 255 : a.cnt[k - 1] - 1;
        j = ms_last_below(a.lvl[k - 1], s, e, l, lane);
    }
    return j;
}

template <typename Levels>
__device__ __forceinline__ u64 ms_right(const Levels& a, u64 r, u64 l, u32 lane) {
    const u64 end0 = (r | 255) < a.cnt[0] ? (r | 255) : a.cnt[0] - 1;
    u64 j = r < end0 ? ms_first_below(a.lvl[0], r + 1, end0, l, lane) : SAB_MS_NONE;
    if (j != SAB_MS_NONE) return j;
    u32 k = 1;
    for (u64 e = r >> 8; k <= a.top; ++k, e >>= 8) {
        const u64 end = (e | 255) < a.cnt[k] ? (e | 255) : a.cnt[k] - 1;
        if (e < end && (j = ms_first_below(a.lvl[k], e + 1, end, l, lane)) != SAB_MS_NONE) break;
    }
    if (k > a.top) return a.cnt[0];  // no suffix behind r shares fewer than l bytes: the interval runs to the end
    for (; k > 0; --k) {
        const u64 s = j << 8, e = s + 255 < a.cnt[k - 1] ? s + 255 : a.cnt[k - 1] - 1;
        j = ms_first_below(a.lvl[k - 1], s, e, l, lane);
    }
    return j;
}

// common prefix of P (m bytes) and the suffix at p, known to be at least h; *less_at as in group_compare
__device__ __forceinline__ u64 ms_compare(const SearchArgs& a, const u8* P, u64 m, u64 p, u64 h, u32 lane, u32* less_at) {
    const u8* ph = P + h;
    const u64 mh = m - h;
    const u32 pw0 = (4u * lane < mh) ? load_be32(ph, 4u * lane) : 0u;
    const u32 pw1 = (128u + 4u * lane < mh) ? load_be32(ph, 128u + 4u * lane) : 0u;
    return h + group_compare<32>(a, ph, mh, p + h, SAB_FULL, lane, 0, pw0, pw1, less_at);
}

// Lower bound of P in [lo, hi), where every suffix of the range shares at least h0 bytes with P, then the longer
// common prefix with the two neighbours of the insertion point (*len) and that neighbour's rank (*rank).  A neighbour
// outside [lo, hi) is compared from scratch when `outside` is set; otherwise it cannot be the longer one.
__device__ __forceinline__ void ms_locate(const MsArgs& a, const u8* P, u64 m, u64 lo, u64 hi, u64 h0, bool outside, u32 lane,
                                          u64* len, u64* rank) {
    const u64 n = a.s.n;
    u64 i = lo, k = hi, li = h0, lk = h0;
    bool li_known = false, lk_known = false;
    while (i < k) {
        const u64 mid = i + (k - i) / 2;
        const u64 p = a.s.sa[mid];
        u32 less_at;
        const u64 d = ms_compare(a.s, P, m, p, li < lk ? li : lk, lane, &less_at);
        const u64 avail = n - p;
        const u64 L = m < avail ? m : avail;
        if ((d < L) ? (less_at != 0) : (avail < m)) {
            i = mid + 1;
            li = d;
            li_known = true;
        } else {
            k = mid;
            lk = d;
            lk_known = true;
        }
    }
    u32 less_at;
    u64 dl = 0, dr = 0;
    if (i > 0) dl = li_known ? li : (outside ? ms_compare(a.s, P, m, a.s.sa[i - 1], 0, lane, &less_at) : 0);
    if (i <= n) dr = lk_known ? lk : (outside ? ms_compare(a.s, P, m, a.s.sa[i], 0, lane, &less_at) : 0);
    if (i <= n && dr >= dl) {
        *len = dr;
        *rank = i;
    } else {
        *len = dl;
        *rank = i - 1;
    }
}

__global__ void __launch_bounds__(SAB_MS_THREADS) ms_kernel(MsArgs a) {
    const u64 w = ((u64)blockIdx.x * SAB_MS_THREADS + threadIdx.x) >> 5;
    const u64 c0 = a.p0 + w * SAB_MS_CHUNK;
    if (c0 >= a.p1) return;  // whole warps
    const u64 c1 = c0 + SAB_MS_CHUNK < a.p1 ? c0 + SAB_MS_CHUNK : a.p1;
    const u32 lane = lane_id();
    const u64 n = a.s.n;
    const u64* offs = a.s.offs;
    // the query that holds c0: the last q with offs[q] <= c0
    u64 q = 0, qh = a.s.np;
    while (qh - q > 1) {
        const u64 mid = q + (qh - q) / 2;
        if (offs[mid] <= c0) q = mid;
        else qh = mid;
    }
    u64 qend = offs[q + 1];
    u64 len = 0, t = 0;  // Q[i-1 .. i-1+len) = s[t .. t+len) of the previous position (len = 0: none to carry)
    for (u64 i = c0; i < c1; ++i) {
        if (i >= qend) {  // a new query starts: nothing carries over (empty queries are skipped)
            while (qend <= i && q + 1 < a.s.np) qend = offs[++q + 1];
            len = 0;
        }
        const u8* P = a.s.pats + i;
        const u64 m = qend - i;
        u64 nlen, rank, olo, ohi;
        if (len >= (u64)a.fresh_below + 1) {
            // carried step: Q[i .. i+b0) = s[t+1 .. t+1+b0)
            const u64 b0 = len - 1;
            const u64 r = a.isa[t + 1];
            const u64 ja = ms_left(a, r, b0, lane), jb = ms_right(a, r, b0, lane);
            if (b0 == m) {  // the match reaches the end of the query
                nlen = b0;
                rank = r;
            } else {
                ms_locate(a, P, m, ja, jb, b0, false, lane, &nlen, &rank);
            }
            if (nlen == b0) {
                olo = ja;
                ohi = jb;
            } else {
                olo = ms_left(a, rank, nlen, lane);
                ohi = ms_right(a, rank, nlen, lane);
            }
        } else {
            u64 lo = 0, hi = n + 1;
            if (a.s.pd.dir) prefix_dir_narrow(a.s.pd, P, m, &lo, &hi);
            ms_locate(a, P, m, lo, hi, 0, true, lane, &nlen, &rank);
            if (nlen) {
                olo = ms_left(a, rank, nlen, lane);
                ohi = ms_right(a, rank, nlen, lane);
            } else {
                olo = 0;
                ohi = n + 1;
            }
        }
        len = nlen;
        if (nlen) t = a.s.sa[rank];
        if (lane == 0) {
            a.len[i] = (u32)nlen;
            a.lo[i] = (u32)olo;
            a.hi[i] = (u32)ohi;
        }
    }
}
