// sab_search.cuh -- the query side of the hot path on the GPU:
//   bucket_pairs / bucket_scan   enable_buckets            (/root/reference/src/sa.rs:89-119)
//   search_kernel                get_bucket + search_all / contains / search_lcp, batched
//                                (src/sa.rs:123-161, 164-170, 173-204, 207-253)
//   sufcheck_*                   linear-time check_integrity (src/sa.rs:72-84; SURVEY.md 8c)
//
// Each pattern is handled by a group of SAB_SEARCH_G lanes; a probe compares 4*G bytes of the
// pattern with the suffix in one step (big-endian word compare + ballot).  The work is a chain
// of dependent random reads (sa[mid], then text[sa[mid]..]): it is bound by the HBM random-
// sector rate, not by arithmetic; many groups per SM keep enough probes in flight.
#pragma once
#include "sab_context.cuh"

// 4 lanes per pattern (16 bytes per compare step): with the prefix directory a query is ~7 probes and most of them
// differ inside the first 16 bytes; 10 M patterns of 8..64 B on the 1 GiB index: 1.61 / 1.89 G queries/s against
// 1.25 / 1.47 with 8 lanes (profiles/r02_search_variants.txt)
#ifndef SAB_SEARCH_G
#define SAB_SEARCH_G 4
#endif
#define SAB_SEARCH_THREADS 256
#define SAB_PDIR_MAXD 27  // deepest prefix directory: 2^27 entries over a binary alphabet

// ------------------------------------------------------------------ enable_buckets
// Dense path: the byte pairs are counted in a shared table indexed by (code(c0), code'(c1)) of the
// bytes present in the text; sparse path (large alphabets): global atomics straight into the table.
// cnt[] has SAB200_BKT_LEN u32 slots, zeroed by the caller; slot layout as in src/sa.rs:94,103,107.
__global__ void __launch_bounds__(256)
bucket_pairs_kernel(const u8* __restrict__ text, u64 n, const u16* __restrict__ lut, u32 sigma, int dense,
                    u32* __restrict__ cnt) {
    SAB_DYN_SMEM(smem);
    u32* s_tab = (u32*)smem;  // [sigma][sigma+1]: column 0 = end-of-text, column c = code c (1..sigma)
    SAB_SHARED_ARRAY(u16, s_lut, 256);
    SAB_SHARED_ARRAY(u8, s_inv, 257);
    s_lut[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
    if (s_lut[threadIdx.x]) s_inv[s_lut[threadIdx.x]] = (u8)threadIdx.x;
    const u32 width = sigma + 1;
    const u32 tab = sigma * width;
    if (dense)
        for (u32 i = threadIdx.x; i < tab; i += blockDim.x) s_tab[i] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const u32 c0 = text[i];
        if (dense) {
            const u32 col = (i + 1 < n) ? (u32)s_lut[text[i + 1]] : 0u;
            atomicAdd(&s_tab[((u32)s_lut[c0] - 1u) * width + col], 1u);
        } else {
            const u32 slot = (i + 1 < n) ? c0 * 257u + (u32)text[i + 1] + 2u : c0 * 257u + 1u;
            atomicAdd(&cnt[slot], 1u);
        }
    }
    __syncthreads();
    if (dense)
        for (u32 i = threadIdx.x; i < tab; i += blockDim.x) {
            const u32 v = s_tab[i];
            if (v) {
                const u32 r = i / width, col = i % width;
                const u32 c0 = s_inv[r + 1];
                const u32 slot = col ? c0 * 257u + (u32)s_inv[col] + 2u : c0 * 257u + 1u;
                atomicAdd(&cnt[slot], v);
            }
        }
}

// inclusive prefix sum of the 65 793 counters (u32 wrap-around as in src/sa.rs:112-116); bkt[0] += 1
// accounts for the empty suffix (src/sa.rs:98).  One block of 1024 threads.
__global__ void __launch_bounds__(1024) bucket_scan_kernel(u32* __restrict__ bkt) {
    SAB_SHARED_ARRAY(u32, s_w, 32);
    constexpr u32 PER = (SAB200_BKT_LEN + 1023u) / 1024u;  // 65
    const u32 t = threadIdx.x, lane = lane_id(), w = warp_id();
    const u32 b0 = t * PER;
    u32 sum = 0;
    for (u32 i = 0; i < PER; ++i) {
        const u32 j = b0 + i;
        if (j < SAB200_BKT_LEN) sum += bkt[j] + (j == 0 ? 1u : 0u);
    }
    u32 incl = warp_incl_sum(sum);
    if (lane == 31) s_w[w] = incl;
    __syncthreads();
    if (w == 0) {
        u32 v = s_w[lane];
        v = warp_incl_sum(v);
        s_w[lane] = v;
    }
    __syncthreads();
    u32 run = incl - sum + (w ? s_w[w - 1] : 0u);
    for (u32 i = 0; i < PER; ++i) {
        const u32 j = b0 + i;
        if (j < SAB200_BKT_LEN) {
            run += bkt[j] + (j == 0 ? 1u : 0u);
            bkt[j] = run;
        }
    }
}

// ------------------------------------------------------------------ batched queries
// 4 bytes at byte offset `off` of `base`, first byte in the most significant position.  Reads the
// two aligned words covering them: buffers are padded by >= 8 readable bytes.
__device__ __forceinline__ u32 load_be32(const u8* __restrict__ base, u64 off) {
    const uintptr_t a = (uintptr_t)(base + off);
    const u32* w = (const u32*)(a & ~(uintptr_t)3);
    const u32 sh = (u32)(a & 3u) * 8u;
    const u32 lo = w[0];
    const u32 hi = sh ? w[1] : 0u;
    const u32 v = __funnelshift_r(lo, hi, sh);
    return __byte_perm(v, 0u, 0x0123u);
}

// Prefix directory of a resident index (built by sab200_index_create, invisible at the API): the suffixes are
// coded by their first `depth` symbols as numbers in base sigma (symbol = number of smaller byte values present in
// the text, the minimum symbol past the end of the text -- the code never decreases along the suffix array) and
// dir[c] = number of suffixes with a code < c.  search_all / contains start their bisection from
// [dir[c_lo], dir[c_hi]) of the pattern's code range instead of the whole two-byte bucket (1 GiB DNA-like text:
// 2^26 entries, ~16 suffixes each, against buckets of 2^26 suffixes); the result is the same index pair, because
// every suffix in front of the range is smaller than the pattern and every suffix behind it greater.
struct PrefixDir {
    const u32* dir;   // entries + 1 values, or null
    const u16* lut;   // byte -> (number of present byte values below it) | 0x8000 if the byte occurs in the text
    u32 sigma;        // base (>= 2)
    u32 depth;        // symbols per code
    u64 pw[SAB_PDIR_MAXD + 1];  // sigma^r
};

// code of the suffix at p (depth symbols, Horner)
__device__ __forceinline__ u64 prefix_code(const u8* __restrict__ text, u64 n, u64 p, const u16* __restrict__ lut, u32 sigma, u32 depth) {
    u64 c = 0;
    for (u32 t = 0; t < depth; ++t) c = c * sigma + ((p + t < n) ? (u64)(lut[text[p + t]] & 0x1ffu) : 0ull);
    return c;
}

// Narrows [*lo, *hi) to the directory range of the pattern's first `depth` symbols (pd.dir must be set).  The lower
// bound of the pattern lies in the narrowed range (or at its end when it is empty) whatever the pattern's length.
__device__ __forceinline__ void prefix_dir_narrow(const PrefixDir& pd, const u8* __restrict__ pat, u64 m, u64* lo, u64* hi) {
    const u32 depth = pd.depth, sigma = pd.sigma;
    u64 code = 0;
    u32 t = 0, e = 0x8000u;
    for (; t < depth && t < m; ++t) {
        e = pd.lut[pat[t]];
        if (!(e & 0x8000u)) break;
        code = code * sigma + (e & 0x1ffu);
    }
    u64 clo, chi;
    if (e & 0x8000u) {  // t symbols of the pattern, all present in the text: every code that starts with them
        clo = code * pd.pw[depth - t];
        chi = clo + pd.pw[depth - t];
    } else {
        // byte t of the pattern does not occur in the text: the pattern falls between two neighbouring codes --
        // unless it is smaller than every symbol, where it still follows the suffixes that END after the t
        // symbols (they are padded with the minimum symbol and share the first code of the prefix)
        clo = (code * sigma + (e & 0x1ffu)) * pd.pw[depth - t - 1];
        chi = clo + ((e & 0x1ffu) == 0 ? 1u : 0u);
    }
    const u64 dlo = pd.dir[clo], dhi = pd.dir[chi];
    if (dlo > *lo) *lo = dlo;
    if (dhi < *hi) *hi = dhi;
    if (*hi < *lo) *hi = *lo;
}

__global__ void __launch_bounds__(256) fill_u32_kernel(u32* __restrict__ out, u64 count, u32 value) {
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) out[i] = value;
}

// dir[c] = j for every code c in (code(sa[j-1]), code(sa[j])]; the caller pre-fills dir with len (codes behind the
// last suffix).  Short runs are written by their thread, long ones (codes no suffix has) by the whole warp.
__global__ void __launch_bounds__(256)
prefix_dir_kernel(const u8* __restrict__ text, u64 n, const u32* __restrict__ sa, u64 len, const u16* __restrict__ lut, u32 sigma,
                  u32 depth, u32* __restrict__ dir) {
    SAB_SHARED_ARRAY(u16, s_lut, 256);
    s_lut[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u32 lane = lane_id();
    u64 c = 0, first = 0, run = 0;
    if (j < len) {
        const u64 p = sa[j];
        c = prefix_code(text, n, p <= n ? p : n, s_lut, sigma, depth);
    }
    u64 cp = __shfl_up_sync(SAB_FULL, c, 1);
    if (lane == 0 && j > 0 && j < len) {
        const u64 p = sa[j - 1];
        cp = prefix_code(text, n, p <= n ? p : n, s_lut, sigma, depth);
    }
    if (j < len) {
        first = j == 0 ? 0 : cp + 1;       // a corrupt array (codes not ascending) writes nothing out of order
        run = c + 1 > first ? c + 1 - first : 0;
    }
    if (run <= 8)
        for (u64 t = 0; t < run; ++t) dir[first + t] = (u32)j;
    u32 todo = __ballot_sync(SAB_FULL, run > 8);
    while (todo) {
        const int src = __ffs((int)todo) - 1;
        todo &= todo - 1;
        const u64 f = __shfl_sync(SAB_FULL, first, src), r = __shfl_sync(SAB_FULL, run, src);
        const u32 v = (u32)(j - lane + (u64)src);
        for (u64 t = lane; t < r; t += 32) dir[f + t] = v;
    }
}

struct SearchArgs {
    PrefixDir pd;
    unsigned long long* probes;  // cumulative number of probes (suffix comparisons), or null
    const u8* text;   // n bytes (+ padding)
    u64 n;
    const u32* sa;    // n + 1
    const u32* bkt;   // SAB200_BKT_LEN or null
    const u8* pats;   // concatenated patterns (+ padding)
    const u64* offs;  // np + 1
    u64 np;
    u32* out0;        // search_all: lo   | search_lcp: start | contains: (u8*) flags
    u32* out1;        // search_all: hi   | search_lcp: end
};

// Compares pattern (pat, m) with the suffix at p.  Returns d = length of their common prefix
// (<= L = min(m, n - p)); *less_at = 1 when d < L and text[p+d] < pat[d].
template <int G>
__device__ __forceinline__ u64 group_compare(const SearchArgs& a, const u8* __restrict__ pat, u64 m, u64 p, u32 gmask,
                                             u32 gl, u32 gbase, u32 pw0, u32 pw1, u32* less_at) {
    const u64 avail = p <= a.n ? a.n - p : 0;  // an entry beyond n (corrupt array) reads as the empty suffix
    const u64 L = m < avail ? m : avail;
    *less_at = 0;
    for (u64 c0 = 0; c0 < L || c0 == 0; c0 += 4 * G) {
        const u64 o = c0 + 4u * gl;
        u32 neq = 0, tw = 0, pw = 0;
        if (o < L) {
            const u64 rem = L - o;
            const u32 mask = rem >= 4 ? 0xffffffffu : (0xffffffffu << (8u * (4u - (u32)rem)));
            tw = load_be32(a.text, p + o) & mask;
            pw = (c0 == 0 ? pw0 : (c0 == 4 * G ? pw1 : load_be32(pat, o))) & mask;
            neq = tw ^ pw;
        }
        const u32 bal = (__ballot_sync(gmask, neq != 0) >> gbase) & ((G == 32) ? 0xffffffffu : ((1u << G) - 1u));
        if (bal) {
            const int first = __ffs((int)bal) - 1;
            const u32 fneq = __shfl_sync(gmask, neq, (int)gbase + first);
            const u32 fless = __shfl_sync(gmask, (u32)(tw < pw), (int)gbase + first);
            *less_at = fless;
            return c0 + 4u * (u32)first + (u32)(__clz((int)fneq) >> 3);
        }
        if (L == 0) break;
    }
    return L;
}

// MODE 0: search_all -> [lo, hi) global SA indices;  1: contains -> u8;  2: search_lcp -> [start, end)
template <int G, int MODE>
__global__ void __launch_bounds__(SAB_SEARCH_THREADS) search_kernel(SearchArgs a) {
    const u64 gtid = (u64)blockIdx.x * SAB_SEARCH_THREADS + threadIdx.x;
    const u64 q = gtid / G;
    if (q >= a.np) return;
    const u32 lane = lane_id();
    const u32 gl = lane % G, gbase = lane - gl;
    const u32 gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << gbase);
    const u64 pbeg = a.offs[q];
    const u64 m = a.offs[q + 1] - pbeg;
    const u8* pat = a.pats + pbeg;
    const u64 n = a.n;
    // pattern words of the first two probe chunks stay in registers
    const u32 pw0 = (4u * gl < m) ? load_be32(pat, 4u * gl) : 0u;
    const u32 pw1 = (4u * G + 4u * gl < m) ? load_be32(pat, 4u * G + 4u * gl) : 0u;

    // get_bucket (src/sa.rs:123-144); MODE 0 with an empty pattern searches the whole array (:175-179)
    u64 lo = 0, hi = n + 1;
    if (a.bkt) {
        if (m > 1) {
            const u32 idx = (u32)pat[0] * 257u + (u32)pat[1] + 2u;
            lo = a.bkt[idx - 1];
            hi = a.bkt[idx];
        } else if (m == 1) {
            const u32 st = (u32)pat[0] * 257u;
            lo = a.bkt[st];
            hi = a.bkt[st + 257];
        } else if (MODE != 0) {
            lo = 0;
            hi = 1;
        }
    }
    if (MODE == 2 && hi == lo) {  // src/sa.rs:211-222 (only reachable with buckets and m > 0)
        const u32 st = (u32)pat[0] * 257u;
        const u64 tl = a.bkt[st], th = a.bkt[st + 257];
        if (gl == 0) {
            if (th > tl) {
                const u32 i = a.sa[tl];
                a.out0[q] = i;
                a.out1[q] = i + 1u;
            } else {
                a.out0[q] = (u32)n;
                a.out1[q] = (u32)n;
            }
        }
        return;
    }
    // narrow [lo, hi) to the suffixes that share the pattern's first symbols (search_lcp keeps the reference's
    // range: its answer depends on the borders of the two-byte bucket, src/sa.rs:224-252)
    if (MODE != 2 && a.pd.dir) prefix_dir_narrow(a.pd, pat, m, &lo, &hi);
    u32 nprobe = 0;
    // lower bound: first index whose suffix is not < pat   (src/sa.rs:181-190)
    u64 i = lo, k = hi;
    while (i < k) {
        ++nprobe;
        const u64 mid = i + (k - i) / 2;
        const u64 p = a.sa[mid];
        u32 less_at;
        const u64 d = group_compare<G>(a, pat, m, p, gmask, gl, gbase, pw0, pw1, &less_at);
        const u64 avail = p <= n ? n - p : 0;
        const u64 L = m < avail ? m : avail;
        const bool suffix_less = (d < L) ? (less_at != 0) : (avail < m);
        if (suffix_less) i = mid + 1;
        else k = mid;
    }
    if (MODE == 0) {
        // upper bound: first index >= i whose suffix does not start with pat   (src/sa.rs:192-201).
        // The reference bisects [i, hi); the matches are a contiguous run starting at i and usually a short one,
        // so the same index is found by galloping from i (1, 2, 4, ... while the probe still matches) and
        // bisecting the last gap: ~2 log2(run) + 1 probes instead of log2(bucket).
        u64 j = i;
        k = hi;
        for (u64 step = 1; j < k; step <<= 1) {
            const u64 t = (k - j > step) ? j + step - 1 : k - 1;
            u32 less_at;
            ++nprobe;
            const u64 d = group_compare<G>(a, pat, m, a.sa[t], gmask, gl, gbase, pw0, pw1, &less_at);
            if (d == m) {
                j = t + 1;
            } else {
                k = t;
                break;
            }
        }
        while (j < k) {
            const u64 mid = j + (k - j) / 2;
            const u64 p = a.sa[mid];
            u32 less_at;
            ++nprobe;
            const u64 d = group_compare<G>(a, pat, m, p, gmask, gl, gbase, pw0, pw1, &less_at);
            if (d == m) j = mid + 1;
            else k = mid;
        }
        if (gl == 0) {
            a.out0[q] = (u32)i;
            a.out1[q] = (u32)j;
            if (a.probes) atomicAdd(a.probes, (unsigned long long)nprobe);
        }
    } else if (MODE == 1) {
        // src/sa.rs:168-169: a suffix whose truncation equals pat exists iff the lower bound starts with pat
        bool found = false;
        if (i < hi) {
            u32 less_at;
            found = group_compare<G>(a, pat, m, a.sa[i], gmask, gl, gbase, pw0, pw1, &less_at) == m;
        }
        if (gl == 0) ((u8*)a.out0)[q] = found ? 1 : 0;
    } else {
        // src/sa.rs:224-252
        u32 less_at;
        u64 st = 0, en = 0;
        u64 pb = 0, db = 0;
        if (i < hi) {
            pb = a.sa[i];
            db = group_compare<G>(a, pat, m, pb, gmask, gl, gbase, pw0, pw1, &less_at);
        }
        if (i < hi && db == m && pb <= n && n - pb == m) {  // Ok(i): a suffix equal to the pattern
            st = pb;
            en = n;
        } else if (i > lo && i < hi) {
            const u64 pa = a.sa[i - 1];
            const u64 da = group_compare<G>(a, pat, m, pa, gmask, gl, gbase, pw0, pw1, &less_at);
            if (da > db) {
                st = pa;
                en = pa + da;
            } else {
                st = pb;
                en = pb + db;
            }
        } else if (i == lo) {
            st = pb;
            en = pb + db;
        } else {
            const u64 pa = a.sa[i - 1];
            const u64 da = group_compare<G>(a, pat, m, pa, gmask, gl, gbase, pw0, pw1, &less_at);
            st = pa;
            en = pa + da;
        }
        if (gl == 0) {
            a.out0[q] = (u32)st;
            a.out1[q] = (u32)en;
        }
    }
}

// ------------------------------------------------------------------ LCP array (Kasai in chunks)
#define SAB_LCP_CHUNK 32
__global__ void __launch_bounds__(256) lcp_isa_kernel(const u32* __restrict__ sa, u64 len, u32* __restrict__ isa) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < len) isa[sa[j]] = (u32)j;
}
// common prefix of the suffixes at a and b (a != b), known to be at least h: 8 bytes per step while both have them
__device__ __forceinline__ u64 lcp_extend(const u8* __restrict__ s, u64 n, u64 a, u64 b, u64 h) {
    while (a + h + 8 <= n && b + h + 8 <= n) {
        u64 x = 0, y = 0;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            x |= (u64)s[a + h + t] << (8 * t);
            y |= (u64)s[b + h + t] << (8 * t);
        }
        const u64 d = x ^ y;
        if (d) return h + (u64)((__ffsll((long long)d) - 1) >> 3);
        h += 8;
    }
    while (a + h < n && b + h < n && s[a + h] == s[b + h]) ++h;
    return h;
}
// thread t owns text positions [t*CHUNK, (t+1)*CHUNK): lcp[isa[i]] = common prefix of suffix i and its
// predecessor in suffix order, each length starting from the previous one minus one
__global__ void __launch_bounds__(256)
lcp_kasai_kernel(const u8* __restrict__ s, u64 n, const u32* __restrict__ sa, const u32* __restrict__ isa, u32* __restrict__ lcp) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 i0 = t * SAB_LCP_CHUNK;
    if (t == 0) lcp[0] = 0;
    u64 h = 0;
    for (u64 i = i0; i < i0 + SAB_LCP_CHUNK && i < n; ++i) {
        const u32 j = isa[i];
        const u64 p = sa[j - 1];
        h = lcp_extend(s, n, i, p, h);
        lcp[j] = (u32)h;
        if (h) --h;
    }
}
static int sab_launch_kasai(SabContext* c, const u8* d_s, u64 n, const u32* d_sa, const u32* d_isa, u32* d_lcp) {
    const u64 chunks = div_up64(n ? n : 1, SAB_LCP_CHUNK);
    SAB_LAUNCH(lcp_kasai_kernel, (unsigned)div_up64(chunks, 256), 256, 0, c->stream, d_s, n, d_sa, d_isa, d_lcp);
    SAB_LAUNCH_CHECK();
    return SAB_OK;
}

// ------------------------------------------------------------------ linear-time integrity check
// flags[0] != 0 -> not a suffix array.  isa must be pre-filled with 0xFFFFFFFF.
__global__ void __launch_bounds__(256)
sufcheck_scatter_kernel(const u32* __restrict__ sa, u64 len, u64 n, u32* __restrict__ isa, u32* __restrict__ flags) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= len) return;
    const u32 v = sa[j];
    if ((u64)v > n || (j == 0 && (u64)v != n)) {
        flags[0] = 1;
        return;
    }
    isa[v] = (u32)j;
}

__global__ void __launch_bounds__(256)
sufcheck_order_kernel(const u8* __restrict__ text, const u32* __restrict__ sa, u64 len, u64 n,
                      const u32* __restrict__ isa, u32* __restrict__ flags) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= len) return;
    const u32 b = sa[j];
    if ((u64)b > n) return;  // already flagged
    if (isa[b] != (u32)j) {  // duplicate entry somewhere -> not a permutation
        flags[0] = 1;
        return;
    }
    if (j < 2) return;  // sa[0] = n was checked; sa[1] follows the empty suffix
    const u32 x = sa[j - 1];
    if ((u64)x >= n || (u64)b >= n) {
        flags[0] = 1;  // the empty suffix anywhere but in front
        return;
    }
    const u8 cx = text[x], cb = text[b];
    if (cx > cb || (cx == cb && isa[x + 1] >= isa[b + 1])) flags[0] = 1;
}

// *bad = 0 when d_sa (sa_len entries) is the suffix array of the text; d_isa (n + 2 words) then holds its inverse.
// Waits for c->stream.
static int sab_isa_check(SabContext* c, const u8* d_s, u64 n, const u32* d_sa, u64 sa_len, u32* d_isa, u32* bad) {
    cudaStream_t st = c->stream;
    u32* flag = &c->scratch->check_flag;
    SAB_CUDA_TRY(cudaMemsetAsync(d_isa, 0xff, ((size_t)n + 2) * sizeof(u32), st));
    SAB_CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(u32), st));
    const unsigned blocks = (unsigned)div_up64(sa_len, 256);
    SAB_LAUNCH(sufcheck_scatter_kernel, blocks, 256, 0, st, d_sa, sa_len, n, d_isa, flag);
    SAB_LAUNCH_CHECK();
    SAB_LAUNCH(sufcheck_order_kernel, blocks, 256, 0, st, d_s, d_sa, sa_len, n, (const u32*)d_isa, flag);
    SAB_LAUNCH_CHECK();
    return sab_read_u32(c, flag, 1, bad);
}
