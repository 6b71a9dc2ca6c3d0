// sab_saca.cuh -- suffix-array construction by GPU prefix doubling.  Replaces the body of
// saca() (/root/reference/src/saca.rs:9-15), i.e. `sa[0] = n; divsufsort(s, sa[1..])`.
//
//   1. alphabet_hist        256-bin byte histogram -> sigma, code LUT (codes 1..sigma; 0 = past the end),
//                           collision entropy H2 -> how many symbols the initial key needs
//   2. pack_keys            key[i] = first k codes of suffix i as a mixed-radix number in base sigma+1
//                           (most significant first).  Code 0 past the end makes a proper prefix sort first and keeps real
//                           0x00 bytes distinct from padding (SURVEY.md H1).  k = whole radix passes chosen by a
//                           cost model (passes vs expected ties from the collision entropy H2), <= 64 bits.
//   3. radix sort (key, i)  sab_sort.cuh
//   4. init_ranks           head flags -> rank = SA position of the first suffix of the group;
//                           sa[pos] = i; groups of size > 1 are compacted into the active list and
//                           only THEIR ranks are scattered; a bucket directory over the sorted keys is
//                           built on the fly (lazy inverse suffix array, see 4b)
//   5. rounds, h = k, 2k, 4k, ...   gather r2 = rank[i+h]; sort active by (r1, r2); re-rank with a
//                           chained scan; settled (singleton) suffixes are written to sa[] and dropped.
//
// Invariants (SURVEY.md 7.2b): after a round at depth h two suffixes share a rank iff their first h
// symbols agree; rank = SA position of the group head, so a singleton's rank is its final position;
// rank[n] = 0 (empty suffix); every active i has i + h <= n.
#pragma once
#include <math.h>

#include "sab_context.cuh"
#include "sab_sort.cuh"
#include "sab_scan_kernels.cuh"
#include "sab_group_sort.cuh"

// The bucket directory of the lazy inverse suffix array has 2^(ceil(log2 n) - SAB_DIR_SHIFT) entries (at most
// 2^28): ~2^SAB_DIR_SHIFT sorted keys per entry for the gallop + bisect that follows the jump.  Measured on the
// 1 GiB DNA-like text (profiles/r02_ab_round2.txt): shift 4 -> 2 takes the gathers from 6.9 to 6.2 ms.
#ifndef SAB_DIR_SHIFT
#define SAB_DIR_SHIFT 2
#endif

#define SAB_RANK_EMPTY 0xffffffffu
#define SAB_PAD(o) ((o) + ((o) >> 5))  // shared-memory padding, one word per 32; NB: evaluates its argument twice
#ifdef SAB_EMU
#ifndef SAB_FILTER_MIN
#define SAB_FILTER_MIN ((u64)3000)
#endif
#else
#define SAB_FILTER_MIN ((u64)1 << 20)
#endif
#ifndef SAB_ACTIVE_COST
#ifdef SAB_EMU
#define SAB_ACTIVE_COST 30.0  // emulator runs are tiny: keep the doubling rounds exercised
#else
#define SAB_ACTIVE_COST 300.0
#endif
#endif

// ------------------------------------------------------------------ 1. alphabet
__global__ void __launch_bounds__(256) alphabet_hist_kernel(const u8* __restrict__ text, u64 n, u32* __restrict__ hist) {
    SAB_SHARED_ARRAY(u32, s_h, 256);
    s_h[threadIdx.x] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * blockDim.x;
    const u64 gtid = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 head = (16 - ((u64)(uintptr_t)text & 15)) & 15;  // bytes before the first 16-byte boundary
    if (head > n) head = n;
    for (u64 i = gtid; i < head; i += stride) atomicAdd(&s_h[text[i]], 1u);
    const u64 nvec = (n - head) / 16;
    const uint4* tv = (const uint4*)(text + head);
    for (u64 i = gtid; i < nvec; i += stride) {
        const uint4 v = tv[i];
        const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            atomicAdd(&s_h[w[j] & 0xff], 1u);
            atomicAdd(&s_h[(w[j] >> 8) & 0xff], 1u);
            atomicAdd(&s_h[(w[j] >> 16) & 0xff], 1u);
            atomicAdd(&s_h[w[j] >> 24], 1u);
        }
    }
    for (u64 i = head + nvec * 16 + gtid; i < n; i += stride) atomicAdd(&s_h[text[i]], 1u);
    __syncthreads();
    const u32 c = s_h[threadIdx.x];
    if (c) atomicAdd(&hist[threadIdx.x], c);
}

// blocks for n items of per_block each, at most `waves` blocks per SM (grid-stride kernels), at least 1
static inline unsigned sab_grid(SabContext* c, u64 n, u64 per_block, int waves) {
    u64 g = div_up64(n, per_block);
    const u64 gmax = (u64)c->sm_count * (u64)waves;
    if (g > gmax) g = gmax;
    return (unsigned)(g ? g : 1);
}

// byte histogram of text[0..n) into the 256 words at d_hist (zeroed first)
static int sab_launch_alphabet_hist(SabContext* c, const u8* d_text, u64 n, u32* d_hist) {
    SAB_CUDA_TRY(cudaMemsetAsync(d_hist, 0, 256 * sizeof(u32), c->stream));
    if (n == 0) return SAB_OK;
    SAB_LAUNCH(alphabet_hist_kernel, sab_grid(c, n, 256 * 64, 8), 256, 0, c->stream, d_text, n, d_hist);
    SAB_LAUNCH_CHECK();
    c->stats.kernel_launches++;
    return SAB_OK;
}

static inline u64 sab_pow_u64(u64 b, int e) {
    u64 r = 1;
    for (int i = 0; i < e; ++i) r *= b;
    return r;
}

// ------------------------------------------------------------------ 2. packed initial keys
#define SAB_PACK_THREADS 256
#define SAB_PACK_ITEMS 8
#define SAB_PACK_TILE (SAB_PACK_THREADS * SAB_PACK_ITEMS)

// key of the suffix starting at i: k codes, MSB first, code 0 beyond the end of the text
__device__ __forceinline__ u64 pack_key_at(const u8* __restrict__ text, u64 n, const u16* __restrict__ lut, u32 base, int k,
                                           u64 i) {
    u64 key = 0;
    for (int t = 0; t < k; ++t) {
        const u64 p = i + (u64)t;
        key = key * base + (u64)(p < n ? lut[text[p]] : (u16)0);
    }
    return key;
}

// lut[c] = code of byte c (1..sigma); key = sum code_t * radix^(k-1-t), radix = sigma + 1, top = radix^(k-1).
// Keys are produced for positions [0, count); positions >= n are past the end of the text (count < n
// when the buffer is a shard + halo).  Each thread owns SAB_PACK_ITEMS consecutive positions: the first
// key costs k multiply-adds, each next one slides the window (drop the leading symbol, append one);
// the keys leave through shared memory so that global stores are coalesced.
struct PackPow {
    u64 p[64];  // p[t] = radix^(k-1-t): weight of symbol t of a key
};
static inline PackPow sab_pack_pow(u32 radix, int k) {
    PackPow w;
    memset(&w, 0, sizeof(w));
    u64 v = 1;
    for (int t = k - 1; t >= 0; --t) {
        w.p[t] = v;
        v *= radix;
    }
    return w;
}
__global__ void __launch_bounds__(SAB_PACK_THREADS)
pack_keys_kernel(const u8* __restrict__ text, u64 n, u64 count, const u16* __restrict__ lut, u32 radix, int k, PackPow pw,
                 u64* __restrict__ keys) {
    // one code per 32-bit word, one pad word per 32: a thread reads its window at a stride of SAB_PACK_ITEMS words
    // from its neighbour's, which a packed u16 array serves with 4-way bank conflicts
    SAB_SHARED_ARRAY(u32, s_code, SAB_PACK_TILE + 64 + (SAB_PACK_TILE + 64) / 32 + 8);
    SAB_SHARED_ARRAY(u16, s_lut, 256);
    SAB_SHARED_ARRAY(u32, s_lo, SAB_PACK_TILE + SAB_PACK_TILE / 32 + 8);
    SAB_SHARED_ARRAY(u32, s_hi, SAB_PACK_TILE + SAB_PACK_TILE / 32 + 8);
    s_lut[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
    const u64 tile0 = (u64)blockIdx.x * SAB_PACK_TILE;
    for (int o = threadIdx.x; o < SAB_PACK_TILE + 64; o += SAB_PACK_THREADS) {
        const u64 i = tile0 + o;
        s_code[SAB_PAD(o)] = i < n ? (u32)s_lut[text[i]] : 0u;
    }
    __syncthreads();
    const int o0 = threadIdx.x * SAB_PACK_ITEMS;
    const u64 top = pw.p[0];
    // first key: independent multiplies by the symbol weights (a Horner chain would serialise k 64-bit multiplies)
    u64 key = 0;
#pragma unroll 4
    for (int t = 0; t < k; ++t) key += (u64)s_code[SAB_PAD(o0 + t)] * pw.p[t];
#pragma unroll
    for (int j = 0; j < SAB_PACK_ITEMS; ++j) {
        s_lo[SAB_PAD(o0 + j)] = (u32)key;
        s_hi[SAB_PAD(o0 + j)] = (u32)(key >> 32);
        key = (key - (u64)s_code[SAB_PAD(o0 + j)] * top) * radix + (u64)s_code[SAB_PAD(o0 + j + k)];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < SAB_PACK_ITEMS; ++j) {
        const int o = threadIdx.x + j * SAB_PACK_THREADS;
        const u64 i = tile0 + o;
        if (i < count) keys[i] = ((u64)s_hi[SAB_PAD(o)] << 32) | s_lo[SAB_PAD(o)];
    }
}

// Fast path of the key packing (round 2): when radix^ka < 2^32 for ka = ceil(k / 2), a key is two HALF keys of ka
// symbols glued together,
//     key(i) = (g(i) - sub) * W + g(i + s),   g(x) = sum_{t < ka} code(x + t) * radix^(ka - 1 - t)   (32 bits),
//     k even: s = ka, W = radix^ka, sub = 0;   k odd: s = ka - 1, W = radix^(ka - 1), sub = code(i + ka - 1)
// (for odd k the two windows overlap in one symbol, which is taken out of the first).  The half keys slide in
// 32-bit arithmetic (two multiply-adds per position instead of two 64-bit multiply chains) and are staged in
// shared memory; the final multiply-add is one 32 x 32 -> 64 bit instruction and the 8-byte stores are coalesced
// without a second staging pass.  Same keys as pack_keys_kernel, bit for bit.
__global__ void __launch_bounds__(SAB_PACK_THREADS)
pack_keys_split_kernel(const u8* __restrict__ text, u64 n, u64 count, const u16* __restrict__ lut, u32 radix, int k, u32 wtop, u32 wmul,
                       u64* __restrict__ keys) {
    SAB_SHARED_ARRAY(u32, s_code, SAB_PACK_TILE + 64 + (SAB_PACK_TILE + 64) / 32 + 8);
    SAB_SHARED_ARRAY(u16, s_lut, 256);
    SAB_SHARED_ARRAY(u32, s_g, SAB_PACK_TILE + 32 + (SAB_PACK_TILE + 32) / 32 + 8);
    s_lut[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
    const u64 tile0 = (u64)blockIdx.x * SAB_PACK_TILE;
    for (int o = threadIdx.x; o < SAB_PACK_TILE + 64; o += SAB_PACK_THREADS) {
        const u64 i = tile0 + o;
        s_code[SAB_PAD(o)] = i < n ? (u32)s_lut[text[i]] : 0u;
    }
    __syncthreads();
    const int ka = (k + 1) / 2;
    const int shift = (k & 1) ? ka - 1 : ka;
    // half keys of the thread's SAB_PACK_ITEMS consecutive positions: Horner for the first, then the window slides;
    // wtop = radix^(ka-1) is the weight of the symbol that leaves
    {
        const int o0 = threadIdx.x * SAB_PACK_ITEMS;
        u32 g = 0;
        for (int t = 0; t < ka; ++t) g = g * radix + s_code[SAB_PAD(o0 + t)];
#pragma unroll
        for (int j = 0; j < SAB_PACK_ITEMS; ++j) {
            s_g[SAB_PAD(o0 + j)] = g;
            g = (g - s_code[SAB_PAD(o0 + j)] * wtop) * radix + s_code[SAB_PAD(o0 + j + ka)];
        }
    }
    if (threadIdx.x < 32) {  // the 32 positions behind the tile that the second halves reach into
        const int o = SAB_PACK_TILE + threadIdx.x;
        u32 g = 0;
        for (int t = 0; t < ka; ++t) g = g * radix + s_code[SAB_PAD(o + t)];
        s_g[SAB_PAD(o)] = g;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < SAB_PACK_ITEMS; ++j) {
        const int o = threadIdx.x + j * SAB_PACK_THREADS;
        const u64 i = tile0 + o;
        if (i < count) {
            const u32 sub = (k & 1) ? s_code[SAB_PAD(o + shift)] : 0u;
            keys[i] = (u64)(s_g[SAB_PAD(o)] - sub) * wmul + (u64)s_g[SAB_PAD(o + shift)];
        }
    }
}

// keys of positions [0, count) of a text (or shard + halo) of n readable bytes: picks the kernel
static int sab_launch_pack(SabContext* c, const u8* d_text, u64 n, u64 count, const u16* d_lut, u32 base, int k, u64* keys) {
    if (count == 0) return SAB_OK;
    const int ka = (k + 1) / 2;
    unsigned __int128 lim = 1;
    for (int t = 0; t < ka; ++t) lim *= base;
    if (k >= 2 && ka <= 32 && lim < ((unsigned __int128)1 << 32)) {
        const u32 wtop = (u32)sab_pow_u64(base, ka - 1);
        const u32 wmul = (u32)sab_pow_u64(base, (k & 1) ? ka - 1 : ka);
        SAB_LAUNCH(pack_keys_split_kernel, (unsigned)div_up64(count, SAB_PACK_TILE), SAB_PACK_THREADS, 0, c->stream, d_text, n, count,
                   d_lut, base, k, wtop, wmul, keys);
    } else {
        SAB_LAUNCH(pack_keys_kernel, (unsigned)div_up64(count, SAB_PACK_TILE), SAB_PACK_THREADS, 0, c->stream, d_text, n, count, d_lut,
                   base, k, sab_pack_pow(base, k), keys);
    }
    SAB_LAUNCH_CHECK();
    c->stats.kernel_launches++;
    return SAB_OK;
}

// ------------------------------------------------------------------ 4b. lazy inverse suffix array
// Scattering all n initial ranks costs a partial-sector write per suffix (~30 G/s on B200, 35-50 ms per
// GiB) although only i + h of the few active i are ever looked up.  So rank[] starts EMPTY except for
// active suffixes; a lookup that hits EMPTY is a suffix that was unique after the initial sort, and
// its rank is 1 + its position in the (kept) sorted key array: re-pack its key from the text, jump
// through the bucket directory, gallop + bisect.  Texts where most suffixes stay active fall back
// to filling rank[] completely (fill_settled_ranks_kernel) so the sorted keys can be dropped.
struct LazyIsa {
    const u8* text;
    const u16* lut;
    const u64* sorted_keys;  // null -> rank[] is complete
    const u32* dir;
    u64 n;
    u32 base;
    int k, dir_shift;
};

// index of the first record of sorted_keys[0..cnt) whose key is >= key, starting from the directory entry
// of the key's bucket (dir is indexed by key >> dir_shift; callers pre-offset the pointer when the array
// only covers a slice of the key space)
__device__ __forceinline__ u64 sorted_key_position(const u64* __restrict__ sorted_keys, u64 cnt, const u32* __restrict__ dir,
                                                   int dir_shift, u64 key) {
    u64 lo = dir[key >> dir_shift];
    u64 hi = lo, step = 1;
    while (hi < cnt && sorted_keys[hi] < key) {  // gallop: keys[lo-1] < key stays true
        lo = hi + 1;
        hi += step;
        step <<= 1;
    }
    if (hi > cnt) hi = cnt;
    while (lo < hi) {  // first position whose key is >= key; the key looked up is present exactly once
        const u64 mid = lo + (hi - lo) / 2;
        if (sorted_keys[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ u32 lazy_rank_lookup(const LazyIsa& z, u64 t) {
    const u64 key = pack_key_at(z.text, z.n, z.lut, z.base, z.k, t);
    return (u32)sorted_key_position(z.sorted_keys, z.n, z.dir, z.dir_shift, key) + 1u;
}

// rank[I[j]] = j + 1 for every singleton record (complete-ISA fallback)
__global__ void __launch_bounds__(256)
fill_settled_ranks_kernel(const u64* __restrict__ K, const u32* __restrict__ I, u64 n, u32* __restrict__ rank) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const u64 key = K[j];
    const bool head = (j == 0) || K[j - 1] != key;
    const bool next_head = (j + 1 >= n) || K[j + 1] != key;
    if (head && next_head) rank[I[j]] = (u32)j + 1u;
}

// ------------------------------------------------------------------ 4c. bucket table from the sorted keys (SURVEY.md 8f N2)
// enable_buckets (/root/reference/src/sa.rs:89-119) counts 2-byte prefixes in a pass over the text.  Inside a
// construction that pass is free: the initial keys are sorted and start with the same two symbols (codes in
// byte order, 0 = end of text), so the inclusive right boundary of a bucket is one lower bound on the sorted key
// array -- 65 793 binary searches, no pass over the text, no second upload.  Needs k >= 2 symbols per key.
//   out[slot] = (add_one ? 1 : 0) + #keys whose 2-symbol prefix is <= the slot's   (slot layout: src/sa.rs:94,103,107)
// add_one accounts for the empty suffix (src/sa.rs:98); a multi-GPU rank passes 0 and the host adds the slices up.
__global__ void __launch_bounds__(256)
bucket_from_keys_kernel(const u64* __restrict__ sorted_keys, u64 cnt, const u16* __restrict__ lut, u32 base, u64 unit /* base^(k-2) */,
                        u32 add_one, u32* __restrict__ out) {
    SAB_SHARED_ARRAY(u16, s_le, 256);  // number of byte values <= c present in the text (= code of c when present)
    SAB_SHARED_ARRAY(u16, s_code, 256);
    {
        const u32 c = threadIdx.x;
        s_code[c] = lut[c];
        u32 le = 0;
        for (u32 b = 0; b <= c; ++b) le += lut[b] ? 1u : 0u;
        s_le[c] = (u16)le;
    }
    __syncthreads();
    const u32 slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= SAB200_BKT_LEN) return;
    if (slot == 0) {
        out[0] = add_one;  // "$": the empty suffix alone
        return;
    }
    const u32 c0 = (slot - 1u) / 257u, r = (slot - 1u) % 257u;
    u64 pre;  // 2-symbol prefixes (as numbers in base `base`) below `pre` are inside or before this slot
    if (!s_code[c0]) pre = ((u64)s_le[c0] + 1ull) * base;                  // absent byte: everything up to the previous present one
    else pre = (u64)s_code[c0] * base + (r ? (u64)s_le[r - 1u] : 0ull) + 1ull;
    u64 lo = 0, hi = cnt;
    if (pre < (u64)base * base) {  // else: every key is below (also avoids base^k = 2^64)
        const u64 upper = pre * unit;
        while (lo < hi) {
            const u64 mid = lo + (hi - lo) / 2;
            if (sorted_keys[mid] < upper) lo = mid + 1;
            else hi = mid;
        }
    } else {
        lo = cnt;
    }
    out[slot] = add_one + (u32)lo;
}

// ------------------------------------------------------------------ 5a. gather the second rank
#define SAB_GATHER_THREADS 256
#define SAB_GATHER_ITEMS 4

__device__ __forceinline__ u32 rank_at(u32* __restrict__ rank, const LazyIsa& z, u64 t) {
    u32 r = rank[t];
    if (r == SAB_RANK_EMPTY) {  // only possible while z.sorted_keys != null
        r = lazy_rank_lookup(z, t);
        rank[t] = r;  // memoise; racing writers store the same value
    }
    return r;
}

// key64[j] = (r1[j] << 32) | rank[idx[j] + h]
__global__ void __launch_bounds__(SAB_GATHER_THREADS)
gather_rank2_kernel(const u32* __restrict__ act_r1, const u32* __restrict__ act_idx, u64 m, u64 h, u32* __restrict__ rank,
                    LazyIsa z, u64* __restrict__ key64) {
    const u64 j0 = ((u64)blockIdx.x * SAB_GATHER_THREADS + threadIdx.x) * SAB_GATHER_ITEMS;
    if (j0 + SAB_GATHER_ITEMS <= m) {
        const uint4 r1 = *(const uint4*)(act_r1 + j0);
        const uint4 ix = *(const uint4*)(act_idx + j0);
        u32 a = rank[(u64)ix.x + h], b = rank[(u64)ix.y + h], c = rank[(u64)ix.z + h], d = rank[(u64)ix.w + h];
        if (a == SAB_RANK_EMPTY) a = rank_at(rank, z, (u64)ix.x + h);
        if (b == SAB_RANK_EMPTY) b = rank_at(rank, z, (u64)ix.y + h);
        if (c == SAB_RANK_EMPTY) c = rank_at(rank, z, (u64)ix.z + h);
        if (d == SAB_RANK_EMPTY) d = rank_at(rank, z, (u64)ix.w + h);
        ulonglong2 o0, o1;
        o0.x = ((u64)r1.x << 32) | a;
        o0.y = ((u64)r1.y << 32) | b;
        o1.x = ((u64)r1.z << 32) | c;
        o1.y = ((u64)r1.w << 32) | d;
        *(ulonglong2*)(key64 + j0) = o0;
        *(ulonglong2*)(key64 + j0 + 2) = o1;
    } else {
        for (u64 j = j0; j < m; ++j) key64[j] = ((u64)act_r1[j] << 32) | rank_at(rank, z, (u64)act_idx[j] + h);
    }
}

// ------------------------------------------------------------------ driver (device pointers)
static inline int sab_ceil_log2_u64(u64 x) {  // smallest b with 2^b >= x
    int b = 0;
    while (b < 64 && (1ull << b) < x) ++b;
    return b;
}

// What sab_plan_alphabet decided, with its code table on the device.
struct SabAlphabet {
    u32 sigma, base;
    int k, key_bits;
    const u16* d_lut;
};

// Code table and key shape from the byte histogram of the whole text (n bytes): codes 1..sigma in byte order (0 =
// absent byte / past the end).  Keys are mixed-radix numbers in base sigma+1 (dense: no bit is wasted on unused
// codes, so more symbols fit a radix pass and the key space is evenly filled), k symbols per key,
// key_bits = bits needed for base^k - 1.  The code table goes to the device, the key shape to c->stats.
//
// Cost model, in bytes moved per suffix: P radix passes of 24 B each, plus ~SAB_ACTIVE_COST bytes over
// all doubling rounds for every suffix still tied after the initial sort; a suffix stays tied with
// probability ~ n * 2^-(k*H2) (H2 = order-0 collision entropy; higher-order structure only makes the
// estimate optimistic, never the result wrong).
static int sab_plan_alphabet(SabContext* c, const u64* hist, u64 n, SabAlphabet* a) {
    u16* lut = c->staging->lut;  // pinned: the upload at the end is asynchronous
    u32 sigma = 0;
    double sum_p2 = 0.0;
    for (int ch = 0; ch < 256; ++ch) {
        if (hist[ch]) ++sigma;
        lut[ch] = (u16)(hist[ch] ? sigma : 0);
        const double p = n ? (double)hist[ch] / (double)n : 0.0;
        sum_p2 += p * p;
    }
    const u32 base = sigma + 1 < 2 ? 2 : sigma + 1;
    // kmax[p] = most symbols whose key fits p radix passes (and 64 bits)
    int k_of_pass[SAB_MAX_PASSES + 1];
    int bits_of_k[65];
    {
        unsigned __int128 pw = 1;
        int kk = 0;
        bits_of_k[0] = 0;
        while (kk < 64) {
            pw *= base;
            if (pw > ((unsigned __int128)1 << 64)) break;
            ++kk;
            unsigned __int128 m = pw - 1;  // largest key
            int bits = 0;
            while (m) {
                ++bits;
                m >>= 1;
            }
            bits_of_k[kk] = bits < 1 ? 1 : bits;
        }
        const int k_full = kk < 1 ? 1 : kk;
        for (int p = 1; p <= SAB_MAX_PASSES; ++p) {
            int best = 0;
            for (int q = 1; q <= k_full; ++q)
                if (bits_of_k[q] <= p * SAB_RADIX_BITS) best = q;
            k_of_pass[p] = best;
        }
    }
    int k = k_of_pass[SAB_MAX_PASSES];
    const double h2 = sum_p2 < 1.0 && sum_p2 > 0.0 ? -log2(sum_p2) : 0.0;
    if (h2 > 1e-3 && n > 0) {
        double best = 1e300;
        for (int p = 1; p <= SAB_MAX_PASSES; ++p) {
            const int kp = k_of_pass[p];
            if (kp < 1) continue;
            double tied = exp2(log2((double)n) - (double)kp * h2);
            if (tied > 1.0) tied = 1.0;
            const double cost = 24.0 * p + SAB_ACTIVE_COST * tied;
            if (cost < best - 1e-9) {
                best = cost;
                k = kp;
            }
        }
    }
    if (k < 1) k = 1;
    a->sigma = sigma;
    a->base = base;
    a->k = k;
    a->key_bits = bits_of_k[k];
    c->stats.sigma = sigma;
    c->stats.bits_per_symbol = (u32)sab_ceil_log2_u64(base);
    c->stats.symbols_per_key = (u32)k;
    SAB_CUDA_TRY(cudaMemcpyAsync(c->scratch->lut, lut, sizeof(c->staging->lut), cudaMemcpyHostToDevice, c->stream));
    a->d_lut = c->scratch->lut;
    return SAB_OK;
}

// The alphabet of a text of n > 0 bytes resident on this GPU.
static int sab_alphabet_local(SabContext* c, const u8* d_text, u64 n, SabAlphabet* a) {
    SAB_TRY(sab_launch_alphabet_hist(c, d_text, n, c->scratch->hist));
    u32 h32[256];
    SAB_TRY(sab_read_u32(c, c->scratch->hist, 256, h32));
    u64 hist[256];
    for (int ch = 0; ch < 256; ++ch) hist[ch] = h32[ch];
    return sab_plan_alphabet(c, hist, n, a);
}

// Bits of the bucket directory of the lazy inverse suffix array over keys of key_bits bits:
// 2^(ceil(log2 n) - shift) entries, at most 2^28 and 2^key_bits, at least 2.
static inline int sab_dir_bits(u64 n, int key_bits, int shift) {
    int dir_bits = sab_ceil_log2_u64(n) - shift;
    if (dir_bits > 28) dir_bits = 28;
    if (dir_bits > key_bits) dir_bits = key_bits;
    if (dir_bits < 1) dir_bits = 1;
    return dir_bits;
}

__global__ void bucket_pairs_kernel(const u8* __restrict__ text, u64 n, const u16* __restrict__ lut, u32 sigma, int dense,
                                    u32* __restrict__ cnt);  // sab_search.cuh
__global__ void bucket_scan_kernel(u32* __restrict__ bkt);

// The bucket table (SAB200_BKT_LEN inclusive boundaries, + 1 for the empty suffix) into d_bkt by counting the byte
// pairs of text[0..n); d_lut, sigma: the code table of the text.
static int sab_pair_buckets(SabContext* c, const u8* d_text, u64 n, const u16* d_lut, u32 sigma, u32* d_bkt) {
    cudaStream_t st = c->stream;
    SAB_CUDA_TRY(cudaMemsetAsync(d_bkt, 0, SAB200_BKT_LEN * sizeof(u32), st));
    if (n > 0) {
        const size_t tab_bytes = (size_t)sigma * (sigma + 1) * sizeof(u32);
        const int dense = tab_bytes <= 160 * 1024;
        const size_t smem = dense ? tab_bytes : 0;
#ifndef SAB_EMU
        SAB_CUDA_TRY(cudaFuncSetAttribute(bucket_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
#endif
        SAB_LAUNCH(bucket_pairs_kernel, sab_grid(c, n, 256 * 64, smem > 64 * 1024 ? 1 : 4), 256, smem, st, d_text, n, d_lut, sigma,
                   dense, d_bkt);
        SAB_LAUNCH_CHECK();
        c->stats.kernel_launches++;
    }
    SAB_LAUNCH(bucket_scan_kernel, 1, 1024, 0, st, d_bkt);
    SAB_LAUNCH_CHECK();
    c->stats.kernel_launches++;
    return SAB_OK;
}

// The bucket table of the running construction into c->want_bkt: from the sorted initial keys (k >= 2), else by
// the pair-counting kernels over the resident text (tiny texts with large alphabets; single GPU only).
static int sab_fused_buckets(SabContext* c, const u8* d_text, u64 n, const u64* sortedK, u64 cnt, const SabAlphabet& al) {
    if (al.k >= 2) {
        SAB_LAUNCH(bucket_from_keys_kernel, (SAB200_BKT_LEN + 255u) / 256u, 256, 0, c->stream, sortedK, cnt, al.d_lut, al.base,
                   sab_pow_u64(al.base, al.k - 2), c->bkt_add_one, c->want_bkt);
        SAB_LAUNCH_CHECK();
        c->stats.kernel_launches++;
        return SAB_OK;
    }
    if (!c->bkt_add_one) {
        sab_set_error("fused bucket table: keys of one symbol on a multi-GPU rank");
        return SAB_ERR_INTERNAL;
    }
    return sab_pair_buckets(c, d_text, n, al.d_lut, al.sigma, c->want_bkt);
}

// The spare buffers of the in-group sort (sab_group_sort) of `count` records at the front of sb: the unused tails of
// the round's buffers behind the first align_up(count, 64) records (sb.k[*] hold key_cap records, sb.v[*] val_cap),
// and the position list `pos`.
static inline GroupSortSpare sab_group_sort_spare(const SortBuffers<u64>& sb, u64 count, u64 key_cap, u64 val_cap, u32* pos) {
    const u64 used = sab_align_up(count, 64);
    const u64 cap_keys = key_cap > used ? key_cap - used : 0;
    const u64 cap_vals = val_cap > used ? val_cap - used : 0;
    GroupSortSpare sp;
    sp.k[0] = sb.k[0] + used;
    sp.k[1] = sb.k[1] + used;
    sp.v[0] = sb.v[0] + used;
    sp.v[1] = sb.v[1] + used;
    sp.pos = pos;
    sp.cap = cap_keys < cap_vals ? cap_keys : cap_vals;
    return sp;
}

// The buffers of the doubling rounds, taken from those of the initial sort of cnt records (result in buf.cur): the
// round keys ping-pong inside the two halves of the free key buffer while the sorted keys are kept (lazy inverse
// suffix array), else over both key buffers.  *key_cap = records each round key buffer holds.
static inline SortBuffers<u64> sab_round_buffers(const SortBuffers<u64>& buf, u64 cnt, bool keep_sorted, u64* key_cap) {
    const u64 half = sab_align_up((size_t)(cnt + 8) / 2, 32);
    SortBuffers<u64> rb;
    rb.k[0] = buf.k[buf.cur ^ 1];
    rb.k[1] = keep_sorted ? buf.k[buf.cur ^ 1] + half : buf.k[buf.cur];
    *key_cap = keep_sorted ? (cnt + 8) - half : cnt + 8;
    rb.v[0] = buf.v[buf.cur ^ 1];
    rb.v[1] = buf.v[buf.cur];
    rb.cur = 0;
    return rb;
}

// init_ranks (4) over the cnt sorted records; *m = the number of records left active
static int sab_init_ranks(SabContext* c, const u64* sortedK, const u32* sortedI, u64 cnt, u32 rank_base, u32* rank, u32* rank_seq,
                          u32* sa_out, u32* act_r1, u32* act_idx, u32* dir, int dir_shift, u64* m) {
    const u64 tiles = div_up64(cnt, SAB_SCAN_TILE);
    TileState<RankScan> ts = sab_tile_state<RankScan>(c, tiles);
    sab_prof_begin(c, SAB_PROF_RANK);
    SAB_LAUNCH(init_ranks_kernel, (unsigned)tiles, SAB_SCAN_THREADS, 0, c->stream, sortedK, sortedI, cnt, rank_base, rank, rank_seq,
               sa_out, act_r1, act_idx, &c->scratch->count, dir, dir_shift, ts);
    sab_prof_end(c);
    SAB_LAUNCH_CHECK();
    c->stats.kernel_launches++;
    u32 active;
    SAB_TRY(sab_read_u32(c, &c->scratch->count, 1, &active));
    *m = active;
    return SAB_OK;
}

// re-rank (5) of the cnt sorted records of a round; the number of survivors is left in c->scratch->count
static int sab_launch_rerank(SabContext* c, const SortBuffers<u64>& sb, u64 cnt, u32* rank, u32* sa, u32* out_r1, u32* out_idx,
                             u32* upd_idx, u32* upd_r, u32* set_pos) {
    const u64 tiles = div_up64(cnt, SAB_SCAN_TILE);
    TileState<RerankScan> ts = sab_tile_state<RerankScan>(c, tiles);
    sab_prof_begin(c, SAB_PROF_RANK);
    SAB_LAUNCH(rerank_kernel, (unsigned)tiles, SAB_SCAN_THREADS, 0, c->stream, (const u64*)sb.k[sb.cur], (const u32*)sb.v[sb.cur], cnt,
               rank, sa, out_r1, out_idx, upd_idx, upd_r, set_pos, &c->scratch->count, ts);
    sab_prof_end(c);
    SAB_LAUNCH_CHECK();
    c->stats.kernel_launches++;
    return SAB_OK;
}

// bytes of arena needed for a text of n bytes (excluding text and sa, which the caller provides)
static inline size_t sab_saca_workspace_bytes(u64 n) {
    const size_t N = (size_t)n + 8;
    const int dir_bits = sab_dir_bits(n, 64, SAB_DIR_SHIFT);
    return 2 * sab_align_up(N * 8, 256) + 3 * sab_align_up(N * 4, 256) + sab_align_up((N + 1) * 4, 256) +
           sab_align_up((((size_t)1 << dir_bits) + 8) * 4, 256) + sab_align_up((N / 32 + 8) * 4, 256) + 4096;
}


// d_text: n bytes; d_sa: n+1 u32; both device memory.  Work is enqueued on c->stream and the
// stream is synchronised before returning.
static int sab_saca_device(SabContext* c, const u8* d_text, u64 n, u32* d_sa) {
    SabStats& S = c->stats;
    memset(&S, 0, sizeof(S));
    S.n = n;
    cudaStream_t st = c->stream;
    if (n == 0) {
        SAB_CUDA_TRY(cudaMemsetAsync(d_sa, 0, sizeof(u32), st));
        SAB_CUDA_TRY(cudaStreamSynchronize(st));
        return SAB_OK;
    }
    SAB_TRY(sab_arena_reserve(c, sab_saca_workspace_bytes(n)));
    c->arena.used = 0;
    SortBuffers<u64> buf;
    buf.k[0] = sab_arena_take<u64>(&c->arena, n + 8);
    buf.k[1] = sab_arena_take<u64>(&c->arena, n + 8);
    buf.v[0] = sab_arena_take<u32>(&c->arena, n + 8);
    buf.v[1] = sab_arena_take<u32>(&c->arena, n + 8);
    u32* r1buf = sab_arena_take<u32>(&c->arena, n + 8);
    u32* rank = sab_arena_take<u32>(&c->arena, n + 9);
    buf.cur = 0;
    SAB_TRY(sab_ensure_scan(c, (size_t)div_up64(n, SAB_SCAN_TILE)));

    // 1. alphabet
    sab_prof_begin(c, SAB_PROF_PACK);
    SabAlphabet al;
    SAB_TRY(sab_alphabet_local(c, d_text, n, &al));

    // 2. packed keys
    SAB_TRY(sab_launch_pack(c, d_text, n, n, al.d_lut, al.base, al.k, buf.k[0]));
    sab_prof_end(c);

    // 3. sort (key, i); the payload of the first pass is generated, not read
    // (the last pass writes the sorted indices straight into sa[1..]: they need no copy afterwards)
    bool sa_written = false;
    SAB_TRY(sab_radix_sort<u64>(c, buf, n, 0, al.key_bits, /*iota=*/true, &S.passes[0], d_sa + 1, &sa_written));

    // 4. ranks, SA skeleton, active list, bucket directory over the sorted keys
    const u64* sortedK = buf.k[buf.cur];
    if (c->want_bkt) SAB_TRY(sab_fused_buckets(c, d_text, n, sortedK, n, al));
    const u32* sortedI = sa_written ? d_sa + 1 : buf.v[buf.cur];
    u32* act_idx = buf.v[buf.cur ^ 1];
    const int dir_bits = sab_dir_bits(n, al.key_bits, SAB_DIR_SHIFT);
    const int dir_shift = al.key_bits - dir_bits;
    u32* dir = sab_arena_take<u32>(&c->arena, ((size_t)1 << dir_bits) + 8);
    u32* split_bitmap = sab_arena_take<u32>(&c->arena, (size_t)n / 32 + 8);
    SAB_CUDA_TRY(cudaMemsetAsync(rank, 0xff, n * sizeof(u32), st));
    SAB_CUDA_TRY(cudaMemsetAsync(rank + n, 0, sizeof(u32), st));  // the empty suffix has rank 0
    c->staging->sa0 = (u32)n;
    SAB_CUDA_TRY(cudaMemcpyAsync(d_sa, &c->staging->sa0, sizeof(u32), cudaMemcpyHostToDevice, st));  // sa[0] = n
    u64 m = 0;
    SAB_TRY(sab_init_ranks(c, sortedK, sortedI, n, 1u, rank, nullptr, sa_written ? nullptr : d_sa + 1, r1buf, act_idx, dir, dir_shift, &m));
    S.active[0] = m;
    if (m == 0) {
        S.rounds = 0;
        return SAB_OK;
    }

    // 4b. lazy or complete inverse suffix array
    LazyIsa z;
    z.text = d_text;
    z.lut = al.d_lut;
    z.dir = dir;
    z.n = n;
    z.base = al.base;
    z.k = al.k;
    z.dir_shift = dir_shift;
    z.sorted_keys = m <= n / 4 ? sortedK : nullptr;  // keep the sorted keys
    if (!z.sorted_keys) {
        sab_prof_begin(c, SAB_PROF_RANK);
        SAB_LAUNCH(fill_settled_ranks_kernel, (unsigned)div_up64(n, 256), 256, 0, st, sortedK, sortedI, n, rank);
        sab_prof_end(c);
        SAB_LAUNCH_CHECK();
        S.kernel_launches++;
    }
    u64 key_cap;  // records each of rb.k[0], rb.k[1] can hold
    SortBuffers<u64> rb = sab_round_buffers(buf, n, z.sorted_keys != nullptr, &key_cap);

    // 5. doubling rounds
    u64 h = (u64)al.k;
    u32 round = 0;
    const int rank_bits = sab_ceil_log2_u64(n + 2);
    // the split filter (5c) pays off while few groups split: repetitive texts, early rounds
    bool filter_on = (z.sorted_keys == nullptr) && m >= SAB_FILTER_MIN;
    bool group_sort_on = true;  // 5d, until most records are in large groups
    // The active list leaves init_ranks ascending in r1.  A round of the split filter parks the unsplit
    // groups in front of the re-ranked ones, so the next list is two ascending runs: groups stay contiguous
    // (all the scan kernels need) but the list is no longer monotone -- sab_group_sort is told, because it
    // returns the radix-sorted records of large groups to their positions in the order of their groups.
    bool list_sorted = true;
    int gs_pause = 0;  // rounds the in-group sort sits out after its large-group records did not fit
    while (m > 0) {
        ++round;
        if (round >= SAB_MAX_ROUNDS || h > n) {
            sab_set_error("prefix doubling did not converge (round %u, h=%llu, m=%llu)", round, (unsigned long long)h,
                          (unsigned long long)m);
            return SAB_ERR_INTERNAL;
        }
        sab_prof_begin(c, SAB_PROF_GATHER);
        SAB_LAUNCH(gather_rank2_kernel, (unsigned)div_up64(m, (u64)SAB_GATHER_THREADS * SAB_GATHER_ITEMS), SAB_GATHER_THREADS,
                   0, st, (const u32*)r1buf, (const u32*)rb.v[rb.cur], m, h, rank, z, rb.k[rb.cur]);
        sab_prof_end(c);
        SAB_LAUNCH_CHECK();
        S.kernel_launches++;
        u64 n_sort = m, n_stay = 0;
        if (filter_on && m >= SAB_FILTER_MIN) {
            const u64 tiles = div_up64(m, SAB_SCAN_TILE);
            TileState<FilterScan> ts = sab_tile_state<FilterScan>(c, tiles);
            sab_prof_begin(c, SAB_PROF_RANK);
            SAB_CUDA_TRY(cudaMemsetAsync(split_bitmap, 0, ((size_t)n / 32 + 8) * sizeof(u32), st));
            SAB_LAUNCH(mark_split_groups_kernel, (unsigned)div_up64(m, 256), 256, 0, st, (const u64*)rb.k[rb.cur], m, split_bitmap);
            SAB_LAUNCH_CHECK();
            SAB_LAUNCH(split_filter_kernel, (unsigned)tiles, SAB_SCAN_THREADS, 0, st, rb.k[rb.cur], rb.v[rb.cur], m,
                       (const u32*)split_bitmap, r1buf, rb.v[rb.cur ^ 1], c->scratch->filter, ts);
            sab_prof_end(c);
            SAB_LAUNCH_CHECK();
            S.kernel_launches += 2;
            u32 split[2];
            SAB_TRY(sab_read_u32(c, c->scratch->filter, 2, split));
            n_sort = split[0];
            n_stay = split[1];
            if (n_sort * 10 > m * 7) filter_on = false;  // from here on most groups split every round
        }
        u32 kept = 0;
        bool order_restored = false;  // the round's records went through the full radix sort: ascending in r1 again
        if (n_sort > 0) {
            // sort the n_sort records at the front of (k[cur], v[cur]); the spare payload buffer starts
            // behind the n_stay records already parked in v[cur^1]
            SortBuffers<u64> sb;
            sb.k[0] = rb.k[rb.cur];
            sb.k[1] = rb.k[rb.cur ^ 1];
            sb.v[0] = rb.v[rb.cur];
            sb.v[1] = rb.v[rb.cur ^ 1] + n_stay;
            sb.cur = 0;
            // 5d. small groups are ordered in one sweep; the spare buffers for the records of big groups are
            // the unused tails of the round buffers (keys, payloads) and of r1buf (positions)
            int sorted = 0;
            if (group_sort_on) {
                const GroupSortSpare sp = sab_group_sort_spare(sb, n_sort, key_cap, n + 8 - n_stay, r1buf + n_stay);
                // the sweep is tried whenever there is any spare room: it reports how many records belong to
                // large groups even when they do not fit (then the round takes the radix sort and the sweep
                // pauses for two rounds -- the list, and with it the need for room, only shrinks)
                if (sp.cap >= 64 && gs_pause == 0) {
                    u64 nbig = 0;
                    sorted = sab_group_sort(c, sb, n_sort, 32 + rank_bits, sp, &S.passes[round], &nbig, list_sorted);
                    if (sorted < 0) return sorted;
                    if (nbig * 2 > n_sort) group_sort_on = false;  // mostly large groups: the sweep does not pay
                    else if (!sorted) gs_pause = 2;
                } else if (gs_pause > 0) {
                    --gs_pause;
                }
            }
            if (!sorted) {
                SAB_TRY(sab_radix_sort<u64>(c, sb, n_sort, 0, 32 + rank_bits, /*iota=*/false, &S.passes[round]));
                order_restored = true;
            }
            u32* out_idx = (sb.cur == 0) ? rb.v[rb.cur ^ 1] + n_stay : rb.v[rb.cur];
            SAB_TRY(sab_launch_rerank(c, sb, n_sort, rank, d_sa, r1buf + n_stay, out_idx, nullptr, nullptr, nullptr));
            SAB_TRY(sab_read_u32(c, &c->scratch->count, 1, &kept));
            if (sb.cur != 0 && kept > 0)  // the survivors were written to the other buffer: append them to the parked ones
                SAB_CUDA_TRY(cudaMemcpyAsync(rb.v[rb.cur ^ 1] + n_stay, rb.v[rb.cur], kept * sizeof(u32), cudaMemcpyDeviceToDevice, st));
        }
        // Parked records first, then the survivors of the sort.  The in-group sort keeps the records where they
        // are: a list of several ascending runs stays one until a round takes the full radix sort.
        list_sorted = n_stay == 0 && (list_sorted || order_restored);
        rb.cur ^= 1;
        m = n_stay + kept;
        S.active[round] = m;
        h *= 2;
    }
    S.rounds = round;
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    return SAB_OK;
}
