// sab_lz.cuh -- Lempel-Ziv (LZ77) factorization and its decoder (include/sab200.h "LZ77").
//
// Forward, after the construction, in its dead workspace:
//   1. isa (lcp_isa_kernel), the LCP array through the permuted LCP array (sab_lz_lcp: O(n log n) compared bytes, no
//      quadratic case), block minima (fan-out 256) over sa[] and over the LCP array.
//   2. lz_lpf_kernel, one warp per suffix-array row j >= 1 with i = sa[j]: PSV / NSV = the nearest rows before / after
//      j whose sa value is below i (ms_left / ms_right over the sa hierarchy), the LCP range minima over (PSV, j] and
//      (j, NSV] (lz_range_min over the LCP hierarchy), hence LPF[i] and its source, written in text order.  Every search
//      reads at most 2 x 256 entries per level, whatever the text: monotone runs of the suffix array (all-'a' text,
//      periodic texts) cost no more per row than any other.
//   3. The greedy parse over next(i) = i + max(1, LPF[i]), with exits of fan-out C = SAB_LZ_CHUNK:
//        g0(i)  the first node >= the end of i's chunk of C positions on the path from i (a reverse walk per chunk);
//        g1(i)  the same for i's block of C^2 positions, from g0 (the chunks of a block last to first, all positions of
//               a chunk in parallel).
//      A descent from 0 then follows g1 across the blocks (at most n / C^2 + 1 <= 1025 steps for n < 2^32), g0 inside
//      every visited block, and next() inside every visited chunk, where it flags the factor starts.  Dependent depth
//      O(C + n / C^2) per phase, work O(n) per phase, whatever z is.
//   4. lz_compact_kernel: the flagged starts become (pos, len) through the chained scan of sab_scan.cuh; the count is z.
//
// Decoder: a chained scan of max(1, len) gives the factor starts b_t and checks the parse.  Every output byte then
// points at its source byte pos + (x - b_t) < x (a literal at itself), and pointer jumping in place runs until a round
// changes nothing: at most ceil(log2 n) + 1 rounds, since every round at least halves each distance to a literal.
#pragma once
#include "sab_bwt.cuh"
#include "sab_ms.cuh"

// Positions per chunk of the parse; a block of the second level holds SAB_LZ_CHUNK^2.  Two stored levels cover
// n < 2^32 at 2048 with a top walk of at most 1025 steps.  The emulator shrinks it so its small texts cross many
// chunks and blocks.
#ifndef SAB_LZ_CHUNK
#ifdef SAB_EMU
#define SAB_LZ_CHUNK 8
#else
#define SAB_LZ_CHUNK 2048
#endif
#endif
#define SAB_LZ_BLOCK ((u64)SAB_LZ_CHUNK * SAB_LZ_CHUNK)
#define SAB_LZ_ROWS 16            // suffix-array rows per warp of lz_lpf_kernel
#define SAB_LZ_EXIT_THREADS 1024  // threads of the block that builds g1 for one block of C^2 positions
#define SAB_LZ_NONE 0xffffffffu

// A block-minimum hierarchy over lvl[0] (the members ms_left / ms_right read)
struct LzLevels {
    const u32* lvl[SAB_MS_LEVELS];
    u64 cnt[SAB_MS_LEVELS];
    u32 top;
};

// ------------------------------------------------------------------ forward
// min of v[lo .. hi] (hi - lo < 256), in every lane
__device__ __forceinline__ u32 lz_warp_min(const u32* __restrict__ v, u64 lo, u64 hi, u32 lane) {
    u32 m = 0xffffffffu;
    for (u64 b = lo; b <= hi; b += 32) {
        if (b + lane <= hi) {
            const u32 x = v[b + lane];
            m = x < m ? x : m;
        }
    }
    for (int o = 16; o; o >>= 1) {
        const u32 x = __shfl_xor_sync(SAB_FULL, m, o);
        m = x < m ? x : m;
    }
    return m;
}

// min of lvl[0][a .. b], a <= b: the partial blocks at both ends at each level, the whole blocks between them one level
// up -- at most 2 x 256 entries per level
__device__ __forceinline__ u32 lz_range_min(const LzLevels& L, u64 a, u64 b, u32 lane) {
    u32 m = 0xffffffffu;
    for (u32 k = 0;; ++k) {
        if ((a >> 8) == (b >> 8) || k == L.top) {  // the top level has at most 256 entries
            const u32 x = lz_warp_min(L.lvl[k], a, b, lane);
            return x < m ? x : m;
        }
        const u32 x = lz_warp_min(L.lvl[k], a, a | 255, lane), y = lz_warp_min(L.lvl[k], b & ~255ull, b, lane);
        m = x < m ? x : m;
        m = y < m ? y : m;
        a = (a >> 8) + 1;
        b = (b >> 8) - 1;
        if (a > b) return m;
    }
}

struct LzArgs {
    LzLevels sa, lcp;  // sa.lvl[0] = the suffix array (n + 1 entries), lcp.lvl[0] = its LCP array
    u64 n;
    u32 *lpf, *src;    // by text position
};

// LPF[i] and its source for the rows j of this warp (Crochemore-Ilie): LPF[i] = max(lcp(i, sa[PSV]), lcp(i, sa[NSV])),
// the source is sa[PSV] unless the NSV side is strictly longer.  Row 0 (sa[0] = n) is below no i, so it never is a PSV.
__global__ void __launch_bounds__(256) lz_lpf_kernel(LzArgs a) {
    const u64 w = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 j0 = 1 + w * SAB_LZ_ROWS, n = a.n;
    if (j0 > n) return;  // whole warps
    const u32 lane = lane_id();
    const u32* sa = a.sa.lvl[0];
    for (u64 j = j0; j < j0 + SAB_LZ_ROWS && j <= n; ++j) {
        const u64 i = sa[j];
        const u64 p = ms_left(a.sa, j - 1, i, lane);  // 0: none
        const u64 q = ms_right(a.sa, j, i, lane);     // n + 1: none
        const u32 lp = p ? lz_range_min(a.lcp, p + 1, j, lane) : 0u;
        const u32 lq = q <= n ? lz_range_min(a.lcp, j + 1, q, lane) : 0u;
        if (lane == 0) {
            a.lpf[i] = lp > lq ? lp : lq;
            a.src[i] = lp >= lq ? (p ? sa[p] : 0u) : sa[q];
        }
    }
}

__device__ __forceinline__ u64 lz_next(const u32* __restrict__ lpf, u64 i) {
    const u32 l = lpf[i];
    return i + (l ? l : 1u);
}

// g0 of every position, one thread per chunk walking it backwards
__global__ void __launch_bounds__(256) lz_exit0_kernel(const u32* __restrict__ lpf, u64 n, u32* __restrict__ g0) {
    const u64 c0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * SAB_LZ_CHUNK;
    if (c0 >= n) return;
    const u64 end = c0 + SAB_LZ_CHUNK < n ? c0 + SAB_LZ_CHUNK : n;
    for (u64 i = end; i-- > c0;) {
        const u64 j = lz_next(lpf, i);
        g0[i] = j >= end ? (u32)j : g0[j];
    }
}

// g1 of every position of block blockIdx.x: its chunks last to first, all positions of a chunk at once (g0 of a
// position lies in a later chunk of the block, already done, or beyond the block)
__global__ void __launch_bounds__(SAB_LZ_EXIT_THREADS) lz_exit1_kernel(const u32* __restrict__ g0, u64 n, u32* g1) {
    const u64 b0 = (u64)blockIdx.x * SAB_LZ_BLOCK;
    const u64 end = b0 + SAB_LZ_BLOCK < n ? b0 + SAB_LZ_BLOCK : n;
    for (u64 c0 = b0 + (end - b0 - 1) / SAB_LZ_CHUNK * SAB_LZ_CHUNK;; c0 -= SAB_LZ_CHUNK) {
        const u64 c1 = c0 + SAB_LZ_CHUNK < end ? c0 + SAB_LZ_CHUNK : end;
        for (u64 i = c0 + threadIdx.x; i < c1; i += blockDim.x) {
            const u32 j = g0[i];
            g1[i] = j >= end ? j : g1[j];
        }
        __syncthreads();
        if (c0 == b0) break;
    }
}

// the top of the descent, one thread: the entry of every block the path from 0 visits
__global__ void lz_walk_top_kernel(const u32* __restrict__ g1, u64 n, u32* __restrict__ e1) {
    for (u64 p = 0; p < n; p = g1[p]) e1[p / SAB_LZ_BLOCK] = (u32)p;
}

// one thread per block: from its entry along g0, the entry of every chunk the path visits
__global__ void __launch_bounds__(256)
lz_walk_block_kernel(const u32* __restrict__ g0, const u32* __restrict__ e1, u64 n, u32* __restrict__ e0) {
    const u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (b * SAB_LZ_BLOCK >= n || e1[b] == SAB_LZ_NONE) return;
    const u64 end = (b + 1) * SAB_LZ_BLOCK < n ? (b + 1) * SAB_LZ_BLOCK : n;
    for (u64 p = e1[b]; p < end; p = g0[p]) e0[p / SAB_LZ_CHUNK] = (u32)p;
}

// one thread per chunk: from its entry along next(), the factor starts inside it
__global__ void __launch_bounds__(256)
lz_walk_chunk_kernel(const u32* __restrict__ lpf, const u32* __restrict__ e0, u64 n, u8* __restrict__ flag) {
    const u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c * SAB_LZ_CHUNK >= n || e0[c] == SAB_LZ_NONE) return;
    const u64 end = (c + 1) * SAB_LZ_CHUNK < n ? (c + 1) * SAB_LZ_CHUNK : n;
    for (u64 p = e0[c]; p < end; p = lz_next(lpf, p)) flag[p] = 1;
}

// The flagged positions of [0, n) in ascending order as factors into pos / len[0, cap); *count = z.  Warp-striped tiles
// chained by the decoupled look-back of sab_scan.cuh, as bwt_sample_list_kernel.
__global__ void __launch_bounds__(SAB_SCAN_THREADS)
lz_compact_kernel(const u8* __restrict__ s, const u8* __restrict__ flag, const u32* __restrict__ lpf, const u32* __restrict__ src,
                  u64 n, u32* __restrict__ pos, u32* __restrict__ len, u64 cap, u32* __restrict__ count, TileState<u32> st) {
    const u32 tile = blockIdx.x, lane = lane_id();
    const u64 base = (u64)tile * SAB_SCAN_TILE;
    const u64 wbase = base + (u64)warp_id() * SAB_WCHUNK;
    u32 fb[SAB_SCAN_ITEMS];
    u32 mine = 0;
#pragma unroll
    for (int k = 0; k < SAB_SCAN_ITEMS; ++k) {
        const u64 j = wbase + (u64)k * 32 + lane;
        fb[k] = __ballot_sync(SAB_FULL, j < n && flag[j]);
        mine += (u32)__popc(fb[k]);
    }
    u32 wpre, total;
    warp_aggregates<u32, CountOp>(mine, CountOp(), 0u, wpre, total);
    const u32 prefix = tile_exclusive_prefix<u32, CountOp>(st, tile, total, CountOp(), 0u);
    u32 run = prefix + wpre;
#pragma unroll
    for (int k = 0; k < SAB_SCAN_ITEMS; ++k) {
        const u64 j = wbase + (u64)k * 32 + lane;
        if ((fb[k] >> lane) & 1u) {
            const u32 t = run + (u32)__popc(fb[k] & lanemask_lt());
            if (t < cap) {
                const u32 l = lpf[j];
                pos[t] = l ? src[j] : (u32)s[j];
                len[t] = l;
            }
        }
        run += (u32)__popc(fb[k]);
    }
    if (threadIdx.x == 0 && base + SAB_SCAN_TILE >= n) *count = prefix + total;  // last tile
}

// ------------------------------------------------------------------ LCP array through the permuted LCP array
// Kasai's chunked recurrence (lcp_kasai_kernel) compares from scratch at the first position of every chunk, which is
// quadratic on long runs: n^2 / 64 bytes on all-'a' text.  Here PLCP[i] = lcp(i, Phi(i)), Phi(i) = sa[isa[i] - 1], is
// compared only at the IRREDUCIBLE positions: i is reducible when s[i-1] = s[Phi(i)-1], and then Phi(i-1) = Phi(i) - 1
// and PLCP[i] = PLCP[i-1] - 1 (Karkkainen, Manzini, Puglisi 2009).  The irreducible values sum to at most 2 n log2 n.
//   lz_plcp_kernel       one thread per position: SAB_LZ_CMP bytes of every irreducible comparison; the longer ones go
//                        to a list
//   lz_plcp_round_kernel round r: every listed comparison continues over 2^r windows of SAB_LZ_CMP bytes at once, one
//                        thread each, and the first mismatch is kept by atomicMin -- the work stays within twice the
//                        common prefix, the rounds are at most log2(n / SAB_LZ_CMP) + 1
//   lz_plcp_fill_kernel  a chained max-scan finds the last irreducible position r <= i; PLCP[i] = PLCP[r] - (i - r),
//                        scattered to lcp[isa[i]]
#define SAB_LZ_CMP 256

struct LzLong {
    u32 i, j;  // the position and Phi(i)
    u32 h;     // bytes known to match
    u32 stop;  // first mismatch found by the running round (SAB_LZ_NONE: none yet)
};

// common prefix of the suffixes a and b from offset h, up to offset e <= n - max(a, b)
__device__ __forceinline__ u64 lz_cmp(const u8* __restrict__ s, u64 a, u64 b, u64 h, u64 e) {
    while (h < e && s[a + h] == s[b + h]) ++h;
    return h;
}

__global__ void __launch_bounds__(256)
lz_plcp_kernel(const u8* __restrict__ s, u64 n, const u32* __restrict__ sa, const u32* __restrict__ isa, u32* __restrict__ plcp,
               LzLong* __restrict__ list, u64 cap, u32* __restrict__ count) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 j = sa[isa[i] - 1];  // isa[i] >= 1: row 0 is the empty suffix
    if (i > 0 && j > 0 && j < n && s[i - 1] == s[j - 1]) {
        plcp[i] = SAB_LZ_NONE;  // reducible
        return;
    }
    const u64 lim = j < n ? n - (i > j ? i : j) : 0;
    const u64 h = lz_cmp(s, i, j, 0, lim < SAB_LZ_CMP ? lim : SAB_LZ_CMP);
    plcp[i] = (u32)h;
    if (h == SAB_LZ_CMP && lim > SAB_LZ_CMP) {
        const u32 k = atomicAdd(count, 1u);
        if (k < cap) list[k] = LzLong{(u32)i, (u32)j, (u32)h, SAB_LZ_NONE};
    }
}

// task t: window t & (2^r - 1) of entry t >> r
__global__ void __launch_bounds__(256) lz_plcp_round_kernel(const u8* __restrict__ s, u64 n, LzLong* list, u64 tasks, int r) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= tasks) return;
    LzLong* e = &list[t >> r];
    const u64 a = e->i, b = e->j;
    const u64 lim = n - (a > b ? a : b);
    const u64 off = (u64)e->h + (t & ((1ull << r) - 1)) * SAB_LZ_CMP;
    if (off >= lim) return;
    const u64 end = off + SAB_LZ_CMP < lim ? off + SAB_LZ_CMP : lim;
    const u64 d = lz_cmp(s, a, b, off, end);
    if (d < end || end == lim) atomicMin(&e->stop, (u32)d);
}

// entries with a mismatch are done; the others move on by the 2^r windows of the round
__global__ void __launch_bounds__(256)
lz_plcp_next_kernel(const LzLong* __restrict__ list, u64 m, int r, u32* __restrict__ plcp, LzLong* __restrict__ next, u32* __restrict__ count) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    LzLong e = list[k];
    if (e.stop != SAB_LZ_NONE) {
        plcp[e.i] = e.stop;
        return;
    }
    e.h += (u32)SAB_LZ_CMP << r;
    next[atomicAdd(count, 1u)] = e;
}

struct LzMaxOp {
    __device__ __forceinline__ u32 operator()(u32 a, u32 b) const { return a > b ? a : b; }
};

// lcp[isa[i]] = PLCP[i] for i < n; r = the last irreducible position <= i by a chained max-scan (position 0 always is
// irreducible).  Tiles as lz_compact_kernel.
__global__ void __launch_bounds__(SAB_SCAN_THREADS)
lz_plcp_fill_kernel(const u32* __restrict__ plcp, const u32* __restrict__ isa, u64 n, u32* __restrict__ lcp, TileState<u32> st) {
    const u32 tile = blockIdx.x, lane = lane_id();
    const u64 base = (u64)tile * SAB_SCAN_TILE;
    const u64 wbase = base + (u64)warp_id() * SAB_WCHUNK;
    u32 v[SAB_SCAN_ITEMS];
    u32 mine = 0;
#pragma unroll
    for (int k = 0; k < SAB_SCAN_ITEMS; ++k) {
        const u64 j = wbase + (u64)k * 32 + lane;
        v[k] = j < n && plcp[j] != SAB_LZ_NONE ? (u32)j : 0u;
        mine = v[k] > mine ? v[k] : mine;
    }
    mine = warp_reduce_pod<u32, LzMaxOp>(mine, LzMaxOp());
    u32 wpre, total;
    warp_aggregates<u32, LzMaxOp>(mine, LzMaxOp(), 0u, wpre, total);
    const u32 prefix = tile_exclusive_prefix<u32, LzMaxOp>(st, tile, total, LzMaxOp(), 0u);
    u32 run = prefix > wpre ? prefix : wpre;
#pragma unroll
    for (int k = 0; k < SAB_SCAN_ITEMS; ++k) {
        const u64 j = wbase + (u64)k * 32 + lane;
        const u32 incl = warp_incl_max(v[k]);
        const u32 r = incl > run ? incl : run;
        if (j < n) {
            const u32 p = plcp[j];
            lcp[isa[j]] = p != SAB_LZ_NONE ? p : plcp[r] - (u32)(j - r);
        }
        const u32 last = __shfl_sync(SAB_FULL, incl, 31);
        run = last > run ? last : run;
    }
}

// lcp[0 .. n] of the suffix array d_sa from its inverse; plcp: n words, la / lb: room for cap list entries each
static int sab_lz_lcp(SabContext* c, const u8* d_s, u64 n, const u32* d_sa, const u32* isa, u32* plcp, LzLong* la, LzLong* lb, u64 cap,
                      u32* lcp) {
    cudaStream_t st = c->stream;
    u32* cnt = &c->scratch->lz[1];
    SAB_CUDA_TRY(cudaMemsetAsync(cnt, 0, sizeof(u32), st));
    SAB_LAUNCH(lz_plcp_kernel, (unsigned)div_up64(n, 256), 256, 0, st, d_s, n, d_sa, isa, plcp, la, cap, cnt);
    SAB_LAUNCH_CHECK();
    u32 m;
    SAB_TRY(sab_read_u32(c, cnt, 1, &m));
    if (m > cap) {
        sab_set_error("sab200_lz77: %u long common prefixes, room for %llu", m, (unsigned long long)cap);
        return SAB_ERR_INTERNAL;
    }
    for (int r = 0; m > 0; ++r) {
        const u64 tasks = (u64)m << r;
        SAB_LAUNCH(lz_plcp_round_kernel, (unsigned)div_up64(tasks, 256), 256, 0, st, d_s, n, la, tasks, r);
        SAB_LAUNCH_CHECK();
        SAB_CUDA_TRY(cudaMemsetAsync(cnt, 0, sizeof(u32), st));
        SAB_LAUNCH(lz_plcp_next_kernel, (unsigned)div_up64(m, 256), 256, 0, st, (const LzLong*)la, (u64)m, r, plcp, lb, cnt);
        SAB_LAUNCH_CHECK();
        SAB_TRY(sab_read_u32(c, cnt, 1, &m));
        LzLong* t = la;
        la = lb;
        lb = t;
    }
    SAB_CUDA_TRY(cudaMemsetAsync(lcp, 0, sizeof(u32), st));  // lcp[0]: the empty suffix
    const u64 tiles = div_up64(n, SAB_SCAN_TILE);
    SAB_TRY(sab_ensure_scan(c, (size_t)tiles));
    TileState<u32> ts = sab_tile_state<u32>(c, tiles);
    SAB_LAUNCH(lz_plcp_fill_kernel, (unsigned)tiles, SAB_SCAN_THREADS, 0, st, (const u32*)plcp, isa, n, lcp, ts);
    SAB_LAUNCH_CHECK();
    return SAB_OK;
}

// d_sa: the suffix array of d_s (n >= 1) from the construction; d_work: its workspace of sab_saca_workspace_bytes(n),
// dead by now.  The factors are left at *d_pos / *d_len inside the workspace, *z of them.
static int sab_lz77_parse(SabContext* c, const u8* d_s, u64 n, const u32* d_sa, char* d_work, u32** d_pos, u32** d_len, u64* z) {
    cudaStream_t st = c->stream;
    LzArgs a = {};
    a.n = n;
    a.sa.cnt[0] = a.lcp.cnt[0] = n + 1;
    while (a.sa.cnt[a.sa.top] > 256) {
        a.sa.cnt[a.sa.top + 1] = a.lcp.cnt[a.sa.top + 1] = div_up64(a.sa.cnt[a.sa.top], 256);
        a.lcp.top = ++a.sa.top;
    }
    const u64 chunks = div_up64(n, SAB_LZ_CHUNK), blocks = div_up64(n, SAB_LZ_BLOCK);
    const size_t arr = ((size_t)n + 2) * sizeof(u32);
    char* w = d_work;
    auto take = [&](size_t bytes) {
        char* p = w;
        w += sab_align_up(bytes, 256);
        return p;
    };
    u32* isa = (u32*)take(arr);  // g0, then pos
    u32* lcp = (u32*)take(arr);  // g1, then len
    a.lpf = (u32*)take(arr);     // the lists of long comparisons of the LCP step, then LPF
    a.src = (u32*)take(arr);
    u32* plcp = (u32*)take(arr);
    u8* flag = (u8*)take((size_t)n);
    u32* e0 = (u32*)take((size_t)chunks * 4);
    u32* e1 = (u32*)take((size_t)blocks * 4);
    a.sa.lvl[0] = d_sa;
    a.lcp.lvl[0] = lcp;
    for (u32 k = 1; k <= a.sa.top; ++k) {
        a.sa.lvl[k] = (u32*)take((size_t)a.sa.cnt[k] * 4);
        a.lcp.lvl[k] = (u32*)take((size_t)a.sa.cnt[k] * 4);
    }
    if ((size_t)(w - d_work) > sab_saca_workspace_bytes(n)) {
        sab_set_error("sab200_lz77: %zu bytes of scratch, the construction leaves %zu", (size_t)(w - d_work), sab_saca_workspace_bytes(n));
        return SAB_ERR_INTERNAL;
    }

    SAB_LAUNCH(lcp_isa_kernel, (unsigned)div_up64(n + 1, 256), 256, 0, st, d_sa, n + 1, isa);
    SAB_LAUNCH_CHECK();
    // (n + 2) / 4 list entries per array: the long comparisons number at most 2 n log2(n) / SAB_LZ_CMP <= n / 4
    SAB_TRY(sab_lz_lcp(c, d_s, n, d_sa, isa, plcp, (LzLong*)a.lpf, (LzLong*)a.src, (n + 2) / 4, lcp));
    for (u32 k = 1; k <= a.sa.top; ++k) {
        const unsigned g = (unsigned)div_up64(a.sa.cnt[k] * 32, 256);
        SAB_LAUNCH(lcp_block_min_kernel, g, 256, 0, st, a.sa.lvl[k - 1], a.sa.cnt[k - 1], (u32*)a.sa.lvl[k], a.sa.cnt[k]);
        SAB_LAUNCH_CHECK();
        SAB_LAUNCH(lcp_block_min_kernel, g, 256, 0, st, a.lcp.lvl[k - 1], a.lcp.cnt[k - 1], (u32*)a.lcp.lvl[k], a.lcp.cnt[k]);
        SAB_LAUNCH_CHECK();
    }
    SAB_LAUNCH(lz_lpf_kernel, (unsigned)div_up64(div_up64(n, SAB_LZ_ROWS) * 32, 256), 256, 0, st, a);
    SAB_LAUNCH_CHECK();

    u32 *g0 = isa, *g1 = lcp;
    SAB_LAUNCH(lz_exit0_kernel, (unsigned)div_up64(chunks, 256), 256, 0, st, (const u32*)a.lpf, n, g0);
    SAB_LAUNCH_CHECK();
    SAB_LAUNCH(lz_exit1_kernel, (unsigned)blocks, SAB_LZ_EXIT_THREADS, 0, st, (const u32*)g0, n, g1);
    SAB_LAUNCH_CHECK();
    SAB_CUDA_TRY(cudaMemsetAsync(e1, 0xff, (size_t)blocks * 4, st));
    SAB_CUDA_TRY(cudaMemsetAsync(e0, 0xff, (size_t)chunks * 4, st));
    SAB_CUDA_TRY(cudaMemsetAsync(flag, 0, (size_t)n, st));
    SAB_LAUNCH(lz_walk_top_kernel, 1, 1, 0, st, (const u32*)g1, n, e1);
    SAB_LAUNCH_CHECK();
    SAB_LAUNCH(lz_walk_block_kernel, (unsigned)div_up64(blocks, 256), 256, 0, st, (const u32*)g0, (const u32*)e1, n, e0);
    SAB_LAUNCH_CHECK();
    SAB_LAUNCH(lz_walk_chunk_kernel, (unsigned)div_up64(chunks, 256), 256, 0, st, (const u32*)a.lpf, (const u32*)e0, n, flag);
    SAB_LAUNCH_CHECK();

    const u64 tiles = div_up64(n, SAB_SCAN_TILE);
    SAB_TRY(sab_ensure_scan(c, (size_t)tiles));
    TileState<u32> ts = sab_tile_state<u32>(c, tiles);
    u32* d_z = &c->scratch->lz[0];
    *d_pos = g0;  // g0 and g1 are dead once the chunk walks have run
    *d_len = g1;
    SAB_LAUNCH(lz_compact_kernel, (unsigned)tiles, SAB_SCAN_THREADS, 0, st, d_s, (const u8*)flag, (const u32*)a.lpf, (const u32*)a.src,
               n, *d_pos, *d_len, n, d_z, ts);
    SAB_LAUNCH_CHECK();
    u32 zz;
    SAB_TRY(sab_read_u32(c, d_z, 1, &zz));
    *z = zz;
    return SAB_OK;
}

// ------------------------------------------------------------------ decoder
struct LzSumOp {
    __device__ __forceinline__ u64 operator()(u64 a, u64 b) const { return a + b; }
};

__device__ __forceinline__ u64 lz_warp_incl_sum64(u64 v) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u64 o = __shfl_up_sync(SAB_FULL, v, d);
        if ((int)lane_id() >= d) v += o;
    }
    return v;
}

#define SAB_LZ_BAD_LITERAL 1u  // a literal with pos > 255
#define SAB_LZ_BAD_SOURCE 2u   // a copy whose source does not lie before its start

// The factor starts b_t = sum of max(1, len) over the factors before t into start[] (valid when the total is n), the
// rule flags into info[0] and the total into info[1..2] (little-endian u64).  Tiles as lz_compact_kernel.
__global__ void __launch_bounds__(SAB_SCAN_THREADS)
lz_dec_scan_kernel(const u32* __restrict__ pos, const u32* __restrict__ len, u64 z, u32* __restrict__ start, u32* __restrict__ info,
                   TileState<u64> st) {
    const u32 tile = blockIdx.x, lane = lane_id();
    const u64 base = (u64)tile * SAB_SCAN_TILE;
    const u64 wbase = base + (u64)warp_id() * SAB_WCHUNK;
    u32 wt[SAB_SCAN_ITEMS];
    u64 mine = 0;
#pragma unroll
    for (int k = 0; k < SAB_SCAN_ITEMS; ++k) {
        const u64 t = wbase + (u64)k * 32 + lane;
        const u32 l = t < z ? len[t] : 0u;
        wt[k] = t < z ? (l ? l : 1u) : 0u;
        mine += wt[k];
    }
    mine = warp_reduce_pod<u64, LzSumOp>(mine, LzSumOp());
    u64 wpre, total;
    warp_aggregates<u64, LzSumOp>(mine, LzSumOp(), 0ull, wpre, total);
    const u64 prefix = tile_exclusive_prefix<u64, LzSumOp>(st, tile, total, LzSumOp(), 0ull);
    u64 run = prefix + wpre;
    u32 bad = 0;
#pragma unroll
    for (int k = 0; k < SAB_SCAN_ITEMS; ++k) {
        const u64 t = wbase + (u64)k * 32 + lane;
        const u64 incl = lz_warp_incl_sum64(wt[k]);
        const u64 b = run + incl - wt[k];
        if (t < z) {
            const u32 l = len[t], p = pos[t];
            if (l == 0 && p > 255) bad |= SAB_LZ_BAD_LITERAL;
            if (l != 0 && p >= b) bad |= SAB_LZ_BAD_SOURCE;
            start[t] = (u32)b;
        }
        run += __shfl_sync(SAB_FULL, incl, 31);
    }
    if (bad) atomicOr(&info[0], bad);
    if (threadIdx.x == 0 && base + SAB_SCAN_TILE >= z) {  // last tile
        const u64 sum = prefix + total;
        info[1] = (u32)sum;
        info[2] = (u32)(sum >> 32);
    }
}

// Byte x of the output, in factor t (the last start <= x): a literal writes its byte and points at itself, a copy
// points at its source byte.
__global__ void __launch_bounds__(256)
lz_dec_point_kernel(const u32* __restrict__ pos, const u32* __restrict__ len, const u32* __restrict__ start, u64 z, u64 n,
                    u32* __restrict__ ptr, u8* __restrict__ out) {
    const u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n) return;
    u64 lo = 0, hi = z;
    while (hi - lo > 1) {
        const u64 mid = (lo + hi) >> 1;
        if (start[mid] <= x) lo = mid;
        else hi = mid;
    }
    if (len[lo] == 0) {
        ptr[x] = (u32)x;
        out[x] = (u8)pos[lo];
    } else {
        ptr[x] = pos[lo] + (u32)(x - start[lo]);
    }
}

// One round of pointer jumping in place: a value read is an ancestor on x's chain whether or not its thread has
// written yet, so the bound of the round count holds.  *changed is set when a pointer moved.
__global__ void __launch_bounds__(256) lz_dec_jump_kernel(u32* ptr, u64 n, u32* __restrict__ changed) {
    const u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n) return;
    const u32 p = ptr[x], q = ptr[p];
    if (q != p) {
        ptr[x] = q;
        *changed = 1;
    }
}

// Every copied byte from the literal at the root of its chain (roots are literals, written by lz_dec_point_kernel)
__global__ void __launch_bounds__(256) lz_dec_fill_kernel(const u32* __restrict__ ptr, u64 n, u8* out) {
    const u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n) return;
    const u32 p = ptr[x];
    if (p != x) out[x] = out[p];
}

// device bytes the decoder needs on top of its input and output
static inline size_t sab_lz77_decode_workspace_bytes(u64 z, u64 n) {
    return sab_align_up(((size_t)z + 1) * 4, 256) + sab_align_up(((size_t)n + 1) * 4, 256);
}

// d_pos, d_len: z >= 1 factors; 1 <= z <= n; d_out receives n bytes.  The workspace is carved from the bottom of the
// arena.  Returns SAB_ERR_ARGS, before anything is written to d_out, when the factors are not a parse of n bytes.
static int sab_lz77_decode_run(SabContext* c, const u32* d_pos, const u32* d_len, u64 z, u64 n, u8* d_out) {
    cudaStream_t st = c->stream;
    u32 *start, *ptr;
    SAB_TRY(sab_arena_carve(c, {{&start, ((size_t)z + 1) * 4}, {&ptr, ((size_t)n + 1) * 4}}));
    u32* info = &c->scratch->lz[0];
    SAB_CUDA_TRY(cudaMemsetAsync(info, 0, 3 * sizeof(u32), st));
    const u64 tiles = div_up64(z, SAB_SCAN_TILE);
    SAB_TRY(sab_ensure_scan(c, (size_t)tiles));
    TileState<u64> ts = sab_tile_state<u64>(c, tiles);
    SAB_LAUNCH(lz_dec_scan_kernel, (unsigned)tiles, SAB_SCAN_THREADS, 0, st, d_pos, d_len, z, start, info, ts);
    SAB_LAUNCH_CHECK();
    u32 got[3];
    SAB_TRY(sab_read_u32(c, info, 3, got));
    const u64 total = (u64)got[1] | ((u64)got[2] << 32);
    if (total != n) {
        sab_set_error("sab200_lz77_decode: the factor lengths (max(1, len) each) sum to %llu, not to n = %llu",
                      (unsigned long long)total, (unsigned long long)n);
        return SAB_ERR_ARGS;
    }
    if (got[0] & SAB_LZ_BAD_LITERAL) {
        sab_set_error("sab200_lz77_decode: a literal factor (len = 0) has pos > 255");
        return SAB_ERR_ARGS;
    }
    if (got[0] & SAB_LZ_BAD_SOURCE) {
        sab_set_error("sab200_lz77_decode: a copy factor has its source at or after its own start");
        return SAB_ERR_ARGS;
    }
    const unsigned g = (unsigned)div_up64(n, 256);
    SAB_LAUNCH(lz_dec_point_kernel, g, 256, 0, st, d_pos, d_len, (const u32*)start, z, n, ptr, d_out);
    SAB_LAUNCH_CHECK();
    u32* changed = &c->scratch->lz[3];
    for (int round = 0;; ++round) {
        if (round > sab_ceil_log2_u64(n) + 1) {
            sab_set_error("sab200_lz77_decode: pointer jumping did not settle after %d rounds", round);
            return SAB_ERR_INTERNAL;
        }
        SAB_CUDA_TRY(cudaMemsetAsync(changed, 0, sizeof(u32), st));
        SAB_LAUNCH(lz_dec_jump_kernel, g, 256, 0, st, ptr, n, changed);
        SAB_LAUNCH_CHECK();
        u32 ch;
        SAB_TRY(sab_read_u32(c, changed, 1, &ch));
        if (!ch) break;
    }
    SAB_LAUNCH(lz_dec_fill_kernel, g, 256, 0, st, (const u32*)ptr, n, d_out);
    SAB_LAUNCH_CHECK();
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    return SAB_OK;
}
