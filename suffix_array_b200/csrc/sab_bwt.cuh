// sab_bwt.cuh -- Burrows-Wheeler transform and its inverse (include/sab200.h "BWT").
//
// Rows are the n+1 entries of the suffix array with sa[0] = n; L[j] = s[sa[j]-1], and L[p] = '$' at the primary
// index p (sa[p] = 0).  The transform U is L without row p.
//
// Forward: the construction as it is (sab_saca.cuh), then bwt_gather_kernel over the n+1 rows (coalesced sa[j], one
// random text byte) into L, which lives in the dead construction workspace; the caller moves L[0, p) and L[p+1, n+1).
//
// Inverse: psi(row of suffix k) = row of suffix k+1, F = first column, s[k] = F[psi^k(p)].
//   1. bwt_widen_kernel + ONE stable radix pass on bits [32, 40) of (U[u] << 32 | u): sorted record q-1 is row q >= 1,
//      carrying F[q] (bits 32..39) and its source u; psi(q) = u < p ? u : u + 1 (U skips row p), psi(0) = p.
//      A step of a walk is one random 8-byte read.
//   2. list ranking by sampled walks: the sample rows (bwt_is_sample) are compacted into an ascending list, every
//      sample walks psi to the next sample (bwt_walk_kernel), pointer jumping over the samples gives each its
//      distance to row 0, and every sample writes its segment of the text from position n - dist.
#pragma once
#include "sab_saca.cuh"

// ------------------------------------------------------------------ forward
// L[j] for the n+1 rows; the row holding the whole text (sa[j] = 0) writes '$' and its index to *primary
__global__ void __launch_bounds__(256)
bwt_gather_kernel(const u8* __restrict__ s, const u32* __restrict__ sa, u64 rows, u8* __restrict__ L, u32* __restrict__ primary) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= rows) return;
    const u32 v = sa[j];
    if (v == 0) {
        L[j] = '$';
        *primary = (u32)j;
    } else {
        L[j] = s[v - 1];
    }
}

// d_sa: the n+1 entries of the suffix array of d_s; L receives n+1 bytes; *primary the row of suffix 0
static int sab_bwt_gather(SabContext* c, const u8* d_s, u64 n, const u32* d_sa, u8* d_L, u64* primary) {
    u32* d_p = &c->scratch->bwt[0];
    SAB_LAUNCH(bwt_gather_kernel, (unsigned)div_up64(n + 1, 256), 256, 0, c->stream, d_s, d_sa, n + 1, d_L, d_p);
    SAB_LAUNCH_CHECK();
    u32 p;
    SAB_TRY(sab_read_u32(c, d_p, 1, &p));
    *primary = p;
    return SAB_OK;
}

// ------------------------------------------------------------------ inverse
// Mean rows per sample.  m = (n+1)/256 walks keep over a million of them in flight from n = 256 MiB on, several
// times the threads a B200 holds resident, so the dependent random reads of the walks overlap.  The longest of m
// walks is about 256 * ln(m) steps (under 4000 at n = 2^32), the tail of walk 1 and walk 2.  Pointer jumping costs
// ceil(log2 m) launches over m records, and the sample arrays take under 0.1 byte per row.
#define SAB_BWT_SAMPLE 256

__host__ __device__ __forceinline__ u64 sab_splitmix64(u64 x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// A row is a sample by a hash of its index, which does not depend on the text: stride sampling would leave long
// unsampled stretches of the walk on periodic texts.  Row 0 (the end of the walk) and row p (its start) always are.
__device__ __forceinline__ bool bwt_is_sample(u64 r, u32 p) {
    return r == 0 || r == p || sab_splitmix64(r) < ~0ull / SAB_BWT_SAMPLE;
}

// capacity of the sample list: about twice the expected count; the compaction reports an overflow instead of writing
static inline u64 sab_bwt_sample_cap(u64 n) { return (n + 1) / SAB_BWT_SAMPLE * 2 + 4096; }

__global__ void __launch_bounds__(256) bwt_widen_kernel(const u8* __restrict__ U, u64 n, u64* __restrict__ rec) {
    const u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < n) rec[u] = ((u64)U[u] << 32) | u;
}

// Sample rows of [0, rows) in ascending order into list[0, cap); out[0] = their count, out[1] = the list position of
// row p.  Warp-striped tiles chained by the decoupled look-back of sab_scan.cuh.
__global__ void __launch_bounds__(SAB_SCAN_THREADS)
bwt_sample_list_kernel(u64 rows, u32 p, u32* __restrict__ list, u64 cap, u32* __restrict__ out, TileState<u32> st) {
    const u32 tile = blockIdx.x, lane = lane_id();
    const u64 base = (u64)tile * SAB_SCAN_TILE;
    const u64 wbase = base + (u64)warp_id() * SAB_WCHUNK;
    u32 sb[SAB_SCAN_ITEMS];
    u32 mine = 0;
#pragma unroll
    for (int k = 0; k < SAB_SCAN_ITEMS; ++k) {
        const u64 j = wbase + (u64)k * 32 + lane;
        sb[k] = __ballot_sync(SAB_FULL, j < rows && bwt_is_sample(j, p));
        mine += (u32)__popc(sb[k]);
    }
    u32 wpre, total;
    warp_aggregates<u32, CountOp>(mine, CountOp(), 0u, wpre, total);
    const u32 prefix = tile_exclusive_prefix<u32, CountOp>(st, tile, total, CountOp(), 0u);
    u32 run = prefix + wpre;
#pragma unroll
    for (int k = 0; k < SAB_SCAN_ITEMS; ++k) {
        const u64 j = wbase + (u64)k * 32 + lane;
        if ((sb[k] >> lane) & 1u) {
            const u32 pos = run + (u32)__popc(sb[k] & lanemask_lt());
            if (pos < cap) list[pos] = (u32)j;
            if (j == p) out[1] = pos;
        }
        run += (u32)__popc(sb[k]);
    }
    if (threadIdx.x == 0 && base + SAB_SCAN_TILE >= rows) out[0] = prefix + total;  // last tile
}

// One step of the walk from row r >= 1: F[r] and psi(r) from sorted record r-1
__device__ __forceinline__ u32 bwt_step(const u64* __restrict__ rec, u32 p, u32 r, u8* f) {
    const u64 x = rec[r - 1];
    *f = (u8)(x >> 32);
    const u32 u = (u32)x;
    return u < p ? u : u + 1u;
}

// Termination: psi is a permutation (it comes out of a stable sort), so a walk from sample r meets a sample at the
// latest when it returns to r itself, after at most n+1 steps, whatever bytes U holds.  No step cap is needed, and a
// transform of no text cannot hang the GPU.  U is a valid transform iff psi is one cycle, i.e. iff the walk from p
// reaches row 0 after exactly n steps; the driver checks that (dist(p) = n) before walk 2 writes anything.
//
// WRITE = false (walk 1): hop[i] = (steps to the next sample) << 32 | its list position.  Row 0 is the end of the
//   ranking: it points at itself with distance 0, so pointer jumping leaves it fixed.
// WRITE = true (walk 2): hop[i] holds dist(row) << 32; sample i != 0 writes F along its walk from text position
//   n - dist(row) until the next sample.
template <bool WRITE>
__global__ void __launch_bounds__(256)
bwt_walk_kernel(const u64* __restrict__ rec, u32 p, u64 n, const u32* __restrict__ list, u64 m, u64* __restrict__ hop,
                u8* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const u32 r0 = list[i];
    if (r0 == 0) {
        if (!WRITE) hop[i] = 0;
        return;
    }
    u32 r = r0;
    u8 f;
    if (WRITE) {
        u8* dst = out + (n - (hop[i] >> 32));
        do {
            r = bwt_step(rec, p, r, &f);
            *dst++ = f;
        } while (!bwt_is_sample(r, p));
    } else {
        u32 steps = 0;
        do {
            r = bwt_step(rec, p, r, &f);  // r >= 1 here: row 0 is a sample
            ++steps;
        } while (!bwt_is_sample(r, p));
        u64 lo = 0, hi = m;  // the next sample's list position
        while (hi - lo > 1) {
            const u64 mid = (lo + hi) >> 1;
            if (list[mid] <= r) lo = mid;
            else hi = mid;
        }
        hop[i] = ((u64)steps << 32) | lo;
    }
}

// one round of pointer jumping: distances add up (mod 2^32: only the chain into row 0 is read, and there they are
// at most n), pointers double
__global__ void __launch_bounds__(256) bwt_jump_kernel(const u64* __restrict__ in, u64 m, u64* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const u64 a = in[i], b = in[(u32)a];
    out[i] = ((u64)((u32)(a >> 32) + (u32)(b >> 32)) << 32) | (u32)b;
}

// device bytes the inverse needs on top of its input and output
static inline size_t sab_inverse_bwt_workspace_bytes(u64 n) {
    const size_t N = (size_t)n + 8, cap = (size_t)sab_bwt_sample_cap(n);
    return 2 * sab_align_up(N * 8, 256) + 2 * sab_align_up(N * 4, 256) + sab_align_up(cap * 4, 256) + 2 * sab_align_up(cap * 8, 256);
}

// d_u: the n >= 1 bytes of the transform, 1 <= p <= n; d_out receives the n bytes of the text.  The workspace is
// carved from the bottom of the arena.  Returns SAB_ERR_ARGS, before anything is written to d_out, when U is not the
// transform of any text.
static int sab_inverse_bwt_run(SabContext* c, const u8* d_u, u64 n, u32 p, u8* d_out) {
    cudaStream_t st = c->stream;
    c->profiling = false;  // the radix pass must not leave events behind for the next construction's statistics
    const u64 cap = sab_bwt_sample_cap(n);
    SortBuffers<u64> buf;
    u32* list;
    u64 *hop[2];
    SAB_TRY(sab_arena_carve(c, {{&buf.k[0], ((size_t)n + 8) * 8}, {&buf.k[1], ((size_t)n + 8) * 8}, {&buf.v[0], ((size_t)n + 8) * 4},
                                {&buf.v[1], ((size_t)n + 8) * 4}, {&list, (size_t)cap * 4}, {&hop[0], (size_t)cap * 8},
                                {&hop[1], (size_t)cap * 8}}));
    buf.cur = 0;
    SAB_LAUNCH(bwt_widen_kernel, (unsigned)div_up64(n, 256), 256, 0, st, d_u, n, buf.k[0]);
    SAB_LAUNCH_CHECK();
    u32 passes;
    SAB_TRY(sab_radix_sort<u64>(c, buf, n, 32, 40, /*iota=*/true, &passes));
    const u64* rec = buf.k[buf.cur];

    const u64 rows = n + 1, tiles = div_up64(rows, SAB_SCAN_TILE);
    SAB_TRY(sab_ensure_scan(c, (size_t)tiles));
    TileState<u32> ts = sab_tile_state<u32>(c, tiles);
    u32* d_out2 = &c->scratch->bwt[0];
    SAB_LAUNCH(bwt_sample_list_kernel, (unsigned)tiles, SAB_SCAN_THREADS, 0, st, rows, p, list, cap, d_out2, ts);
    SAB_LAUNCH_CHECK();
    u32 got[2];
    SAB_TRY(sab_read_u32(c, d_out2, 2, got));
    const u64 m = got[0], at_p = got[1];
    if (m > cap) {
        sab_set_error("sab200_inverse_bwt: %llu sample rows, room for %llu", (unsigned long long)m, (unsigned long long)cap);
        return SAB_ERR_INTERNAL;
    }
    const unsigned blocks = (unsigned)div_up64(m, 256);
    SAB_LAUNCH(bwt_walk_kernel<false>, blocks, 256, 0, st, rec, p, n, (const u32*)list, m, hop[0], (u8*)nullptr);
    SAB_LAUNCH_CHECK();
    int cur = 0;
    for (int k = sab_ceil_log2_u64(m); k > 0; --k, cur ^= 1) {
        SAB_LAUNCH(bwt_jump_kernel, blocks, 256, 0, st, (const u64*)hop[cur], m, hop[cur ^ 1]);
        SAB_LAUNCH_CHECK();
    }
    // Row 0 and row p lie on one cycle (psi(0) = p), so dist(p) is exact: the length of that cycle minus one.
    u32 dist_p[2];
    SAB_TRY(sab_read_u32(c, (const u32*)(hop[cur] + at_p), 2, dist_p));  // little-endian: word 1 is the distance
    if (dist_p[1] != n) {
        sab_set_error("sab200_inverse_bwt: not the Burrows-Wheeler transform of any text (the walk from the primary index "
                      "returns to row 0 after %u of %llu rows)", dist_p[1] + 1u, (unsigned long long)rows);
        return SAB_ERR_ARGS;
    }
    SAB_LAUNCH(bwt_walk_kernel<true>, blocks, 256, 0, st, rec, p, n, (const u32*)list, m, hop[cur], d_out);
    SAB_LAUNCH_CHECK();
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    return SAB_OK;
}
