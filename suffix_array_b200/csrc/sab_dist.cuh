// sab_dist.cuh -- multi-GPU suffix-array construction: one rank per GPU, distributed sample sort of the packed
// keys followed by prefix doubling with a fixed number of exchange steps per round (include/sab200.h,
// "multi-GPU").  The reference has nothing distributed (SURVEY.md 2.1); this is the sharded form of the same
// saca() (/root/reference/src/saca.rs:9-15).
//
//   rank g of P owns text positions [g*B, (g+1)*B) and the rank[] entries the RankLayout gives it
//   1  byte histogram                       all_reduce   -> common code table / key shape (sab_plan_alphabet)
//   2  keys of own positions; splitters     all_gather   of 2048 sampled keys per rank
//   3  partition by destination (onesweep pass, digit = #splitters <= key)         all_to_all (key, i)
//   4  local radix sort -> a contiguous slice of the suffix array; equal keys share a destination, so groups
//      never straddle GPUs and all re-ranking is local
//   5  init_ranks: slice of sa[], active list (r1, i), bucket directory over the slice's sorted keys
//   6  inverse suffix array at the owners: LAZY when at most a quarter of the suffixes is active (only their
//      ranks travel; a request that finds EMPTY is a suffix that was unique after step 4: the owner packs its
//      key from its text shard, the key travels to the slice that holds it and its rank comes back), else all
//      ranks travel and rank[] is dealt block-cyclically (any region of the text is spread over all owners)
//   7  rounds h = k, 2k, ...:  requests i+h -> owners, answers back                2 x all_to_all (+2 lazy)
//      the list keeps its order (answers are placed by list position), so the in-group sort of the
//      single-GPU path applies; re-rank; changed ranks -> owners                     all_to_all
//
// Every step is enqueued on the rank's library stream; the host only waits where it needs a count.
#pragma once
#include <unistd.h>

#include <algorithm>
#include <thread>

#include "sab_comm.cuh"
#include "sab_saca.cuh"

// ------------------------------------------------------------------ kernels
// d_n != null: the record count lives on the device (the grid is sized for the bound n)
template <typename KeyT, typename DigitOp>
__global__ void __launch_bounds__(256) digit_count_kernel(const KeyT* __restrict__ keys, u64 n, const u32* __restrict__ d_n, DigitOp dop,
                                                          u64* __restrict__ counts) {
    SAB_SHARED_ARRAY(u32, s_c, 256);
    s_c[threadIdx.x] = 0;
    if (d_n) n = *d_n;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) atomicAdd(&s_c[dop(keys[i])], 1u);
    __syncthreads();
    const u32 c = s_c[threadIdx.x];
    if (c) atomicAdd((unsigned long long*)&counts[threadIdx.x], (unsigned long long)c);
}

// One block of 256 threads: gbase[] = exclusive prefix of the 256 bin counts (record offsets of the partition
// pass), and the row this rank contributes to the count exchange: [P counts | nd device-side u32 extras].
__global__ void __launch_bounds__(256)
count_row_kernel(const u64* __restrict__ cnt, u64* __restrict__ gbase, int P, const u32* __restrict__ extra32, int nd,
                 u64* __restrict__ row) {
    SAB_SHARED_ARRAY(u64, s_v, 256);
    const u32 t = threadIdx.x;
    const u64 mine = cnt[t];
    s_v[t] = mine;
    __syncthreads();
    for (u32 off = 1; off < 256; off <<= 1) {
        const u64 v = t >= off ? s_v[t - off] : 0ull;
        __syncthreads();
        s_v[t] += v;
        __syncthreads();
    }
    gbase[t] = s_v[t] - mine;
    if ((int)t < P) row[t] = mine;
    else if ((int)t < P + nd) row[t] = extra32[t - P];
}

__global__ void hist_widen_kernel(const u32* __restrict__ h32, u64* __restrict__ h64) { h64[threadIdx.x] = h32[threadIdx.x]; }

// out[j] = keys[j * step] for the first min(S, ceil(count / step)) samples; out[S] = how many
__global__ void sample_keys_kernel(const u64* __restrict__ keys, u64 count, u64 step, u32 S, u64* __restrict__ out) {
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    const u64 have = count ? (count + step - 1) / step : 0;
    const u32 ns = have < S ? (u32)have : S;
    if (j < ns) out[j] = keys[(u64)j * step];
    if (j == 0) out[S] = ns;
}

// local slot of position q on its owner: q - lo under the block layout (lay.cyc = 0), lay.slot() otherwise
__global__ void dist_scatter_kernel(const u32* __restrict__ pos, const u32* __restrict__ val, u64 n, u32 lo, RankLayout lay,
                                    u32* __restrict__ rank_local) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rank_local[lay.cyc ? lay.slot(pos[i], 0) : (u64)(pos[i] - lo)] = val[i];
}
__global__ void dist_gather_kernel(const u32* __restrict__ pos, u64 n, u32 add, u32 lo, RankLayout lay,
                                   const u32* __restrict__ rank_local, u32* __restrict__ out) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const u64 q = (u64)pos[i] + add;
        out[i] = rank_local[lay.cyc ? lay.slot(q, 0) : q - lo];
    }
}
// The requests left in owner order; the answers come back in the same order and return to the LIST position
// of their record: key64[pos[t]] = (r1[pos[t]] << 32) | r2[t].  The list stays grouped by r1.
__global__ void dist_place_keys_kernel(const u32* __restrict__ r1, const u32* __restrict__ pos, const u32* __restrict__ r2, u64 m,
                                       u64* __restrict__ key64) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < m) {
        const u32 p = pos[t];
        key64[p] = ((u64)r1[p] << 32) | r2[t];
    }
}

// SA entries that became final on a GPU that does not hold their position (rebalanced lists): sa[pos] = idx
__global__ void dist_store_sa_kernel(const u32* __restrict__ pos, const u32* __restrict__ idx, u64 n, u32 sa_off,
                                     u32* __restrict__ sa_local) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sa_local[pos[i] - sa_off] = idx[i];
}
// For every cut c = cuts[j] inside the rank-sorted list r1[0..m) (j = blockIdx.x / blocks_per_cut): the smallest
// p in [c + woff, c + woff + window) with r1[p] != r1[c-1] (atomicMin into out[j], pre-set to ~0).
__global__ void find_boundary_kernel(const u32* __restrict__ r1, u64 m, const u64* __restrict__ cuts, u32 blocks_per_cut, u64 woff,
                                     u64 window, unsigned long long* __restrict__ out) {
    const u32 j = blockIdx.x / blocks_per_cut;
    const u64 c = cuts[j];
    if (c == 0 || c >= m) return;
    const u64 t = (u64)(blockIdx.x % blocks_per_cut) * blockDim.x + threadIdx.x;
    const u64 p = c + woff + t;
    if (t < window && p < m && r1[p] != r1[c - 1]) atomicMin(&out[j], (unsigned long long)p);
}

// ---- peer-to-peer rounds: the arenas of all GPUs are mapped into every rank (sab_peers_update), so a SMALL round
// needs no exchange step at all: the gather loads rank[i+h] straight from the owner GPU over NVLink (and resolves
// an EMPTY slot through the owner's text, the slice's directory and sorted keys, all remote loads), the changed
// ranks are stored straight into the owner's block.  Two stream-ordered all_reduces per round order the phases
// (every rank has finished reading before anybody writes, and vice versa) and carry the survivor counts.
struct P2PTable {
    u32* rank_local[SAB_MAX_RANKS];
    const u8* text[SAB_MAX_RANKS];
    const u64* sorted[SAB_MAX_RANKS];
    const u32* dir[SAB_MAX_RANKS];  // pre-shifted: indexed by key >> dir_shift
    u64 R[SAB_MAX_RANKS];
    u64 n_rel[SAB_MAX_RANKS];       // readable text bytes of the shard (own positions + halo)
    u32 sa_off[SAB_MAX_RANKS];
};
__global__ void __launch_bounds__(256)
dist_gather_p2p_kernel(const u32* __restrict__ r1, const u32* __restrict__ idx, u64 m, u32 h, RankLayout lay, P2PTable pt, int lazy,
                       const u16* __restrict__ lut, u32 base, int k, int dir_shift, SplitterDigit sd, u64* __restrict__ key64) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const u64 q = (u64)idx[t] + h;
    const u32 o = lay.owner(q);
    const u64 slot = lay.slot(q, o);
    u32 r2 = pt.rank_local[o][slot];
    if (lazy && r2 == SAB_RANK_EMPTY) {  // block layout: the owner of q holds text position q at offset slot
        const u64 key = pack_key_at(pt.text[o], pt.n_rel[o], lut, base, k, slot);
        const u32 d = sd(key);
        r2 = pt.sa_off[d] + (u32)sorted_key_position(pt.sorted[d], pt.R[d], pt.dir[d], dir_shift, key);
        pt.rank_local[o][slot] = r2;  // memoise; racing writers store the same value
    }
    key64[t] = ((u64)r1[t] << 32) | r2;
}
// rank[idx[t]] = val[t] on the owner of idx[t]; idx == 0xFFFFFFFF marks "nothing to write"
__global__ void __launch_bounds__(256)
dist_scatter_p2p_kernel(const u32* __restrict__ idx, const u32* __restrict__ val, u64 cnt, RankLayout lay, P2PTable pt) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    const u32 i = idx[t];
    if (i == 0xffffffffu) return;
    const u32 o = lay.owner(i);
    pt.rank_local[o][lay.slot(i, o)] = val[t];
}
__global__ void put_u64_kernel(u64* dst, const u32* src32) { *dst = *src32; }

// ---- lazy inverse suffix array, distributed (see the file header, step 6)
__global__ void __launch_bounds__(256)
dist_lazy_collect_kernel(const u32* __restrict__ q, const u32* __restrict__ ans, u64 count, u32 h, u64 shard_lo,
                         const u8* __restrict__ text, u64 n_rel, const u16* __restrict__ lut, u32 base, int k,
                         u64* __restrict__ keys_out, u32* __restrict__ slot_out, u32* __restrict__ counter) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count || ans[t] != SAB_RANK_EMPTY) return;
    const u32 p = atomicAdd(counter, 1u);
    keys_out[p] = pack_key_at(text, n_rel, lut, base, k, (u64)q[t] + h - shard_lo);
    slot_out[p] = (u32)t;
}
// rank of a suffix that was unique after the initial sort = SA position of its key in this slice
__global__ void __launch_bounds__(256)
dist_lookup_kernel(const u64* __restrict__ sorted, u64 R, const u32* __restrict__ dir, int dir_shift, const u64* __restrict__ keys,
                   u64 count, u32 sa_off, u32* __restrict__ rank_out) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    rank_out[t] = sa_off + (u32)sorted_key_position(sorted, R, dir, dir_shift, keys[t]);
}
__global__ void __launch_bounds__(256)
dist_lazy_fill_kernel(const u32* __restrict__ slot, const u32* __restrict__ rank, u64 count, const u32* __restrict__ q, u32 h,
                      u32 lo, u32* __restrict__ ans, u32* __restrict__ rank_local) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const u32 s = slot[t], r = rank[t];
    ans[s] = r;
    rank_local[(u64)q[s] + h - lo] = r;  // memoised: the next request for this position is answered directly
}

// ------------------------------------------------------------------ host helpers
// Rank g of P owns the text positions [lo, hi), B = ceil(n / P) of them (the last ranks fewer, or none).  Its shard
// holds len readable bytes from lo on: its own positions and SAB200_SHARD_HALO bytes of the next shard, cut at n.
struct ShardBounds {
    u64 B, lo, hi, len;
};
static inline ShardBounds sab_shard_bounds(u64 n, int P, int g) {
    ShardBounds s;
    s.B = n ? div_up64(n, (u64)P) : 1;
    s.lo = (u64)g * s.B < n ? (u64)g * s.B : n;
    s.hi = s.lo + s.B < n ? s.lo + s.B : n;
    s.len = (n - s.lo) < (s.hi - s.lo) + SAB200_SHARD_HALO ? (n - s.lo) : (s.hi - s.lo) + SAB200_SHARD_HALO;
    return s;
}

// Directory shift of the lazy inverse suffix array on a multi-GPU rank.  One GPU uses SAB_DIR_SHIFT = 2; that value
// was measured on one GPU only, so the multi-GPU driver keeps its own.
#define SAB_DIST_DIR_SHIFT 4

// Plans one variable all-to-all with a single host synchronisation:
//   per-destination counts of keys[0..count) (count read from *d_count32 when given; `count` is then its bound)
//   -> exclusive bases of all 256 bins in c->d_gbase (the partition pass of the same records follows)
//   -> row [P counts | nd device u32 extras | nh host u64 extras] all-gathered: rows[s*W + i], W = P + nd + nh
//   -> pl: what this rank sends to / receives from everybody.
template <typename KeyT, typename DigitOp>
static int sab_plan_exchange(sab200_comm* cm, SabContext* c, const KeyT* d_keys, u64 count, const u32* d_count32, DigitOp dop,
                             const u32* d_extra32, int nd, const u64* h_extra, int nh, A2APlan* pl, u64* rows) {
    cudaStream_t st = c->stream;
    const int P = cm->P, W = P + nd + nh;
    u64* d_cnt = c->d_ghist;  // 256 x u64 scratch
    SAB_CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 256 * sizeof(u64), st));
    if (count) {
        SAB_LAUNCH((digit_count_kernel<KeyT, DigitOp>), sab_grid(c, count, 256 * 16, 8), 256, 0, st, d_keys, count, d_count32, dop, d_cnt);
        SAB_LAUNCH_CHECK();
        c->stats.kernel_launches++;
    }
    SAB_LAUNCH(count_row_kernel, 1, 256, 0, st, (const u64*)d_cnt, c->d_gbase, P, d_extra32, nd, cm->d_small);
    SAB_LAUNCH_CHECK();
    if (nh) {
        u64* h = cm->h_small + 32;  // pinned staging (rows come back at h_small + 64)
        for (int i = 0; i < nh; ++i) h[i] = h_extra[i];
        SAB_CUDA_TRY(cudaMemcpyAsync(cm->d_small + P + nd, h, (size_t)nh * sizeof(u64), cudaMemcpyHostToDevice, st));
    }
    u64 rows_[SAB_MAX_RANKS * 32];
    u64* rr = rows ? rows : rows_;
    SAB_TRY(sab_comm_gather_rows(cm, st, W, rr));
    pl->stotal = pl->rtotal = 0;
    for (int d = 0; d < P; ++d) {
        pl->scount[d] = rr[(size_t)cm->rank * W + d];
        pl->rcount[d] = rr[(size_t)d * W + cm->rank];
        pl->stotal += pl->scount[d];
        pl->rtotal += pl->rcount[d];
    }
    return SAB_OK;
}

// Two-ended bump allocator over the context arena: long-lived arrays grow from the bottom, the temporaries of
// a phase / round from the top (released by restoring `hi`).
struct DistArena {
    char* base;
    size_t lo, hi;
    bool ok;
    template <typename T>
    T* bot(size_t count) {
        const size_t o = sab_align_up(lo, 256), e = o + count * sizeof(T);
        if (e > hi) {
            ok = false;
            return nullptr;
        }
        lo = e;
        return (T*)(base + o);
    }
    template <typename T>
    T* top(size_t count) {
        const size_t bytes = sab_align_up(count * sizeof(T), 256);
        if (hi < lo + bytes) {
            ok = false;
            return nullptr;
        }
        hi -= bytes;
        return (T*)(base + hi);
    }
};
#define SAB_ARENA_CHECK(A)                                                                                     \
    do {                                                                                                       \
        if (!(A).ok) {                                                                                         \
            sab_set_error("%s:%d: device arena exhausted (%zu bytes)", __FILE__, __LINE__, c->arena.bytes);    \
            return SAB_ERR_OOM;                                                                                \
        }                                                                                                      \
    } while (0)

// phase timer: CUDA events at the phase boundaries of the rank's stream, read once at the end
struct DistPhases {
    SabContext* c;
    std::vector<std::pair<int, cudaEvent_t> > ev;
    void mark(int phase) {
        cudaEvent_t e = sab_event_get(c);
        cudaEventRecord(e, c->stream);
        ev.push_back(std::make_pair(phase, e));
    }
    void collect(double* phase_ms, double* total_ms) {  // the stream must be idle
        for (size_t i = 0; i + 1 < ev.size(); ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[i].second, ev[i + 1].second);
            if (ev[i].first >= 0 && ev[i].first < SAB200_PHASES) phase_ms[ev[i].first] += ms;
        }
        if (ev.size() >= 2) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev.front().second, ev.back().second);
            *total_ms = ms;
        }
        for (auto& p : ev) c->event_pool.push_back(p.second);
        ev.clear();
    }
};

struct DistResult {
    u32* d_slice;
    u64 slice_len, sa_off;
};

static inline int sab_env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// Arena for a rank that owns B text positions: sized for slices up to ~1.3 B records with all suffixes active,
// capped by the free device memory (a grow-only arena: no cudaMalloc in steady state).
static inline size_t sab_dist_want(u64 B) {
    const size_t recs = (size_t)(B + B / 3) + ((size_t)1 << 20);
    return recs * 72 + ((size_t)256 << 20);
}
static int sab_dist_reserve(SabContext* c, u64 B) {
    size_t want = sab_dist_want(B);
    if (c->arena.bytes >= want || c->arena_want_seen == want) return SAB_OK;  // steady state: no driver call at all
    c->arena_want_seen = want;
    size_t free_b = 0, total_b = 0;
    SAB_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    const size_t avail = (size_t)((double)(free_b + c->arena.bytes) * 0.94);
    if (want > avail) want = avail;
    return sab_arena_reserve(c, want);
}

#ifndef SAB_EMU
// Keeps the peers' arenas mapped into this rank.  rows[s*W + P + {0,1,2,3}] = process id, device, arena address and
// size of rank s (all-gathered with the key counts, so every rank sees the same table and takes the same
// decisions).  A changed entry (first call, re-allocated arena) re-opens the mapping: cudaIpcOpenMemHandle for
// another process, the pointer itself + cudaDeviceEnablePeerAccess inside one process.  Collective.
static int sab_peers_update(sab200_comm* cm, SabContext* c, const u64* rows, int W) {
    const int P = cm->P, g = cm->rank;
    cudaStream_t st = c->stream;
    bool changed = false;
    for (int s = 0; s < P; ++s) {
        const u64* r = rows + (size_t)s * W + P;
        const sab200_comm::Peer& p = cm->peers[s];
        if (p.pid != r[0] || p.dev != r[1] || p.ptr != r[2] || p.bytes != r[3]) changed = true;
    }
    if (!changed) return SAB_OK;  // peers_ok keeps its value
    // 64-byte IPC handles of every arena
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof(mine));
    u64 fail = 0;
    if (cudaIpcGetMemHandle(&mine, c->arena.base) != cudaSuccess) {
        cudaGetLastError();
        fail = 1;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(cm->h_small + 32, &mine, 64);
    SAB_CUDA_TRY(cudaMemcpyAsync(cm->d_small, cm->h_small + 32, 64, cudaMemcpyHostToDevice, st));
    SAB_TRY(sab_comm_all_gather(cm, st, cm->d_small, cm->d_small + 64, 64));
    SAB_CUDA_TRY(cudaMemcpyAsync(cm->h_small + 64, cm->d_small + 64, (size_t)P * 64, cudaMemcpyDeviceToHost, st));
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    const u64 mypid = rows[(size_t)g * W + P];
    for (int s = 0; s < P; ++s) {
        const u64* r = rows + (size_t)s * W + P;
        sab200_comm::Peer& p = cm->peers[s];
        if (p.ipc && p.base) cudaIpcCloseMemHandle(p.base);
        p.pid = r[0];
        p.dev = r[1];
        p.ptr = r[2];
        p.bytes = r[3];
        p.base = nullptr;
        p.ipc = false;
        if (s == g) {
            p.base = c->arena.base;
            continue;
        }
        if (p.pid == mypid) {
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, c->device, (int)p.dev) != cudaSuccess || !can) {
                cudaGetLastError();
                fail = 1;
                continue;
            }
            const cudaError_t e = cudaDeviceEnablePeerAccess((int)p.dev, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) fail = 1;
            cudaGetLastError();
            p.base = (void*)(uintptr_t)p.ptr;
        } else {
            cudaIpcMemHandle_t h;
            memcpy(&h, (const char*)(cm->h_small + 64) + (size_t)s * 64, 64);
            void* base = nullptr;
            if (cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                fail = 1;
                continue;
            }
            p.base = base;
            p.ipc = true;
        }
    }
    SAB_TRY(sab_comm_sum_u64(cm, st, &fail, 1));
    cm->peers_ok = fail == 0;
    return SAB_OK;
}
#endif

// Phases of a construction: the indices of sab200_dist_stats::phase_ms (include/sab200.h); PH_END closes the last one
enum DistPhase {
    PH_ALPHABET, PH_SPLITTERS, PH_PARTITION, PH_KEY_EXCHANGE, PH_LOCAL_SORT, PH_INIT_RANKS, PH_RANKS_TO_OWNERS, PH_REBALANCE,
    PH_REQUESTS, PH_LAZY, PH_ROUND_SORT, PH_RERANK, PH_RANK_UPDATES, PH_NEW_SA, PH_H2D, PH_D2H, PH_END = -1
};
static_assert(PH_D2H + 1 == SAB200_PHASES, "one phase per slot of sab200_dist_stats::phase_ms");

// One rank's construction, phase by phase (sab_dist_saca runs them; the file header numbers the steps).  The
// members are what one phase leaves for the later ones.
struct DistRun {
    sab200_comm* cm;
    SabContext* c;
    cudaStream_t st;
    sab200_dist_stats* ds;
    DistArena A;
    size_t top0;  // A.hi at the start: the temporaries of the key exchange are released down to it
    int P, g;
    u64 n;
    ShardBounds sh;  // this rank's text positions
    u64 count;       // own positions: sh.hi - sh.lo
    const u8* d_text;
    DistPhases ph;
    SabAlphabet al;
    SplitterDigit sdop;  // slice that holds a key
    SliceDigit slices;   // slice that holds an SA position
    u64 R, sa_off;       // this rank's slice: SA positions [sa_off, sa_off + R)
    bool fused;          // the key exchange went peer to peer (so can the rounds)
    // 5, 6: the slice, its sorted keys and bucket directory (dir[0] is entry dlo), the active list (r1buf, rb.v)
    SortBuffers<u64> buf;
    u32 *sa_local, *r1buf, *rank_seq, *dir;
    const u64* sortedK;
    const u32* sortedI;
    u64 dlo;
    int dir_shift;
    u64 m, tot;  // active records here / over all ranks
    // 7: rank[] at the owners; the buffers of the rounds
    bool lazy = false, rebalanced = false;
    int layout_cyc = 0;
    RankLayout lay;
    u32* rank_local = nullptr;
    SortBuffers<u64> rb;
    u64 key_cap, val_cap;  // records each key / payload buffer of rb can hold
    bool p2p_ready = false;  // 7c: peer-to-peer rounds
    bool lead_barrier = false;  // the first gather is ordered by the row exchange of the peer table
    P2PTable pt;
    bool group_sort_on = true;  // the in-group sort, until most records are in large groups
    // the current round: what the re-rank leaves for the new SA entries and the rank updates
    u32 *upd_idx, *upd_r, *set_pos;
    const u32* sorted_idx;
    int sorted_in;  // which of the two index buffers holds the sorted list

    DistRun(sab200_comm* cm_, SabContext* c_, sab200_dist_stats* ds_, DistArena A0, const u8* text, u64 n_)
        : cm(cm_), c(c_), st(c_->stream), ds(ds_), A(A0), top0(A0.hi), P(cm_->P), g(cm_->rank), n(n_),
          sh(sab_shard_bounds(n_, cm_->P, cm_->rank)), count(sh.hi - sh.lo), d_text(text) { ph.c = c_; }

    static constexpr int PTILE = PassShape<u64>::THREADS * PassShape<u64>::ITEMS;

    // rank[idx[t]] = val[t] on the GPU that owns text position idx[t]; records with idx = 0xFFFFFFFF are dropped.
    // d_extra32 / rows: nd device-side u32 values ride along with the count exchange (rows[s*(P+nd) + P + e]).
    int send_ranks(const u32* idx, const u32* val, u64 cnt, const u32* d_extra32 = nullptr, int nd = 0, u64* rows = nullptr) {
        const size_t mark = A.hi;
        u32* kp = A.top<u32>(cnt + 8);
        u32* vp = A.top<u32>(cnt + 8);
        SAB_ARENA_CHECK(A);
        OwnerDigit dop;
        dop.add = 0;
        dop.lay = lay;
        A2APlan pl;
        SAB_TRY((sab_plan_exchange<u32, OwnerDigit>(cm, c, idx, cnt, nullptr, dop, d_extra32, nd, nullptr, 0, &pl, rows)));
        if (cnt) {
            SAB_TRY(sab_ensure_lookback(c, (size_t)div_up64(cnt, PassShape<u32>::THREADS * PassShape<u32>::ITEMS)));
            SAB_TRY((sab_launch_pass_op<u32, false, OwnerDigit>(c, idx, kp, val, vp, cnt, dop, c->d_gbase)));
        }
        u32* ri = A.top<u32>(pl.rtotal + 8);
        u32* rr = A.top<u32>(pl.rtotal + 8);
        SAB_ARENA_CHECK(A);
        SAB_TRY(sab_comm_exchange(cm, st, pl, kp, ri, sizeof(u32)));
        SAB_TRY(sab_comm_exchange(cm, st, pl, vp, rr, sizeof(u32)));
        if (pl.rtotal) {
            SAB_LAUNCH(dist_scatter_kernel, (unsigned)div_up64(pl.rtotal, 256), 256, 0, st, (const u32*)ri, (const u32*)rr, pl.rtotal,
                       (u32)sh.lo, lay, rank_local);
            SAB_LAUNCH_CHECK();
            c->stats.kernel_launches++;
        }
        A.hi = mark;
        return SAB_OK;
    }

    // ---- 1. common alphabet / key shape: the byte histograms of all shards add up
    int alphabet() {
        ph.mark(PH_ALPHABET);
        SAB_TRY(sab_launch_alphabet_hist(c, d_text, count, c->scratch->hist));
        SAB_LAUNCH(hist_widen_kernel, 1, 256, 0, st, (const u32*)c->scratch->hist, c->d_ghist);
        SAB_LAUNCH_CHECK();
        SAB_TRY(sab_comm_all_reduce_u64(cm, st, c->d_ghist, 256));
        u64* h64 = c->staging->wide;
        SAB_CUDA_TRY(cudaMemcpyAsync(h64, c->d_ghist, 256 * sizeof(u64), cudaMemcpyDeviceToHost, st));
        SAB_CUDA_TRY(cudaStreamSynchronize(st));
        return sab_plan_alphabet(c, h64, n, &al);
    }

    // ---- 2. keys of own positions (into *keys_out), splitters from a sample
    int keys_and_splitters(u64** keys_out) {
        ph.mark(PH_SPLITTERS);
        u64* keysA = A.top<u64>(count + 8);
        SAB_ARENA_CHECK(A);
        if (count) {
            sab_prof_begin(c, SAB_PROF_PACK);
            SAB_TRY(sab_launch_pack(c, d_text, sh.len, count, al.d_lut, al.base, al.k, keysA));
            sab_prof_end(c);
        }
        sdop.np = P - 1;
        for (int i = 0; i < SAB_MAX_RANKS - 1; ++i) sdop.s[i] = ~0ull;
        if (P > 1) {
            // ~8 Ki samples over all ranks (slice sizes within a few per cent); the pool is sorted on the host
            const u32 NS = 8192 / (u32)P < 512 ? 512u : (8192 / (u32)P > 2048 ? 2048u : 8192 / (u32)P);
            const u64 step = count / NS ? count / NS : 1;
            u64* d_sample = cm->d_small;
            SAB_LAUNCH(sample_keys_kernel, (NS + 255) / 256, 256, 0, st, (const u64*)keysA, count, step, NS, d_sample);
            SAB_LAUNCH_CHECK();
            SAB_TRY(sab_comm_all_gather(cm, st, d_sample, d_sample + (NS + 1), (NS + 1) * sizeof(u64)));
            SAB_CUDA_TRY(cudaMemcpyAsync(cm->h_small, d_sample + (NS + 1), (size_t)P * (NS + 1) * sizeof(u64), cudaMemcpyDeviceToHost, st));
            SAB_CUDA_TRY(cudaStreamSynchronize(st));
            std::vector<u64> pool;
            pool.reserve((size_t)P * NS);
            for (int r = 0; r < P; ++r) {
                const u64* row = cm->h_small + (size_t)r * (NS + 1);
                const u64 have = row[NS] <= NS ? row[NS] : NS;
                pool.insert(pool.end(), row, row + have);
            }
            std::sort(pool.begin(), pool.end());
            for (int i = 0; i + 1 < P; ++i) {
                size_t at = (size_t)(i + 1) * pool.size() / (size_t)P;
                if (at >= pool.size()) at = pool.size() - 1;
                sdop.s[i] = pool.empty() ? 0 : pool[at];
            }
        }
        *keys_out = keysA;
        return SAB_OK;
    }

    // ---- 3, 4. partition by destination (digit = number of splitters <= key), payload = global position; the records
    // land in buf.k[0] / buf.v[0], either stored straight into the destination over NVLink (fused) or by all-to-all
    int key_exchange(const u64* keysA) {
        ph.mark(PH_PARTITION);
        A2APlan pk;
        u64 mat[SAB_MAX_RANKS * SAB_MAX_RANKS];
        // the count exchange also carries what the peers need to address this rank's receive buffers directly
        // (fused exchange, below): process, device, arena, offset of the key buffer inside it
        const u64 k0_off = sab_align_up(A.lo, 256);
        u64 extra[5] = {(u64)getpid(), (u64)c->device, (u64)(uintptr_t)c->arena.base, (u64)c->arena.bytes, k0_off};
        constexpr int NX = 5;
        u64 rows[SAB_MAX_RANKS * 32];
        SAB_TRY((sab_plan_exchange<u64, SplitterDigit>(cm, c, keysA, count, nullptr, sdop, nullptr, 0, extra, NX, &pk, rows)));
        const int W = P + NX;
        for (int s = 0; s < P; ++s)
            for (int d = 0; d < P; ++d) mat[(size_t)s * P + d] = rows[(size_t)s * W + d];
        R = pk.rtotal;
        u64 run = 1;  // first SA position of every slice
        for (int r = 0; r < SAB_MAX_RANKS; ++r) {
            slices.start[r] = r < P ? (u32)run : 0xffffffffu;
            if (r == g) sa_off = run;
            if (r < P)
                for (int s = 0; s < P; ++s) run += mat[(size_t)s * P + r];
        }
        slices.pmax = (u32)P - 1;
        SAB_TRY(sab_ensure_lookback(c, (size_t)div_up64((count > R ? count : R) + 1, PTILE)));
        SAB_TRY(sab_ensure_scan(c, (size_t)div_up64(R + 4096, SAB_GSORT_TILE)));
        buf.k[0] = A.bot<u64>(R + 8);
        buf.v[0] = A.bot<u32>(R + 8);
        SAB_ARENA_CHECK(A);
        fused = false;
#ifndef SAB_EMU
        if (P > 1 && cm->kind == 0 && sab_env_int("SAB_DIST_P2P", 1) != 0) {
            SAB_TRY(sab_peers_update(cm, c, rows, W));
            fused = cm->peers_ok;
        }
#endif
        if (fused) {
            // the partition pass stores every record straight into its destination GPU's receive buffers over NVLink
            // (rank s writes behind the records of the ranks before it): no staging copy, no all-to-all; the transfer
            // overlaps the ranking tile by tile.  Every rank entered this call (alphabet all_reduce) before anybody
            // stores, and the all_reduce below orders the stores before the local sort.
            PeerOut po;
            memset(&po, 0, sizeof(po));
            u64* h = c->staging->wide;
            for (int i = 0; i < 256; ++i) h[i] = 0;
            for (int d = 0; d < P; ++d) {
                u64 Rd = 0, before = 0;
                for (int s = 0; s < P; ++s) {
                    Rd += mat[(size_t)s * P + d];
                    if (s < g) before += mat[(size_t)s * P + d];
                }
                const u64 koff = rows[(size_t)d * W + P + 4];
                const u64 voff = sab_align_up(koff + (Rd + 8) * sizeof(u64), 256);
                char* base = d == g ? c->arena.base : (char*)cm->peers[d].base;
                po.k[d] = (u64)(uintptr_t)(base + koff);
                po.v[d] = (u64)(uintptr_t)(base + voff);
                h[d] = before;
            }
            SAB_CUDA_TRY(cudaMemcpyAsync(c->d_gbase, h, 256 * sizeof(u64), cudaMemcpyHostToDevice, st));
            if (count)
                SAB_TRY((sab_launch_pass_op<u64, true, SplitterDigit, true>(c, keysA, (u64*)nullptr, nullptr, (u32*)nullptr, count, sdop,
                                                                           c->d_gbase, &po, (u32)sh.lo)));
            ph.mark(PH_KEY_EXCHANGE);
            SAB_TRY(sab_comm_all_reduce_u64(cm, st, cm->d_small, 1));  // barrier: all peers' stores have landed
            for (int d = 0; d < P; ++d)
                if (d != g) cm->bytes_sent += mat[(size_t)g * P + d] * 12;
        } else {
            u64* partK = A.top<u64>(count + 8);
            u32* partI = A.top<u32>(count + 8);
            SAB_ARENA_CHECK(A);
            if (count)
                SAB_TRY((sab_launch_pass_op<u64, true, SplitterDigit>(c, keysA, partK, nullptr, partI, count, sdop, c->d_gbase, nullptr,
                                                                     (u32)sh.lo)));
            ph.mark(PH_KEY_EXCHANGE);
            SAB_TRY(sab_comm_exchange(cm, st, pk, partK, buf.k[0], sizeof(u64)));
            SAB_TRY(sab_comm_exchange(cm, st, pk, partI, buf.v[0], sizeof(u32)));
        }
        A.hi = top0;  // keysA, partK, partI are dead once the exchange has run (stream order)
        return SAB_OK;
    }

    // ---- 5, 6. local sort -> this rank's slice of the suffix array; init_ranks: ranks, slice of sa[], active list,
    // bucket directory over the slice's keys.  Ends with the active count over all ranks (tot).
    int local_slice(bool* halves_fit) {
        ph.mark(PH_LOCAL_SORT);
        buf.k[1] = A.bot<u64>(R + 8);
        buf.v[1] = A.bot<u32>(R + 8);
        buf.cur = 0;
        sa_local = A.bot<u32>(R + 8);
        r1buf = A.bot<u32>(R + 8);
        SAB_ARENA_CHECK(A);
        bool sa_written = false;  // the last pass writes the sorted indices straight into the slice of sa[]
        SAB_TRY(sab_radix_sort<u64>(c, buf, R, 0, al.key_bits, /*iota=*/false, &c->stats.passes[0], sa_local, &sa_written));

        ph.mark(PH_INIT_RANKS);
        sortedK = buf.k[buf.cur];
        if (c->want_bkt) SAB_TRY(sab_fused_buckets(c, d_text, n, sortedK, R, al));  // this slice's share
        sortedI = sa_written ? sa_local : buf.v[buf.cur];
        u32* act_idx = buf.v[buf.cur ^ 1];
        rank_seq = (u32*)buf.k[buf.cur ^ 1];
        dir_shift = al.key_bits - sab_dir_bits(n, al.key_bits, SAB_DIST_DIR_SHIFT);
        const u64 kmax = al.key_bits >= 64 ? ~0ull : ((1ull << al.key_bits) - 1ull);
        const u64 klo = g > 0 ? sdop.s[g - 1] : 0ull;
        u64 khi = g < P - 1 ? sdop.s[g] : kmax;
        if (khi > kmax) khi = kmax;
        if (khi < klo) khi = klo;
        dlo = klo >> dir_shift;
        const u64 dir_len = (khi >> dir_shift) - dlo + 2;
        dir = A.bot<u32>(dir_len + 8);
        SAB_ARENA_CHECK(A);
        m = 0;
        if (R)
            SAB_TRY(sab_init_ranks(c, sortedK, sortedI, R, (u32)sa_off, nullptr, rank_seq, sa_written ? nullptr : sa_local, r1buf, act_idx,
                                   dir - dlo, dir_shift, &m));
        const u64 half = sab_align_up((size_t)(R + 8) / 2, 32);  // lazy mode: the local list must fit a half (sab_round_buffers)
        u64 sums[2] = {m, (m > (R + 8) - half) ? 1ull : 0ull};
        SAB_TRY(sab_comm_sum_u64(cm, st, sums, 2));
        tot = sums[0];
        *halves_fit = sums[1] == 0;
        c->stats.active[0] = m;
        ds->active[0] = tot;
        return SAB_OK;
    }

    // ---- 7. inverse suffix array at the owners (file header, step 6), and the buffers of the rounds
    int ranks_to_owners(bool halves_fit) {
        ph.mark(PH_RANKS_TO_OWNERS);
        lazy = tot <= n / 4 && halves_fit && sab_env_int("SAB_DIST_LAZY", 1) != 0;
        const char* lenv = getenv("SAB_RANK_LAYOUT");
        layout_cyc = lazy ? 0 : 1;  // lazy look-ups pack keys from the owner's text shard: block ownership
        if (!lazy && lenv && !strcmp(lenv, "block")) layout_cyc = 0;
        u64 local_len;
        if (layout_cyc) {
            u64 per = n / (8ull * (u64)P);
            int shift = 0;
            while (shift < 20 && (2ull << shift) <= per) ++shift;
            const u64 width = 1ull << shift;
            const u64 blocks = div_up64(n + 1, width);
            local_len = div_up64(blocks, (u64)P) << shift;
            sab_rank_layout((u32)width, P, shift, &lay);
        } else {
            local_len = sh.B + 1;  // the last GPU also owns position n
            sab_rank_layout((u32)sh.B, P, -1, &lay);
        }
        rank_local = A.bot<u32>(local_len + 8);
        SAB_ARENA_CHECK(A);
        if (lazy) SAB_CUDA_TRY(cudaMemsetAsync(rank_local, 0xff, local_len * sizeof(u32), st));
        const u32 on = lay.owner(n);  // the empty suffix has rank 0
        if ((int)on == g) SAB_CUDA_TRY(cudaMemsetAsync(rank_local + lay.slot(n, on), 0, sizeof(u32), st));
        if (lazy) SAB_TRY(send_ranks(buf.v[buf.cur ^ 1], r1buf, m));
        else SAB_TRY(send_ranks(sortedI, rank_seq, R));
        rb = sab_round_buffers(buf, R, lazy, &key_cap);
        val_cap = R + 8;
        return SAB_OK;
    }

    // ---- 7b. even out the active lists.  The slices hold equal numbers of SUFFIXES, not of active ones (on the
    // mixed text the English-like key ranges hold nearly all of them) and a round costs what its longest list
    // costs.  The lists are globally sorted by rank and groups never straddle GPUs: cut points move to group
    // boundaries and contiguous chunks are shipped, which keeps both properties.  A suffix that becomes unique
    // on a GPU that does not hold its SA position is then routed to the slice owner (new_sa_entries).
    int rebalance() {
        ph.mark(PH_REBALANCE);
        if (P == 1) return SAB_OK;
        u64 mine[SAB_MAX_RANKS], mm[SAB_MAX_RANKS * SAB_MAX_RANKS];
        for (int d = 0; d < P; ++d) mine[d] = m;
        SAB_TRY(sab_comm_count_matrix(cm, st, mine, mm));  // mm[s*P + *] = list length of rank s
        u64 M = 0, mx = 0, off = 0;
        for (int s = 0; s < P; ++s) {
            const u64 v = mm[(size_t)s * P];
            M += v;
            if (v > mx) mx = v;
            if (s < g) off += v;
        }
        const u64 rebal_min = (u64)sab_env_int("SAB_REBALANCE_MIN", 1 << 20);
        if (M < rebal_min * (u64)P || (double)mx * P <= 1.1 * (double)M) return SAB_OK;
        const u64 Q = div_up64(M, (u64)P);
        u64 *h_cuts = c->staging->wide, *h_found = c->staging->wide + SAB_MAX_RANKS;  // as d_cuts, d_found below
        u64 cuts[SAB_MAX_RANKS], found[SAB_MAX_RANKS];
        for (int j = 1; j < P; ++j) {
            const u64 want = (u64)j * Q;
            cuts[j - 1] = want <= off ? 0 : (want - off >= m ? m : want - off);
            found[j - 1] = (cuts[j - 1] == 0 || cuts[j - 1] >= m) ? cuts[j - 1] : ~0ull;
        }
        u64* d_cuts = c->d_ghist;  // [P-1] cuts, then [P-1] results
        unsigned long long* d_found = (unsigned long long*)(c->d_ghist + SAB_MAX_RANKS);
        memcpy(h_cuts, cuts, sizeof(u64) * (P - 1));
        SAB_CUDA_TRY(cudaMemcpyAsync(d_cuts, h_cuts, sizeof(u64) * (P - 1), cudaMemcpyHostToDevice, st));
        u64 woff = 0, window = 1 << 16;
        for (;;) {
            bool open = false;
            for (int j = 0; j < P - 1; ++j) open = open || found[j] == ~0ull;
            if (!open) break;
            SAB_CUDA_TRY(cudaMemsetAsync(d_found, 0xff, sizeof(u64) * (P - 1), st));
            const u32 bpc = (u32)div_up64(window, 256);
            SAB_LAUNCH(find_boundary_kernel, bpc * (unsigned)(P - 1), 256, 0, st, (const u32*)r1buf, m, (const u64*)d_cuts, bpc, woff,
                       window, d_found);
            SAB_LAUNCH_CHECK();
            SAB_CUDA_TRY(cudaMemcpyAsync(h_found, d_found, sizeof(u64) * (P - 1), cudaMemcpyDeviceToHost, st));
            SAB_CUDA_TRY(cudaStreamSynchronize(st));
            for (int j = 0; j < P - 1; ++j) {
                if (found[j] != ~0ull) continue;
                if (h_found[j] != ~0ull) found[j] = h_found[j];
                else if (cuts[j] + woff + window >= m) found[j] = m;  // the group runs to the end of the list
            }
            woff += window;
            window *= 8;
        }
        u64 bounds[SAB_MAX_RANKS + 1], sendc[SAB_MAX_RANKS];
        bounds[0] = 0;
        for (int j = 1; j < P; ++j) bounds[j] = found[j - 1] > bounds[j - 1] ? found[j - 1] : bounds[j - 1];
        bounds[P] = m;
        for (int j = 0; j < P; ++j) sendc[j] = bounds[j + 1] - bounds[j];
        A2APlan pb;
        SAB_TRY(sab_comm_plan(cm, st, sendc, &pb, nullptr));
        const u64 cap = key_cap < val_cap ? key_cap : val_cap;
        u64 bad = pb.rtotal + 64 > cap ? 1 : 0;
        SAB_TRY(sab_comm_sum_u64(cm, st, &bad, 1));
        if (bad != 0) return SAB_OK;
        const size_t mark = A.hi;
        u32* t1 = A.top<u32>(pb.rtotal + 8);
        u32* t2 = A.top<u32>(pb.rtotal + 8);
        SAB_ARENA_CHECK(A);
        SAB_TRY(sab_comm_exchange(cm, st, pb, r1buf, t1, sizeof(u32)));
        SAB_TRY(sab_comm_exchange(cm, st, pb, rb.v[rb.cur], t2, sizeof(u32)));
        m = pb.rtotal;
        if (m) {
            SAB_CUDA_TRY(cudaMemcpyAsync(r1buf, t1, m * sizeof(u32), cudaMemcpyDeviceToDevice, st));
            SAB_CUDA_TRY(cudaMemcpyAsync(rb.v[rb.cur], t2, m * sizeof(u32), cudaMemcpyDeviceToDevice, st));
        }
        A.hi = mark;
        rebalanced = true;
        return SAB_OK;
    }

    // ---- 7c. peer table of the peer-to-peer rounds (same precondition as the fused key exchange)
    int peer_table() {
        memset(&pt, 0, sizeof(pt));
        if (!fused || rebalanced) return SAB_OK;
        // row: offsets of rank_local, text, sorted keys, directory inside the arena; directory origin, slice length, offset
        u64* hrow = cm->h_small + 32;
        hrow[0] = (u64)((char*)rank_local - c->arena.base);
        hrow[1] = (u64)((const char*)d_text - c->arena.base);
        hrow[2] = (u64)((const char*)sortedK - c->arena.base);
        hrow[3] = (u64)((char*)dir - c->arena.base);
        hrow[4] = dlo;
        hrow[5] = R;
        hrow[6] = sa_off;
        hrow[7] = ((const char*)d_text >= c->arena.base && (const char*)d_text < c->arena.base + c->arena.bytes) ? 1 : 0;
        SAB_CUDA_TRY(cudaMemcpyAsync(cm->d_small, hrow, 8 * sizeof(u64), cudaMemcpyHostToDevice, st));
        u64 prow[SAB_MAX_RANKS * 8];
        SAB_TRY(sab_comm_gather_rows(cm, st, 8, prow));  // also orders every rank's ISA scatter before the first gather
        bool ok = true;
        for (int d = 0; d < P; ++d) {
            const u64* r = prow + (size_t)d * 8;
            char* pb = d == g ? c->arena.base : (char*)cm->peers[d].base;
            ok = ok && r[7] == 1 && pb != nullptr;
            pt.rank_local[d] = (u32*)(pb + r[0]);
            pt.text[d] = (const u8*)(pb + r[1]);
            pt.sorted[d] = (const u64*)(pb + r[2]);
            pt.dir[d] = (const u32*)(pb + r[3]) - r[4];
            pt.R[d] = r[5];
            pt.sa_off[d] = (u32)r[6];
            pt.n_rel[d] = sab_shard_bounds(n, P, d).len;
        }
        p2p_ready = ok;
        return SAB_OK;
    }

    // ---- round, a. (peer to peer): rank[i + h] loaded straight from the owner GPU
    int second_ranks_p2p(u64 h) {
        ph.mark(PH_REQUESTS);
        if (lead_barrier) {  // the owners' scatters of an all-to-all round must have finished everywhere
            SAB_TRY(sab_comm_all_reduce_u64(cm, st, cm->d_small + 8, 1));
            lead_barrier = false;
        }
        if (m) {
            sab_prof_begin(c, SAB_PROF_GATHER);
            SAB_LAUNCH(dist_gather_p2p_kernel, (unsigned)div_up64(m, 256), 256, 0, st, (const u32*)r1buf, (const u32*)rb.v[rb.cur], m,
                       (u32)h, lay, pt, lazy ? 1 : 0, al.d_lut, al.base, al.k, dir_shift, sdop, rb.k[rb.cur]);
            sab_prof_end(c);
            SAB_LAUNCH_CHECK();
            c->stats.kernel_launches++;
        }
        return SAB_OK;
    }

    // ---- round, a + b. (all-to-all): requests i + h to the owners (payload = list position), answers back in the same
    // order.  The buffers are temporaries at the top of the arena; the caller releases them.
    int second_ranks_a2a(u64 h) {
        ph.mark(PH_REQUESTS);
        u32* cur_idx = rb.v[rb.cur];
        u32* ipart = A.top<u32>(m + 8);
        u32* ppart = A.top<u32>(m + 8);
        SAB_ARENA_CHECK(A);
        OwnerDigit odop;
        odop.add = (u32)h;
        odop.lay = lay;
        A2APlan pr;
        SAB_TRY((sab_plan_exchange<u32, OwnerDigit>(cm, c, cur_idx, m, nullptr, odop, nullptr, 0, nullptr, 0, &pr, nullptr)));
        if (m) {
            SAB_TRY(sab_ensure_lookback(c, (size_t)div_up64(m, PTILE)));
            SAB_TRY((sab_launch_pass_op<u32, true, OwnerDigit>(c, cur_idx, ipart, nullptr, ppart, m, odop, c->d_gbase)));
        }
        const u64 nq = pr.rtotal;
        u32* q = A.top<u32>(nq + 8);
        u32* ans = A.top<u32>(nq + 8);
        SAB_ARENA_CHECK(A);
        SAB_TRY(sab_comm_exchange(cm, st, pr, ipart, q, sizeof(u32)));
        if (nq) {
            sab_prof_begin(c, SAB_PROF_GATHER);
            SAB_LAUNCH(dist_gather_kernel, (unsigned)div_up64(nq, 256), 256, 0, st, (const u32*)q, nq, (u32)h, (u32)sh.lo, lay,
                       (const u32*)rank_local, ans);
            sab_prof_end(c);
            SAB_LAUNCH_CHECK();
            c->stats.kernel_launches++;
        }
        if (lazy) {
            // b. requests that found EMPTY: key at the owner -> slice that holds the key -> rank back.  Their
            // number stays on the device until it comes back with the count exchange (one synchronisation).
            ph.mark(PH_LAZY);
            u64* keys_u = A.top<u64>(nq + 8);
            u32* slot_u = A.top<u32>(nq + 8);
            SAB_ARENA_CHECK(A);
            u32* d_nu = &c->scratch->nu;
            SAB_CUDA_TRY(cudaMemsetAsync(d_nu, 0, sizeof(u32), st));
            if (nq) {
                SAB_LAUNCH(dist_lazy_collect_kernel, (unsigned)div_up64(nq, 256), 256, 0, st, q, (const u32*)ans, nq, (u32)h, sh.lo, d_text,
                           sh.len, al.d_lut, al.base, al.k, keys_u, slot_u, d_nu);
                SAB_LAUNCH_CHECK();
                c->stats.kernel_launches++;
            }
            A2APlan pu;
            u64 rows_u[SAB_MAX_RANKS * 32];
            SAB_TRY((sab_plan_exchange<u64, SplitterDigit>(cm, c, keys_u, nq, d_nu, sdop, d_nu, 1, nullptr, 0, &pu, rows_u)));
            const u64 nu = rows_u[(size_t)g * (P + 1) + P];
            ds->resolved_empty += nu;
            u64* kp = A.top<u64>(nu + 8);
            u32* sp = A.top<u32>(nu + 8);
            SAB_ARENA_CHECK(A);
            if (nu) {
                SAB_TRY(sab_ensure_lookback(c, (size_t)div_up64(nu, PTILE)));
                SAB_TRY((sab_launch_pass_op<u64, false, SplitterDigit>(c, keys_u, kp, slot_u, sp, nu, sdop, c->d_gbase)));
            }
            u64* kq = A.top<u64>(pu.rtotal + 8);
            u32* rk = A.top<u32>(pu.rtotal + 8);
            u32* back = A.top<u32>(nu + 8);
            SAB_ARENA_CHECK(A);
            SAB_TRY(sab_comm_exchange(cm, st, pu, kp, kq, sizeof(u64)));
            if (pu.rtotal) {
                SAB_LAUNCH(dist_lookup_kernel, (unsigned)div_up64(pu.rtotal, 256), 256, 0, st, sortedK, R, (const u32*)(dir - dlo), dir_shift,
                           (const u64*)kq, pu.rtotal, (u32)sa_off, rk);
                SAB_LAUNCH_CHECK();
                c->stats.kernel_launches++;
            }
            SAB_TRY(sab_comm_exchange_back(cm, st, pu, rk, back, sizeof(u32)));
            if (nu) {
                SAB_LAUNCH(dist_lazy_fill_kernel, (unsigned)div_up64(nu, 256), 256, 0, st, (const u32*)sp, (const u32*)back, nu, q, (u32)h,
                           (u32)sh.lo, ans, rank_local);
                SAB_LAUNCH_CHECK();
                c->stats.kernel_launches++;
            }
            ph.mark(PH_REQUESTS);
        }
        u32* r2 = A.top<u32>(m + 8);
        SAB_ARENA_CHECK(A);
        SAB_TRY(sab_comm_exchange_back(cm, st, pr, ans, r2, sizeof(u32)));
        if (m) {
            SAB_LAUNCH(dist_place_keys_kernel, (unsigned)div_up64(m, 256), 256, 0, st, (const u32*)r1buf, (const u32*)ppart, (const u32*)r2,
                       m, rb.k[rb.cur]);
            SAB_LAUNCH_CHECK();
            c->stats.kernel_launches++;
        }
        return SAB_OK;
    }

    // ---- round, c + d. order inside the groups (as on one GPU: the list is still grouped by r1, ascending), then
    // re-rank: newly unique suffixes go to sa[], changed ranks are collected for their owners (upd_idx, upd_r); the
    // number of survivors stays on the device and comes back with the count exchange of the rank updates
    int refine(u32 round) {
        ph.mark(PH_ROUND_SORT);
        upd_idx = A.top<u32>(m + 8);
        upd_r = A.top<u32>(m + 8);
        set_pos = rebalanced ? A.top<u32>(m + 8) : nullptr;
        sorted_idx = nullptr;
        sorted_in = 0;
        SAB_ARENA_CHECK(A);
        SAB_CUDA_TRY(cudaMemsetAsync(&c->scratch->count, 0, sizeof(u32), st));  // kept = 0 unless the re-rank says otherwise
        if (m == 0) return SAB_OK;
        const int rank_bits = sab_ceil_log2_u64(n + 2);
        SortBuffers<u64> sb;
        sb.k[0] = rb.k[rb.cur];
        sb.k[1] = rb.k[rb.cur ^ 1];
        sb.v[0] = rb.v[rb.cur];
        sb.v[1] = rb.v[rb.cur ^ 1];
        sb.cur = 0;
        int sorted = 0;
        if (group_sort_on) {
            // the first ranks live in the key words until the re-rank writes them back: r1buf holds the positions
            const GroupSortSpare sp = sab_group_sort_spare(sb, m, key_cap, val_cap, r1buf);
            if (sp.cap * 8 >= m) {
                u64 nbig = 0;
                sorted = sab_group_sort(c, sb, m, 32 + rank_bits, sp, &c->stats.passes[round], &nbig);
                if (sorted < 0) return sorted;
                if (nbig * 2 > m) group_sort_on = false;
            }
        }
        if (!sorted) SAB_TRY(sab_radix_sort<u64>(c, sb, m, 0, 32 + rank_bits, /*iota=*/false, &c->stats.passes[round]));
        ph.mark(PH_RERANK);
        u32* out_idx = (sb.cur == 0) ? rb.v[rb.cur ^ 1] : rb.v[rb.cur];
        // ranks are global SA positions
        SAB_TRY(sab_launch_rerank(c, sb, m, nullptr, sa_local - (size_t)sa_off, r1buf, out_idx, upd_idx, upd_r, set_pos));
        sorted_idx = sb.v[sb.cur];
        sorted_in = sb.cur;
        return SAB_OK;
    }

    // ---- round, f. (rebalanced lists) new SA entries to the GPUs that hold their positions, before the buffer of the
    // sorted indices is reused for the next list; a rank with an empty list still takes part in the exchange
    int new_sa_entries() {
        ph.mark(PH_NEW_SA);
        const size_t mark = A.hi;
        u32* kp = A.top<u32>(m + 8);
        u32* vp = A.top<u32>(m + 8);
        SAB_ARENA_CHECK(A);
        A2APlan ps;
        SAB_TRY((sab_plan_exchange<u32, SliceDigit>(cm, c, set_pos, m, nullptr, slices, nullptr, 0, nullptr, 0, &ps, nullptr)));
        if (m) {
            SAB_TRY(sab_ensure_lookback(c, (size_t)div_up64(m, PTILE)));
            SAB_TRY((sab_launch_pass_op<u32, false, SliceDigit>(c, set_pos, kp, sorted_idx, vp, m, slices, c->d_gbase)));
        }
        u32* rp = A.top<u32>(ps.rtotal + 8);
        u32* ri = A.top<u32>(ps.rtotal + 8);
        SAB_ARENA_CHECK(A);
        SAB_TRY(sab_comm_exchange(cm, st, ps, kp, rp, sizeof(u32)));
        SAB_TRY(sab_comm_exchange(cm, st, ps, vp, ri, sizeof(u32)));
        if (ps.rtotal) {
            SAB_LAUNCH(dist_store_sa_kernel, (unsigned)div_up64(ps.rtotal, 256), 256, 0, st, (const u32*)rp, (const u32*)ri, ps.rtotal,
                       (u32)sa_off, sa_local);
            SAB_LAUNCH_CHECK();
            c->stats.kernel_launches++;
        }
        A.hi = mark;
        return SAB_OK;
    }

    // ---- round, e. changed ranks to their owners; the same exchange returns every rank's number of survivors (tot
    // over all ranks).  The survivors here become the next list.
    int rank_updates(bool p2p_round) {
        u64 kept = 0;
        u32* d_m = &c->scratch->count;
        ph.mark(PH_RANK_UPDATES);
        if (p2p_round) {
            // all_reduce #1: the survivors add up (termination) and every rank has finished LOADING ranks;
            // then the stores go straight into the owners' blocks; all_reduce #2: every store has landed
            SAB_LAUNCH(put_u64_kernel, 1, 1, 0, st, cm->d_small, (const u32*)d_m);
            SAB_LAUNCH_CHECK();
            SAB_TRY(sab_comm_all_reduce_u64(cm, st, cm->d_small, 1));
            if (m) {
                SAB_LAUNCH(dist_scatter_p2p_kernel, (unsigned)div_up64(m, 256), 256, 0, st, (const u32*)upd_idx, (const u32*)upd_r, m, lay, pt);
                SAB_LAUNCH_CHECK();
                c->stats.kernel_launches++;
            }
            SAB_TRY(sab_comm_all_reduce_u64(cm, st, cm->d_small + 8, 1));
            SAB_CUDA_TRY(cudaMemcpyAsync(cm->h_small, cm->d_small, sizeof(u64), cudaMemcpyDeviceToHost, st));
            u32 survivors;
            SAB_TRY(sab_read_u32(c, d_m, 1, &survivors));  // its synchronisation also lands the total
            tot = cm->h_small[0];
            kept = survivors;
            ds->p2p_rounds++;
        } else {
            u64 rows_k[SAB_MAX_RANKS * 32];
            SAB_TRY(send_ranks(upd_idx, upd_r, m, d_m, 1, rows_k));
            kept = rows_k[(size_t)g * (P + 1) + P];
            tot = 0;
            for (int s2 = 0; s2 < P; ++s2) tot += rows_k[(size_t)s2 * (P + 1) + P];
            lead_barrier = true;
        }
        if (m && sorted_in != 0 && kept > 0)
            SAB_CUDA_TRY(cudaMemcpyAsync(rb.v[rb.cur ^ 1], rb.v[rb.cur], kept * sizeof(u32), cudaMemcpyDeviceToDevice, st));
        rb.cur ^= 1;
        m = kept;
        return SAB_OK;
    }
};

// d_text: this rank's shard + halo on the device (text_len bytes).  The arena `A0` starts behind whatever the
// caller placed at its bottom.  Enqueues on c->stream; the stream is idle when the function returns.
static int sab_dist_saca(sab200_comm* cm, SabContext* c, DistArena A0, const u8* d_text, u64 text_len, u64 n, DistResult* res,
                         sab200_dist_stats* ds) {
    cudaStream_t st = c->stream;
    SabStats& S = c->stats;
    S.n = n;
    cm->bytes_sent = 0;
    cm->collectives = 0;
    DistRun run(cm, c, ds, A0, d_text, n);
    *res = DistResult{nullptr, 0, 1};
    ds->nranks = (u32)run.P;
    ds->rank = (u32)run.g;
    if (n == 0) return SAB_OK;  // the suffix array is the sentinel alone
    if (text_len < run.sh.len) {
        sab_set_error("rank %d: shard of %llu bytes, need %llu (own positions + halo)", run.g, (unsigned long long)text_len,
                      (unsigned long long)run.sh.len);
        return SAB_ERR_ARGS;
    }
    SAB_TRY(sab_ensure_scan(c, (size_t)div_up64(run.count + run.count / 2 + 4096, SAB_GSORT_TILE)));

    u64* keysA = nullptr;
    SAB_TRY(run.alphabet());
    SAB_TRY(run.keys_and_splitters(&keysA));
    SAB_TRY(run.key_exchange(keysA));
    bool halves_fit = false;
    SAB_TRY(run.local_slice(&halves_fit));
    u32 round = 0;
    if (run.tot > 0) {
        SAB_TRY(run.ranks_to_owners(halves_fit));
        SAB_TRY(run.rebalance());
        SAB_TRY(run.peer_table());
        // records per rank; above it the all-to-all form wins (measured on 8 B200, 1 GiB text: every round peer to peer
        // 20.3 ms, limit 2 Mi 18.8 ms; on 2 GPUs limits of 4 Mi .. 16 Mi are within 1 % of each other)
        const u64 p2p_max = (u64)sab_env_int("SAB_P2P_MAX_RECORDS", 2 << 20);
        u64 h = (u64)run.al.k;
        while (run.tot > 0) {
            ++round;
            if (round >= SAB_MAX_ROUNDS || h > n) {
                sab_set_error("prefix doubling did not converge (round %u, h=%llu, active=%llu)", round, (unsigned long long)h,
                              (unsigned long long)run.tot);
                return SAB_ERR_INTERNAL;
            }
            const size_t topmark = run.A.hi;
            // Small rounds go peer to peer (no exchange step, one host round trip); large ones through partition +
            // all-to-all (bulk NVLink transfers, local random access).  Same decision on every rank.
            const bool p2p_round = run.p2p_ready && run.tot <= p2p_max * (u64)run.P;
            if (p2p_round) SAB_TRY(run.second_ranks_p2p(h));
            else SAB_TRY(run.second_ranks_a2a(h));
            run.A.hi = topmark;  // requests, answers and look-up buffers are dead (stream order)
            SAB_TRY(run.refine(round));
            if (run.rebalanced) SAB_TRY(run.new_sa_entries());
            SAB_TRY(run.rank_updates(p2p_round));
            run.A.hi = topmark;
            S.active[round] = run.m;
            ds->active[round] = run.tot;
            h *= 2;
        }
    }
    run.ph.mark(PH_END);
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    run.ph.collect(ds->phase_ms, &ds->total_ms);
    S.rounds = round;
    S.total_ms = ds->total_ms;
    res->d_slice = run.sa_local;
    res->slice_len = run.R;
    res->sa_off = run.sa_off;
    ds->rounds = round;
    ds->lazy_isa = run.lazy ? 1u : 0u;
    ds->rank_layout = (u32)run.layout_cyc;
    ds->rebalanced = run.rebalanced ? 1u : 0u;
    ds->fused_exchange = run.fused ? 1u : 0u;
    ds->slice_len = run.R;
    ds->sa_off = run.sa_off;
    ds->all_to_all_bytes = cm->bytes_sent;
    ds->collectives = cm->collectives;
    return SAB_OK;
}

// ------------------------------------------------------------------ extern "C": communicators
extern "C" int32_t sab200_comm_unique_id(uint8_t id[128]) {
#ifndef SAB_EMU
    if (!id) return SAB_ERR_ARGS;
    SAB_TRY(sab_nccl_load());
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId u;
    SAB_NCCL_TRY(g_nccl.GetUniqueId(&u));
    memcpy(id, &u, 128);
    return SAB_OK;
#else
    (void)id;
    sab_set_error("the emulator build has no NCCL");
    return SAB_ERR_NCCL;
#endif
}

extern "C" sab200_comm* sab200_comm_create_nccl(const uint8_t id[128], int32_t rank, int32_t nranks, int32_t device) {
#ifndef SAB_EMU
    if (!id || nranks < 1 || nranks > SAB_MAX_RANKS || rank < 0 || rank >= nranks) {
        sab_set_error("sab200_comm_create_nccl: bad arguments (rank %d of %d)", (int)rank, (int)nranks);
        return nullptr;
    }
    if (sab_nccl_load() != SAB_OK) return nullptr;
    if (!sab_get_context(device)) return nullptr;
    sab200_comm* cm = new (std::nothrow) sab200_comm();
    if (!cm) return nullptr;
    cm->rank = rank;
    cm->P = nranks;
    cm->device = device;
    cm->kind = 0;
    memset(&cm->cb, 0, sizeof(cm->cb));
    memset(&cm->last, 0, sizeof(cm->last));
    if (cudaSetDevice(device) != cudaSuccess || sab_comm_alloc_scratch(cm) != SAB_OK) {
        sab_comm_free(cm);
        return nullptr;
    }
    ncclUniqueId u;
    memcpy(&u, id, 128);
    ncclComm_t nc = nullptr;
    ncclResult_t r = g_nccl.CommInitRank(&nc, nranks, u, rank);
    if (r != ncclSuccess) {
        sab_set_error("ncclCommInitRank(rank %d of %d): %s", (int)rank, (int)nranks, g_nccl.GetErrorString(r));
        sab_comm_free(cm);
        return nullptr;
    }
    cm->nccl = nc;
    return cm;
#else
    (void)id; (void)rank; (void)nranks; (void)device;
    sab_set_error("the emulator build has no NCCL");
    return nullptr;
#endif
}

extern "C" sab200_comm* sab200_comm_create_callbacks(const sab200_comm_callbacks* cb, int32_t rank, int32_t nranks, int32_t device) {
    if (!cb || !cb->all_gather || !cb->all_reduce_sum_u64 || !cb->all_to_all_v || nranks < 1 || nranks > SAB_MAX_RANKS || rank < 0 ||
        rank >= nranks) {
        sab_set_error("sab200_comm_create_callbacks: bad arguments (rank %d of %d)", (int)rank, (int)nranks);
        return nullptr;
    }
    if (!sab_get_context(device)) return nullptr;
    sab200_comm* cm = new (std::nothrow) sab200_comm();
    if (!cm) return nullptr;
    cm->rank = rank;
    cm->P = nranks;
    cm->device = device;
    cm->kind = 1;
    cm->cb = *cb;
    memset(&cm->last, 0, sizeof(cm->last));
    if (sab_comm_alloc_scratch(cm) != SAB_OK) {
        sab_comm_free(cm);
        return nullptr;
    }
    return cm;
}

extern "C" void sab200_comm_destroy(sab200_comm* cm) { sab_comm_free(cm); }

extern "C" int32_t sab200_comm_stats(sab200_comm* cm, sab200_dist_stats* out) {
    if (!cm || !out) return SAB_ERR_ARGS;
    *out = cm->last;
    return SAB_OK;
}

// ------------------------------------------------------------------ one rank of a sharded construction
// host_out_base != null: the slice is copied to host_out_base + sa_off (the caller's whole sa[] array)
// h_bkt_part != null: this rank's share of the fused bucket table (SAB200_BKT_LEN counts, host) -- the caller adds the
// shares of all ranks and 1 for the empty suffix
static int sab_sharded_run(sab200_comm* cm, const u8* shard, u64 shard_len, u64 n, int shard_on_device, u32* out, u64 out_cap,
                           int out_on_device, u32* host_out_base, u64* slice_len, u64* sa_off, const u32** d_slice,
                           u32* h_bkt_part = nullptr) {
    if (!cm || (shard_len > 0 && !shard) || n > SAB200_MAX_LENGTH) {
        sab_set_error("sab200_saca_sharded: bad arguments (n=%llu)", (unsigned long long)n);
        return SAB_ERR_ARGS;
    }
    const double w0 = now_ms();
    SabUse u;
    SAB_TRY(sab_use(cm->device, &u));
    SabContext* c = u.c;
    memset(&c->stats, 0, sizeof(c->stats));
    c->profiling = g_profiling;
    sab200_dist_stats& ds = cm->last;
    memset(&ds, 0, sizeof(ds));
    const u64 B = sab_shard_bounds(n, cm->P, cm->rank).B;
    if (cm->last_want != sab_dist_want(B)) {
        // another text size than last time (every rank sees the same change): arenas may be re-allocated, so all
        // peer mappings are closed first, on every rank, before anybody frees
        cm->last_want = sab_dist_want(B);
        sab_comm_close_peers(cm);
        u64 z = 0;
        SAB_TRY(sab_comm_sum_u64(cm, c->stream, &z, 1));
    }
    SAB_TRY(sab_dist_reserve(c, B));
    DistArena A;
    A.base = c->arena.base;
    A.lo = 0;
    A.hi = c->arena.bytes & ~(size_t)255;
    A.ok = true;
    cudaStream_t st = c->stream;
    const u8* d_text = shard;
    cudaEvent_t e0 = sab_event_get(c), e1 = sab_event_get(c), e2 = sab_event_get(c), e3 = sab_event_get(c);
    cudaEventRecord(e0, st);
    if (!shard_on_device || (cm->P > 1 && cm->kind == 0)) {
        // host shard: upload; device shard on a multi-GPU run: a copy inside the arena, which is what the peers have
        // mapped (the lazy look-ups of the peer-to-peer rounds read the owner's text)
        u8* t = A.bot<u8>((size_t)shard_len + 64);
        SAB_ARENA_CHECK(A);
        if (shard_len && shard_on_device) SAB_CUDA_TRY(cudaMemcpyAsync(t, shard, shard_len, cudaMemcpyDeviceToDevice, st));
        else if (shard_len) SAB_TRY(sab_copy_h2d(c, t, shard, shard_len));
        d_text = t;
    }
    cudaEventRecord(e1, st);
    u32* d_bkt = nullptr;
    if (h_bkt_part) {
        d_bkt = A.bot<u32>((size_t)SAB200_BKT_LEN + 8);
        SAB_ARENA_CHECK(A);
        SAB_CUDA_TRY(cudaMemsetAsync(d_bkt, 0, (size_t)SAB200_BKT_LEN * sizeof(u32), st));
    }
    c->want_bkt = d_bkt;
    c->bkt_add_one = 0;
    DistResult res;
    const double w1 = now_ms();
    int rc = sab_dist_saca(cm, c, A, d_text, shard_len, n, &res, &ds);
    const double w2 = now_ms();
    c->want_bkt = nullptr;
    c->bkt_add_one = 1;
    if (rc != SAB_OK) {
        sab_reset_after_failure(c);
        return rc;
    }
    if (slice_len) *slice_len = res.slice_len;
    if (sa_off) *sa_off = res.sa_off;
    if (d_slice) *d_slice = res.d_slice;
    cudaEventRecord(e2, st);
    if (h_bkt_part) SAB_CUDA_TRY(cudaMemcpyAsync(h_bkt_part, d_bkt, (size_t)SAB200_BKT_LEN * sizeof(u32), cudaMemcpyDeviceToHost, st));
    if (host_out_base) {
        if (res.slice_len) SAB_TRY(sab_copy_d2h(c, host_out_base + res.sa_off, res.d_slice, res.slice_len * sizeof(u32)));
        if (cm->rank == 0) host_out_base[0] = (u32)n;  // src/saca.rs:13
    } else if (out) {
        if (out_cap < res.slice_len) {
            sab_set_error("sab200_saca_sharded: the slice has %llu entries, the buffer holds %llu", (unsigned long long)res.slice_len,
                          (unsigned long long)out_cap);
            return SAB_ERR_ARGS;
        }
        if (res.slice_len && out_on_device)
            SAB_CUDA_TRY(cudaMemcpyAsync(out, res.d_slice, res.slice_len * sizeof(u32), cudaMemcpyDeviceToDevice, st));
        else if (res.slice_len)
            SAB_TRY(sab_copy_d2h(c, out, res.d_slice, res.slice_len * sizeof(u32)));
    }
    cudaEventRecord(e3, st);
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    ds.phase_ms[PH_H2D] = ms;
    cudaEventElapsedTime(&ms, e2, e3);
    ds.phase_ms[PH_D2H] = ms;
    c->stats.h2d_ms = ds.phase_ms[PH_H2D];
    c->stats.d2h_ms = ds.phase_ms[PH_D2H];
    c->event_pool.push_back(e0);
    c->event_pool.push_back(e1);
    c->event_pool.push_back(e2);
    c->event_pool.push_back(e3);
    sab_prof_collect(c);
    g_last_stats = c->stats;
    ds.wall_ms = now_ms() - w0;
    ds.host_setup_ms = w1 - w0;
    ds.host_finish_ms = (w2 - w1) - ds.total_ms;  // host time of the construction that its stream did not cover
    return SAB_OK;
}

extern "C" int32_t sab200_sort_pairs_device(uint64_t* d_k0, uint64_t* d_k1, uint32_t* d_v0, uint32_t* d_v1, uint64_t count,
                                            int32_t key_bits, int32_t device) {
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    if (key_bits < 0 || key_bits > 64) return SAB_ERR_ARGS;
    SortBuffers<u64> buf;
    buf.k[0] = d_k0;
    buf.k[1] = d_k1;
    buf.v[0] = d_v0;
    buf.v[1] = d_v1;
    buf.cur = 0;
    u32 passes = 0;
    const int rc = sab_radix_sort<u64>(u.c, buf, count, 0, key_bits, false, &passes);
    if (rc != SAB_OK) return rc;
    SAB_CUDA_TRY(cudaStreamSynchronize(u.c->stream));
    return buf.cur;
}

extern "C" int32_t sab200_group_sort_device(uint64_t* d_k0, uint64_t* d_k1, uint32_t* d_v0, uint32_t* d_v1, uint64_t count,
                                            int32_t key_bits, int32_t ascending, int32_t device, uint64_t* nbig_out) {
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    if (key_bits < 32 || key_bits > 64 || count > 0xfffffff0ull) return SAB_ERR_ARGS;
    if (nbig_out) *nbig_out = 0;
    if (count == 0) return 0;
    const u64 cap = sab_align_up((size_t)count * 2 + 64, 64);  // room for every record, and for the position sort
    GroupSortSpare sp;
    SAB_TRY(sab_arena_carve(u.c, {{&sp.k[0], cap * 8}, {&sp.k[1], cap * 8}, {&sp.v[0], cap * 4}, {&sp.v[1], cap * 4}, {&sp.pos, cap * 4}}));
    sp.cap = cap;
    SortBuffers<u64> sb;
    sb.k[0] = d_k0;
    sb.k[1] = d_k1;
    sb.v[0] = d_v0;
    sb.v[1] = d_v1;
    sb.cur = 0;
    u32 passes = 0;
    u64 nbig = 0;
    const int rc = sab_group_sort(u.c, sb, count, key_bits, sp, &passes, &nbig, ascending != 0);
    if (rc < 0) return rc;
    if (rc == 0) {
        sab_set_error("group sort: the records of large groups did not fit the spare buffers");
        return SAB_ERR_INTERNAL;
    }
    SAB_CUDA_TRY(cudaStreamSynchronize(u.c->stream));
    if (nbig_out) *nbig_out = nbig;
    return sb.cur;
}

extern "C" int32_t sab200_copy_from_device(void* dst, const void* d_src, uint64_t bytes, int32_t device) {
    if (!dst || !d_src) return bytes ? SAB_ERR_ARGS : SAB_OK;
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    SAB_CUDA_TRY(cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, u.c->stream));
    SAB_CUDA_TRY(cudaStreamSynchronize(u.c->stream));
    return SAB_OK;
}

extern "C" int32_t sab200_saca_sharded(sab200_comm* cm, const uint8_t* shard, uint64_t shard_len, uint64_t n, int32_t shard_on_device,
                                       uint32_t* out, uint64_t out_cap, int32_t out_on_device, uint64_t* slice_len,
                                       uint64_t* sa_off, const uint32_t** d_slice) {
    return sab_sharded_run(cm, shard, shard_len, n, shard_on_device, out, out_cap, out_on_device, nullptr, slice_len, sa_off, d_slice);
}

// ------------------------------------------------------------------ one process, ngpus GPUs: sab200_saca(..., ngpus > 1)
static std::mutex g_multi_mu;
static std::vector<sab200_comm*> g_multi_comms;  // ncclCommInitAll over devices 0..P-1, cached between calls

static int sab_multi_comms(int P) {
#ifndef SAB_EMU
    if ((int)g_multi_comms.size() == P) return SAB_OK;
    for (auto* cm : g_multi_comms) sab_comm_free(cm);
    g_multi_comms.clear();
    SAB_TRY(sab_nccl_load());
    std::vector<int> devs(P);
    for (int i = 0; i < P; ++i) {
        devs[i] = i;
        if (!sab_get_context(i)) return SAB_ERR_CUDA;
    }
    std::vector<ncclComm_t> nc(P);
    SAB_NCCL_TRY(g_nccl.CommInitAll(nc.data(), P, devs.data()));
    for (int i = 0; i < P; ++i) {
        sab200_comm* cm = new (std::nothrow) sab200_comm();
        if (!cm) return SAB_ERR_OOM;
        cm->rank = i;
        cm->P = P;
        cm->device = i;
        cm->kind = 0;
        cm->nccl = nc[i];
        memset(&cm->cb, 0, sizeof(cm->cb));
        memset(&cm->last, 0, sizeof(cm->last));
        g_multi_comms.push_back(cm);
        SAB_TRY(sab_comm_alloc_scratch(cm));
    }
    return SAB_OK;
#else
    (void)P;
    sab_set_error("the emulator build has no NCCL");
    return SAB_ERR_NCCL;
#endif
}

static int sab_saca_multi(const u8* s, u64 n, u32* sa, int P, u32* bkt) {
    std::lock_guard<std::mutex> lk(g_multi_mu);
    SAB_TRY(sab_multi_comms(P));
    std::vector<int> rcs(P, SAB_OK);
    std::vector<std::thread> th;
    std::vector<u32> parts;
    if (bkt) parts.assign((size_t)P * SAB200_BKT_LEN, 0u);
    for (int g = 0; g < P; ++g) {
        th.emplace_back([&, g]() {
            const ShardBounds sh = sab_shard_bounds(n, P, g);
            rcs[g] = sab_sharded_run(g_multi_comms[g], s + sh.lo, sh.len, n, 0, nullptr, 0, 0, sa, nullptr, nullptr, nullptr,
                                     bkt ? parts.data() + (size_t)g * SAB200_BKT_LEN : nullptr);
        });
    }
    for (auto& t : th) t.join();
    if (n == 0) sa[0] = 0;
    if (bkt) {  // inclusive boundaries: the slices' shares add up; + 1 for the empty suffix (src/sa.rs:98)
        for (u32 i = 0; i < SAB200_BKT_LEN; ++i) {
            u32 v = 1;
            for (int g = 0; g < P; ++g) v += parts[(size_t)g * SAB200_BKT_LEN + i];
            bkt[i] = v;
        }
    }
    for (int g = 0; g < P; ++g)
        if (rcs[g] != SAB_OK) return rcs[g];
    return SAB_OK;
}

extern "C" int32_t sab200_multi_stats(int32_t rank, sab200_dist_stats* out) {
    std::lock_guard<std::mutex> lk(g_multi_mu);
    if (!out || rank < 0 || rank >= (int)g_multi_comms.size()) return SAB_ERR_ARGS;
    *out = g_multi_comms[rank]->last;
    return SAB_OK;
}

static void sab_multi_shutdown() {
    std::lock_guard<std::mutex> lk(g_multi_mu);
    for (auto* cm : g_multi_comms) sab_comm_free(cm);
    g_multi_comms.clear();
}
