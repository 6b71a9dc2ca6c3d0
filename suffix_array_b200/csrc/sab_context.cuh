// sab_context.cuh -- per-device context: stream, scratch for the radix sort and the chained scans,
// and a grow-only arena for the big arrays.  Device memory, streams and events are the only
// resources the library owns (SURVEY.md 8b "Ownership"); no host pointer is retained.
#pragma once
#include <stdarg.h>

#include <cstddef>
#include <initializer_list>
#include <mutex>
#include <vector>

#include "sab_common.cuh"
#include "sab_scan.cuh"

#define SAB_MAX_ROUNDS 64

// mirrors sab200_stats in include/sab200.h (kept in sync by a static_assert in sab_api.cu)
struct SabStats {
    u64 n;                  // text length of the last construction
    u32 sigma;              // distinct byte values
    u32 bits_per_symbol;    // b
    u32 symbols_per_key;    // k
    u32 rounds;             // doubling rounds executed (0 = settled by the initial sort)
    u64 active[SAB_MAX_ROUNDS];   // active suffixes entering round r (r = 0: after the initial sort)
    u32 passes[SAB_MAX_ROUNDS];   // radix passes executed in the sort of round r (index 0 = initial)
    u64 radix_pass_launches;      // onesweep launches
    u64 radix_pass_records;       // sum over launches of records moved
    u64 radix_pass_bytes;         // sum over launches of 2*(K+V)*m  (algorithmic bytes)
    double radix_pass_ms;         // sum of CUDA-event durations of those launches (profiling on)
    double hist_ms;               // radix histogram kernels
    double pack_ms;               // alphabet + key packing
    double rank_ms;               // head-flag / rank / compaction kernels
    double gather_ms;             // rank[i+h] gathers
    double total_ms;              // whole device pipeline (events around it)
    double h2d_ms, d2h_ms;        // host entry only
    u64 kernel_launches;          // all kernels launched by the last call
    double group_sort_ms;         // in-group sorts of the rounds (group_sort_kernel + scatter-back)
    u64 group_sort_records;       // records that went through group_sort_kernel
    u64 group_big_records;        // ... of which in groups too large for it (radix-sorted)
};

enum SabProfKind { SAB_PROF_RADIX_PASS, SAB_PROF_HIST, SAB_PROF_PACK, SAB_PROF_RANK, SAB_PROF_GATHER, SAB_PROF_GROUP_SORT };

struct SabEventPair {
    cudaEvent_t a, b;
    SabProfKind kind;  // the SabStats timing the pair adds to (sab_prof_collect)
};

// Device scalars and small tables of a context: one member per user, so no step overwrites a value another still needs.
struct SabScratch {
    u32 count;      // init_ranks / re-rank: records still active
    u32 filter[2];  // split filter: records to sort, records parked
    u32 check_flag; // sab200_check, matching-statistics extension: set when the array is not the suffix array of the text
    u32 big;        // in-group sort: records of groups too large for it
    u32 nu;         // multi-GPU lazy look-ups: requests that found no rank
    u32 skip[16];   // radix sort: 1 for each digit place where all keys agree (SAB_MAX_PASSES of them)
    u32 hist[256];  // byte histogram of a text
    u16 lut[256];   // code table of the running construction (sab_plan_alphabet)
    u32 bwt[2];     // sab200_bwt: the primary index; sab200_inverse_bwt: sample rows, list position of row p
    u32 ms_offs;    // sab200_matching_statistics_batch_device: set when the query offsets decrease
    u32 lz[4];      // sab200_lz77: the factor count; sab200_lz77_decode: rule flags, factor total (2 words), round changed
};

// Pinned host staging of a context: readbacks land here, and small uploads leave from here, not from the caller's stack.
struct SabStaging {
    u32 read[256];  // sab_read_u32
    u32 sa0;        // sa[0] = n of a single-GPU construction
    u16 lut[256];   // a code table, built here for its asynchronous upload
    u64 wide[256];  // u64 rows of the multi-GPU driver, both ways
};

// A grow-only device buffer that an entry point carves into the buffers of one call.
struct SabArena {
    char* base = nullptr;
    size_t bytes = 0, used = 0;
};

struct SabContext {
    int device = 0;
    cudaStream_t stream = 0;
    int sm_count = 148;
    // radix scratch
    u64* d_ghist = nullptr;   // [8][256]
    u64* d_gbase = nullptr;   // [8][256]
    u64* d_lookback = nullptr;
    size_t lookback_tiles = 0;
    u32* d_ticket = nullptr;
    u32 ticket_host = 0;
    u32 lb_epoch = 0;
    // chained-scan scratch (3 x u32 states at most)
    ScanSlot* d_scan_slots = nullptr;  // chained-scan status, one 16-byte slot per tile
    size_t scan_tiles = 0;
    u32 scan_epoch = 0;
    SabScratch* scratch = nullptr;  // device
    SabStaging* staging = nullptr;  // pinned host
    SabArena arena;
    size_t arena_want_seen = 0;  // request the arena was last sized for (it may have been capped by the free memory)
    void* bounce[2] = {nullptr, nullptr};        // pinned bounce buffers for pageable caller memory (sab_copy_*)
    cudaEvent_t bounce_ev[2] = {nullptr, nullptr};
    u32* want_bkt = nullptr;     // device buffer for the fused bucket table of the running construction (or null)
    u32 bkt_add_one = 1;  // added to every boundary of the fused table: 1 counts the empty suffix, 0 for a rank's share
    // profiling
    bool profiling = false;
    std::vector<SabEventPair> events;
    std::vector<cudaEvent_t> event_pool;
    SabStats stats;
    std::mutex mu;
};

SabContext* sab_get_context(int device);
int sab_context_init(SabContext* c);
void sab_context_destroy(SabContext* c);
int sab_arena_reserve(SabArena* a, cudaStream_t st, size_t bytes);
static inline int sab_arena_reserve(SabContext* c, size_t bytes) { return sab_arena_reserve(&c->arena, c->stream, bytes); }
int sab_ensure_lookback(SabContext* c, size_t tiles);
int sab_ensure_scan(SabContext* c, size_t tiles);

static inline size_t sab_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bump allocation inside the arena (call sab_arena_reserve first)
template <typename T>
static inline T* sab_arena_take(SabArena* a, size_t count) {
    size_t off = sab_align_up(a->used, 256);
    a->used = off + count * sizeof(T);
    return (T*)(a->base + off);
}

// One buffer of an entry point's arena: *dst receives its address; a null dst reserves the room without handing it out.
struct SabSlice {
    void** dst;
    size_t bytes;
    template <typename T>
    SabSlice(T** p, size_t b) : dst((void**)p), bytes(b) {}
    SabSlice(std::nullptr_t, size_t b) : dst(nullptr), bytes(b) {}
};

// Reserves the sum of the 256-aligned sizes and hands the buffers out in order from the bottom of the arena.
// A reallocation first waits for `st`, the stream that last used the arena.
static inline int sab_arena_carve(SabArena* a, cudaStream_t st, std::initializer_list<SabSlice> slices) {
    size_t total = 0;
    for (const SabSlice& s : slices) total += sab_align_up(s.bytes, 256);
    SAB_TRY(sab_arena_reserve(a, st, total));
    a->used = 0;
    for (const SabSlice& s : slices) {
        char* p = sab_arena_take<char>(a, s.bytes);
        if (s.dst) *s.dst = p;
    }
    return SAB_OK;
}
static inline int sab_arena_carve(SabContext* c, std::initializer_list<SabSlice> slices) {
    return sab_arena_carve(&c->arena, c->stream, slices);
}

// The context of `device`, locked and current on the calling thread: the prologue of the entry points.
struct SabUse {
    SabContext* c = nullptr;
    std::unique_lock<std::mutex> lk;
};
static inline int sab_use(int device, SabUse* u) {
    u->c = sab_get_context(device);
    if (!u->c) return SAB_ERR_CUDA;
    u->lk = std::unique_lock<std::mutex>(u->c->mu);
    SAB_CUDA_TRY(cudaSetDevice(u->c->device));
    return SAB_OK;
}

// n <= 256 device words into out[] through the pinned staging, with one stream synchronisation
static inline int sab_read_u32(SabContext* c, const u32* d_src, int n, u32* out) {
    SAB_CUDA_TRY(cudaMemcpyAsync(c->staging->read, d_src, (size_t)n * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
    SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    memcpy(out, c->staging->read, (size_t)n * sizeof(u32));
    return SAB_OK;
}

cudaEvent_t sab_event_get(SabContext* c);
int sab_copy_h2d(SabContext* c, void* d_dst, const void* h_src, size_t bytes);
int sab_copy_d2h(SabContext* c, void* h_dst, const void* d_src, size_t bytes);
void sab_prof_begin(SabContext* c, SabProfKind kind);
void sab_prof_end(SabContext* c);
void sab_prof_collect(SabContext* c);

template <typename T>
static inline TileState<T> sab_tile_state(SabContext* c, size_t tiles) {
    (void)tiles;
    TileState<T> st;
    st.slots = c->d_scan_slots;
    if (++c->scan_epoch >= (1u << 30)) {  // wrap: stale tags of 2^30 launches ago must not match
        cudaMemsetAsync(c->d_scan_slots, 0, c->scan_tiles * sizeof(ScanSlot), c->stream);
        c->scan_epoch = 1;
    }
    st.epoch = c->scan_epoch;
    return st;
}
