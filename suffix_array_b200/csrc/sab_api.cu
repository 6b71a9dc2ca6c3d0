// sab_api.cu -- context management and the extern "C" surface declared in include/sab200.h.
// Single translation unit: the kernels live in the .cuh headers included below.
#include "../../include/sab200.h"
#include "sab_common.cuh"
#include "sab_context.cuh"
#include "sab_saca.cuh"
#include "sab_search.cuh"
#include "sab_pack.cuh"
#include "sab_bwt.cuh"
#include "sab_lz.cuh"

#include <chrono>
#include <cstdlib>
#include <new>
#include <thread>

static_assert(sizeof(SabStats) == sizeof(sab200_stats), "SabStats must mirror sab200_stats");
static_assert(SAB_MAX_ROUNDS == SAB200_MAX_ROUNDS, "round table size");
static_assert(SAB_MAX_PASSES * sizeof(u32) <= sizeof(SabScratch::skip), "a skip flag for every radix pass");

// ------------------------------------------------------------------ error string
static char g_err[1024] = "";
static std::mutex g_err_mu;
void sab_set_error(const char* fmt, ...) {
    std::lock_guard<std::mutex> lk(g_err_mu);
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ------------------------------------------------------------------ contexts
#define SAB_MAX_DEVICES 16
static SabContext* g_ctx[SAB_MAX_DEVICES];
static std::mutex g_ctx_mu;
static bool g_profiling = false;
static SabStats g_last_stats;

int sab_context_init(SabContext* c) {
    SAB_CUDA_TRY(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    SAB_CUDA_TRY(cudaGetDeviceProperties(&prop, c->device));
    c->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    SAB_CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    SAB_CUDA_TRY(cudaMalloc(&c->d_ghist, sizeof(u64) * SAB_MAX_PASSES * SAB_RADIX_BINS));
    SAB_CUDA_TRY(cudaMalloc(&c->d_gbase, sizeof(u64) * SAB_MAX_PASSES * SAB_RADIX_BINS));
    SAB_CUDA_TRY(cudaMallocHost(&c->staging, sizeof(SabStaging)));
    SAB_CUDA_TRY(cudaMalloc(&c->d_ticket, sizeof(u32) * 4));
    SAB_CUDA_TRY(cudaMemset(c->d_ticket, 0, sizeof(u32) * 4));
    SAB_CUDA_TRY(cudaMalloc(&c->scratch, sizeof(SabScratch)));
    SAB_CUDA_TRY(cudaMemset(c->scratch, 0, sizeof(SabScratch)));
    return SAB_OK;
}

void sab_context_destroy(SabContext* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (auto& e : c->events) {
        cudaEventDestroy(e.a);
        cudaEventDestroy(e.b);
    }
    for (auto e : c->event_pool) cudaEventDestroy(e);
    cudaFree(c->d_ghist);
    cudaFree(c->d_gbase);
    cudaFreeHost(c->staging);
    for (int i = 0; i < 2; ++i) {
        if (c->bounce[i]) cudaFreeHost(c->bounce[i]);
        if (c->bounce_ev[i]) cudaEventDestroy(c->bounce_ev[i]);
    }
    cudaFree(c->d_lookback);
    cudaFree(c->d_ticket);
    cudaFree(c->d_scan_slots);
    cudaFree(c->scratch);
    cudaFree(c->arena.base);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

SabContext* sab_get_context(int device) {
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    if (device < 0 || device >= SAB_MAX_DEVICES) {
        sab_set_error("device %d out of range", device);
        return nullptr;
    }
    if (g_ctx[device]) return g_ctx[device];
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= device) {
        sab_set_error("no CUDA device %d available (%s); libsab200 has no CPU fallback", device,
                      e != cudaSuccess ? cudaGetErrorString(e) : "device count too small");
        return nullptr;
    }
    SabContext* c = new (std::nothrow) SabContext();
    if (!c) return nullptr;
    c->device = device;
    if (sab_context_init(c) != SAB_OK) {
        delete c;
        return nullptr;
    }
    g_ctx[device] = c;
    return c;
}

int sab_arena_reserve(SabArena* a, cudaStream_t st, size_t bytes) {
    if (a->bytes >= bytes) return SAB_OK;
    if (a->base) {
        SAB_CUDA_TRY(cudaStreamSynchronize(st));
        SAB_CUDA_TRY(cudaFree(a->base));
        a->base = nullptr;
        a->bytes = 0;
    }
    const size_t want = sab_align_up(bytes, (size_t)1 << 21);
    cudaError_t e = cudaMalloc(&a->base, want);
    if (e != cudaSuccess) {
        a->base = nullptr;
        sab_set_error("device arena of %zu bytes: %s", want, cudaGetErrorString(e));
        cudaGetLastError();
        return SAB_ERR_OOM;
    }
    a->bytes = want;
    return SAB_OK;
}

// Status words of one radix pass over `tiles` tiles: one per tile and bin, followed by one per group of
// SAB_LB_GROUP tiles and bin (two-level look-back).  lookback_tiles counts allocated 256-word rows.
int sab_ensure_lookback(SabContext* c, size_t tiles) {
    tiles += tiles / SAB_LB_GROUP + 2;
    if (c->lookback_tiles >= tiles) return SAB_OK;
    if (c->d_lookback) {
        SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
        SAB_CUDA_TRY(cudaFree(c->d_lookback));
        c->d_lookback = nullptr;
        c->lookback_tiles = 0;
    }
    const size_t want = tiles + tiles / 8 + 64;
    SAB_CUDA_TRY(cudaMalloc(&c->d_lookback, want * SAB_RADIX_BINS * sizeof(u64)));
    SAB_CUDA_TRY(cudaMemsetAsync(c->d_lookback, 0, want * SAB_RADIX_BINS * sizeof(u64), c->stream));
    c->lookback_tiles = want;
    c->lb_epoch = 0;
    return SAB_OK;
}

int sab_ensure_scan(SabContext* c, size_t tiles) {
    if (c->scan_tiles >= tiles) return SAB_OK;
    if (c->d_scan_slots) {
        SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
        cudaFree(c->d_scan_slots);
        c->d_scan_slots = nullptr;
        c->scan_tiles = 0;
    }
    const size_t want = tiles + tiles / 8 + 64;
    SAB_CUDA_TRY(cudaMalloc(&c->d_scan_slots, want * sizeof(ScanSlot)));
    SAB_CUDA_TRY(cudaMemsetAsync(c->d_scan_slots, 0, want * sizeof(ScanSlot), c->stream));
    c->scan_tiles = want;
    c->scan_epoch = 0;
    return SAB_OK;
}

// ------------------------------------------------------------------ per-launch event timing
cudaEvent_t sab_event_get(SabContext* c) {
    if (!c->event_pool.empty()) {
        cudaEvent_t e = c->event_pool.back();
        c->event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
void sab_prof_begin(SabContext* c, SabProfKind kind) {
    if (!c->profiling) return;
    SabEventPair p;
    p.a = sab_event_get(c);
    p.b = sab_event_get(c);
    p.kind = kind;
    cudaEventRecord(p.a, c->stream);
    c->events.push_back(p);
}
void sab_prof_end(SabContext* c) {
    if (!c->profiling || c->events.empty()) return;
    cudaEventRecord(c->events.back().b, c->stream);
}
void sab_prof_collect(SabContext* c) {
    if (!c->profiling) return;
    cudaStreamSynchronize(c->stream);
    for (auto& p : c->events) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, p.a, p.b);
        switch (p.kind) {
            case SAB_PROF_RADIX_PASS: c->stats.radix_pass_ms += ms; break;
            case SAB_PROF_HIST: c->stats.hist_ms += ms; break;
            case SAB_PROF_PACK: c->stats.pack_ms += ms; break;
            case SAB_PROF_RANK: c->stats.rank_ms += ms; break;
            case SAB_PROF_GATHER: c->stats.gather_ms += ms; break;
            case SAB_PROF_GROUP_SORT: c->stats.group_sort_ms += ms; break;
        }
        c->event_pool.push_back(p.a);
        c->event_pool.push_back(p.b);
    }
    c->events.clear();
}

// ------------------------------------------------------------------ host <-> device copies of caller buffers
// The seam hands over whatever the caller allocated -- for the Rust crate a plain Vec (pageable memory).  CUDA
// stages pageable copies through a small internal buffer at 12-15 GB/s; here they go through two pinned bounce
// buffers of the context instead: the DMA of chunk i+1 (PCIe rate) overlaps the host memcpy of chunk i, which a
// few threads share.  Pinned / registered caller buffers take the direct path.
#define SAB_BOUNCE_BYTES ((size_t)32 << 20)
static int sab_copy_threads() {
    static int t = 0;
    if (!t) {
        int hw = (int)std::thread::hardware_concurrency();
        t = hw >= 16 ? 6 : (hw >= 8 ? 4 : (hw >= 4 ? 2 : 1));
        const char* e = getenv("SAB_COPY_THREADS");
        if (e && atoi(e) > 0) t = atoi(e);
    }
    return t;
}
static void sab_parallel_memcpy(void* dst, const void* src, size_t bytes) {
    const int T = sab_copy_threads();
    if (T <= 1 || bytes < ((size_t)4 << 20)) {
        memcpy(dst, src, bytes);
        return;
    }
    std::vector<std::thread> th;
    const size_t per = (((bytes + (size_t)T - 1) / (size_t)T) + 4095) & ~(size_t)4095;  // T * per >= bytes
    for (int i = 1; i < T; ++i) {
        const size_t lo = (size_t)i * per;
        if (lo >= bytes) break;
        const size_t len = lo + per < bytes ? per : bytes - lo;
        th.emplace_back([=]() { memcpy((char*)dst + lo, (const char*)src + lo, len); });
    }
    memcpy(dst, src, per < bytes ? per : bytes);
    for (auto& t : th) t.join();
}
static bool sab_is_pageable(const void* p) {
    const char* f = getenv("SAB_FORCE_STAGED");
    if (f && *f == '1') return true;
#ifdef SAB_EMU
    (void)p;
    return false;
#else
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
#endif
}
static int sab_bounce_init(SabContext* c) {
    if (c->bounce[0]) return SAB_OK;
    for (int i = 0; i < 2; ++i) {
        SAB_CUDA_TRY(cudaMallocHost(&c->bounce[i], SAB_BOUNCE_BYTES));
        SAB_CUDA_TRY(cudaEventCreateWithFlags(&c->bounce_ev[i], cudaEventDisableTiming));
    }
    return SAB_OK;
}
// host -> device on c->stream; returns with the copy ENQUEUED (pinned source) or COMPLETE (pageable source)
int sab_copy_h2d(SabContext* c, void* d_dst, const void* h_src, size_t bytes) {
    if (!bytes) return SAB_OK;
    if (!sab_is_pageable(h_src)) {
        SAB_CUDA_TRY(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, c->stream));
        return SAB_OK;
    }
    SAB_TRY(sab_bounce_init(c));
    size_t off = 0;
    for (int i = 0; off < bytes; ++i) {
        const int b = i & 1;
        const size_t len = bytes - off < SAB_BOUNCE_BYTES ? bytes - off : SAB_BOUNCE_BYTES;
        if (i >= 2) SAB_CUDA_TRY(cudaEventSynchronize(c->bounce_ev[b]));  // the DMA out of this buffer has finished
        sab_parallel_memcpy(c->bounce[b], (const char*)h_src + off, len);
        SAB_CUDA_TRY(cudaMemcpyAsync((char*)d_dst + off, c->bounce[b], len, cudaMemcpyHostToDevice, c->stream));
        SAB_CUDA_TRY(cudaEventRecord(c->bounce_ev[b], c->stream));
        off += len;
    }
    SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SAB_OK;
}
// device -> host; everything enqueued on c->stream before the call is waited for; returns with the data in place
int sab_copy_d2h(SabContext* c, void* h_dst, const void* d_src, size_t bytes) {
    if (!bytes) return SAB_OK;
    if (!sab_is_pageable(h_dst)) {
        SAB_CUDA_TRY(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, c->stream));
        SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
        return SAB_OK;
    }
    SAB_TRY(sab_bounce_init(c));
    const size_t nchunks = (bytes + SAB_BOUNCE_BYTES - 1) / SAB_BOUNCE_BYTES;
    auto issue = [&](size_t i) -> int {
        const size_t off = i * SAB_BOUNCE_BYTES;
        const size_t len = bytes - off < SAB_BOUNCE_BYTES ? bytes - off : SAB_BOUNCE_BYTES;
        SAB_CUDA_TRY(cudaMemcpyAsync(c->bounce[i & 1], (const char*)d_src + off, len, cudaMemcpyDeviceToHost, c->stream));
        SAB_CUDA_TRY(cudaEventRecord(c->bounce_ev[i & 1], c->stream));
        return SAB_OK;
    };
    SAB_TRY(issue(0));
    for (size_t i = 0; i < nchunks; ++i) {
        if (i + 1 < nchunks) SAB_TRY(issue(i + 1));  // its buffer was emptied by the memcpy of chunk i-1
        SAB_CUDA_TRY(cudaEventSynchronize(c->bounce_ev[i & 1]));
        const size_t off = i * SAB_BOUNCE_BYTES;
        const size_t len = bytes - off < SAB_BOUNCE_BYTES ? bytes - off : SAB_BOUNCE_BYTES;
        sab_parallel_memcpy((char*)h_dst + off, c->bounce[i & 1], len);
    }
    return SAB_OK;
}

static double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// a failed launch may have left the ticket counter of the radix passes out of step with its host mirror
static void sab_reset_after_failure(SabContext* c) {
    cudaMemsetAsync(c->d_ticket, 0, sizeof(u32) * 4, c->stream);
    cudaStreamSynchronize(c->stream);
    c->ticket_host = 0;
}

static int run_device(SabContext* c, const u8* d_s, u64 n, u32* d_sa) {
    c->profiling = g_profiling;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, c->stream);
    int rc = sab_saca_device(c, d_s, n, d_sa);
    cudaEventRecord(e1, c->stream);
    cudaStreamSynchronize(c->stream);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    sab_prof_collect(c);
    c->stats.total_ms = ms;
    if (rc != SAB_OK) sab_reset_after_failure(c);
    return rc;
}

static int sab_saca_multi(const u8* s, u64 n, u32* sa, int P, u32* bkt);  // sab_dist.cuh
static void sab_multi_shutdown();

// ------------------------------------------------------------------ extern "C"
extern "C" {

int32_t sab200_saca_device(const uint8_t* d_s, uint64_t n, uint32_t* d_sa, int32_t device) {
    if (!d_sa || (n > 0 && !d_s) || n > SAB200_MAX_LENGTH) {
        sab_set_error("sab200_saca_device: bad arguments (n=%llu)", (unsigned long long)n);
        return SAB_ERR_ARGS;
    }
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    int rc = run_device(u.c, d_s, n, d_sa);
    g_last_stats = u.c->stats;
    return rc;
}

static int32_t saca_host(const uint8_t* s, uint64_t n, uint32_t* sa, uint32_t* bkt, int32_t ngpus);

int32_t sab200_saca(const uint8_t* s, uint64_t n, uint32_t* sa, int32_t ngpus) { return saca_host(s, n, sa, nullptr, ngpus); }

int32_t sab200_saca_buckets(const uint8_t* s, uint64_t n, uint32_t* sa, uint32_t* bkt, int32_t ngpus) {
    if (!bkt) {
        sab_set_error("sab200_saca_buckets: bkt is null");
        return SAB_ERR_ARGS;
    }
    return saca_host(s, n, sa, bkt, ngpus);
}

static int32_t saca_host(const uint8_t* s, uint64_t n, uint32_t* sa, uint32_t* bkt, int32_t ngpus) {
    if (ngpus == 0) ngpus = sab200_device_count() > SAB_MAX_RANKS ? SAB_MAX_RANKS : sab200_device_count();
    if (!sa || (n > 0 && !s) || n > SAB200_MAX_LENGTH || ngpus < 0 || ngpus > SAB_MAX_RANKS) {
        sab_set_error("sab200_saca: bad arguments (n=%llu, ngpus=%d)", (unsigned long long)n, (int)ngpus);
        return SAB_ERR_ARGS;
    }
    if (sab200_device_count() < 1) {
        sab_set_error("no CUDA device available; libsab200 has no CPU fallback");
        return SAB_ERR_CUDA;
    }
    if (ngpus > sab200_device_count()) {
        sab_set_error("sab200_saca: %d GPUs requested, %d visible", (int)ngpus, (int)sab200_device_count());
        return SAB_ERR_ARGS;
    }
    if (bkt && n < ((u64)1 << 20)) ngpus = 1;  // tiny texts may pack a single symbol per key: the table then needs the text
    if (ngpus > 1) return sab_saca_multi(s, n, sa, ngpus, bkt);
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    SabContext* c = u.c;
    // the construction workspace first (sab_saca_device takes it from the bottom), text, SA and bucket table above it
    u8* d_s;
    u32 *d_sa, *d_bkt;
    SAB_TRY(sab_arena_carve(c, {{nullptr, sab_saca_workspace_bytes(n)}, {&d_s, (size_t)n + 64}, {&d_sa, ((size_t)n + 1) * sizeof(u32)},
                                {&d_bkt, (size_t)SAB200_BKT_LEN * sizeof(u32)}}));
    c->want_bkt = bkt ? d_bkt : nullptr;
    c->bkt_add_one = 1;
    double t0 = now_ms();
    SAB_TRY(sab_copy_h2d(c, d_s, s, n));
    SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    double t1 = now_ms();
    int rc = run_device(c, d_s, n, d_sa);
    c->want_bkt = nullptr;
    if (rc == SAB_OK) {
        double t2 = now_ms();
        if (bkt) {
            if (n == 0) {
                for (u32 i = 0; i < SAB200_BKT_LEN; ++i) bkt[i] = 1;  // src/sa.rs:98,112-116 on an empty text
            } else {
                SAB_CUDA_TRY(cudaMemcpyAsync(bkt, d_bkt, (size_t)SAB200_BKT_LEN * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
            }
        }
        SAB_TRY(sab_copy_d2h(c, sa, d_sa, (n + 1) * sizeof(u32)));
        c->stats.h2d_ms = t1 - t0;
        c->stats.d2h_ms = now_ms() - t2;
    }
    g_last_stats = c->stats;
    return rc;
}

}  // extern "C"

// ---- buckets -------------------------------------------------------------------------------
extern "C" int32_t sab200_enable_buckets(const uint8_t* s, uint64_t n, uint32_t* bkt) {
    if (!bkt || (n > 0 && !s) || n > SAB200_MAX_LENGTH) {
        sab_set_error("sab200_enable_buckets: bad arguments");
        return SAB_ERR_ARGS;
    }
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    SabContext* c = u.c;
    u8* d_s;
    u32* d_bkt;
    SAB_TRY(sab_arena_carve(c, {{&d_s, (size_t)n + 64}, {&d_bkt, (size_t)SAB200_BKT_LEN * sizeof(u32)}}));
    if (n) SAB_CUDA_TRY(cudaMemcpyAsync(d_s, s, n, cudaMemcpyHostToDevice, c->stream));
    SabAlphabet al = {};
    if (n) SAB_TRY(sab_alphabet_local(c, d_s, n, &al));
    SAB_TRY(sab_pair_buckets(c, d_s, n, al.d_lut, al.sigma, d_bkt));
    SAB_CUDA_TRY(cudaMemcpyAsync(bkt, d_bkt, SAB200_BKT_LEN * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
    SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SAB_OK;
}

// ---- integrity check -----------------------------------------------------------------------
extern "C" int32_t sab200_check(const uint8_t* s, uint64_t n, const uint32_t* sa, uint64_t sa_len) {
    if (!sa || (n > 0 && !s) || n > SAB200_MAX_LENGTH) {
        sab_set_error("sab200_check: bad arguments");
        return SAB_ERR_ARGS;
    }
    if (sa_len != n + 1) return 0;  // src/sa.rs:73-75
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    const size_t text_bytes = sab_align_up((size_t)n + 64, 256);
    const size_t arr_bytes = sab_align_up(((size_t)n + 2) * sizeof(u32), 256);
    u8* d_s;
    u32 *d_sa, *d_isa;
    SAB_TRY(sab_arena_carve(u.c, {{&d_s, text_bytes}, {&d_sa, arr_bytes}, {&d_isa, arr_bytes}}));
    cudaStream_t st = u.c->stream;
    SAB_CUDA_TRY(cudaMemsetAsync(d_s, 0, text_bytes, st));
    if (n) SAB_CUDA_TRY(cudaMemcpyAsync(d_s, s, n, cudaMemcpyHostToDevice, st));
    SAB_CUDA_TRY(cudaMemcpyAsync(d_sa, sa, sa_len * sizeof(u32), cudaMemcpyHostToDevice, st));
    u32 bad;
    SAB_TRY(sab_isa_check(u.c, d_s, n, d_sa, sa_len, d_isa, &bad));
    return bad ? 0 : 1;
}

// ---- LCP array ------------------------------------------------------------------------------
extern "C" int32_t sab200_lcp_array(const uint8_t* s, uint64_t n, const uint32_t* sa, uint64_t sa_len, uint32_t* lcp) {
    if (!sa || !lcp || (n > 0 && !s) || n > SAB200_MAX_LENGTH || sa_len != n + 1) {
        sab_set_error("sab200_lcp_array: bad arguments (n=%llu, sa_len=%llu)", (unsigned long long)n, (unsigned long long)sa_len);
        return SAB_ERR_ARGS;
    }
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    const size_t arr_bytes = ((size_t)n + 2) * sizeof(u32);
    u8* d_s;
    u32 *d_sa, *d_isa, *d_lcp;
    SAB_TRY(sab_arena_carve(u.c, {{&d_s, (size_t)n + 64}, {&d_sa, arr_bytes}, {&d_isa, arr_bytes}, {&d_lcp, arr_bytes}}));
    cudaStream_t st = u.c->stream;
    if (n) SAB_CUDA_TRY(cudaMemcpyAsync(d_s, s, n, cudaMemcpyHostToDevice, st));
    SAB_CUDA_TRY(cudaMemcpyAsync(d_sa, sa, sa_len * sizeof(u32), cudaMemcpyHostToDevice, st));
    SAB_LAUNCH(lcp_isa_kernel, (unsigned)div_up64(sa_len, 256), 256, 0, st, (const u32*)d_sa, sa_len, d_isa);
    SAB_LAUNCH_CHECK();
    SAB_TRY(sab_launch_kasai(u.c, d_s, n, d_sa, d_isa, d_lcp));
    SAB_CUDA_TRY(cudaMemcpyAsync(lcp, d_lcp, sa_len * sizeof(u32), cudaMemcpyDeviceToHost, st));
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    return SAB_OK;
}

// ---- Burrows-Wheeler transform --------------------------------------------------------------
// The construction, then the last column L of its n+1 rows into d_L (n+1 bytes; the bottom of the construction
// workspace is free for it once the construction is done).  The construction's statistics stay readable.
static int bwt_forward(SabContext* c, const u8* d_s, u64 n, u32* d_sa, u8* d_L, u64* primary) {
    const int rc = run_device(c, d_s, n, d_sa);
    g_last_stats = c->stats;
    SAB_TRY(rc);
    return sab_bwt_gather(c, d_s, n, d_sa, d_L, primary);
}

static bool bwt_bad_args(const char* who, const void* in, uint64_t n, const void* out) {
    if ((n > 0 && (!in || !out)) || n > SAB200_MAX_LENGTH) {
        sab_set_error("%s: bad arguments (n=%llu)", who, (unsigned long long)n);
        return true;
    }
    return false;
}

static bool bwt_bad_primary(const char* who, uint64_t n, uint64_t primary) {
    if (n == 0 ? primary != 0 : (primary < 1 || primary > n)) {
        sab_set_error("%s: primary index %llu outside [1, %llu] (0 for the empty text)", who, (unsigned long long)primary,
                      (unsigned long long)n);
        return true;
    }
    return false;
}

extern "C" int32_t sab200_bwt(const uint8_t* s, uint64_t n, uint8_t* bwt, uint64_t* primary) {
    if (!primary || bwt_bad_args("sab200_bwt", s, n, bwt)) return SAB_ERR_ARGS;
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    SabContext* c = u.c;
    u8 *d_L, *d_s;
    u32* d_sa;
    SAB_TRY(sab_arena_carve(c, {{&d_L, sab_saca_workspace_bytes(n)}, {&d_s, (size_t)n + 64}, {&d_sa, ((size_t)n + 1) * sizeof(u32)}}));
    SAB_TRY(sab_copy_h2d(c, d_s, s, n));
    u64 p;
    SAB_TRY(bwt_forward(c, d_s, n, d_sa, d_L, &p));
    SAB_TRY(sab_copy_d2h(c, bwt, d_L, p));  // U = L without row p: two pieces of L, no compaction
    SAB_TRY(sab_copy_d2h(c, bwt + p, d_L + p + 1, n - p));
    *primary = p;
    return SAB_OK;
}

extern "C" int32_t sab200_bwt_device(const uint8_t* d_s, uint64_t n, uint8_t* d_bwt, uint64_t* primary, int32_t device) {
    if (!primary || bwt_bad_args("sab200_bwt_device", d_s, n, d_bwt)) return SAB_ERR_ARGS;
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    SabContext* c = u.c;
    u8* d_L;
    u32* d_sa;
    SAB_TRY(sab_arena_carve(c, {{&d_L, sab_saca_workspace_bytes(n)}, {&d_sa, ((size_t)n + 1) * sizeof(u32)}}));
    u64 p;
    SAB_TRY(bwt_forward(c, d_s, n, d_sa, d_L, &p));
    if (p > 0) SAB_CUDA_TRY(cudaMemcpyAsync(d_bwt, d_L, p, cudaMemcpyDeviceToDevice, c->stream));
    if (n > p) SAB_CUDA_TRY(cudaMemcpyAsync(d_bwt + p, d_L + p + 1, n - p, cudaMemcpyDeviceToDevice, c->stream));
    SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    *primary = p;
    return SAB_OK;
}

static int inverse_bwt_run(SabContext* c, const u8* d_u, u64 n, u64 primary, u8* d_s) {
    const int rc = sab_inverse_bwt_run(c, d_u, n, (u32)primary, d_s);
    if (rc != SAB_OK) sab_reset_after_failure(c);
    return rc;
}

extern "C" int32_t sab200_inverse_bwt(const uint8_t* bwt, uint64_t n, uint64_t primary, uint8_t* s) {
    if (bwt_bad_args("sab200_inverse_bwt", bwt, n, s) || bwt_bad_primary("sab200_inverse_bwt", n, primary)) return SAB_ERR_ARGS;
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    if (n == 0) return SAB_OK;
    SabContext* c = u.c;
    u8* d_u;  // the transform in, the text out: U is dead once it has been widened into the sort records
    SAB_TRY(sab_arena_carve(c, {{nullptr, sab_inverse_bwt_workspace_bytes(n)}, {&d_u, (size_t)n + 64}}));
    SAB_TRY(sab_copy_h2d(c, d_u, bwt, n));
    SAB_TRY(inverse_bwt_run(c, d_u, n, primary, d_u));
    return sab_copy_d2h(c, s, d_u, n);
}

extern "C" int32_t sab200_inverse_bwt_device(const uint8_t* d_bwt, uint64_t n, uint64_t primary, uint8_t* d_s, int32_t device) {
    if (bwt_bad_args("sab200_inverse_bwt_device", d_bwt, n, d_s) || bwt_bad_primary("sab200_inverse_bwt_device", n, primary))
        return SAB_ERR_ARGS;
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    if (n == 0) return SAB_OK;
    return inverse_bwt_run(u.c, d_bwt, n, primary, d_s);
}

// ---- Lempel-Ziv factorization ----------------------------------------------------------------
// The construction, then the parse in its workspace d_work (dead once the construction is done).  The construction's
// statistics stay readable.  *d_pos / *d_len: the z factors, inside the workspace.
static int lz77_forward(SabContext* c, const u8* d_s, u64 n, u32* d_sa, char* d_work, u32** d_pos, u32** d_len, u64* z) {
    const int rc = run_device(c, d_s, n, d_sa);
    g_last_stats = c->stats;
    SAB_TRY(rc);
    *z = 0;
    if (n == 0) return SAB_OK;
    return sab_lz77_parse(c, d_s, n, d_sa, d_work, d_pos, d_len, z);
}

static bool lz77_bad_args(const char* who, const void* s, uint64_t n, const void* pos, const void* len, uint64_t cap, const void* z) {
    if (!z || (n > 0 && !s) || (cap > 0 && (!pos || !len)) || n > SAB200_MAX_LENGTH) {
        sab_set_error("%s: bad arguments (n=%llu, cap=%llu)", who, (unsigned long long)n, (unsigned long long)cap);
        return true;
    }
    return false;
}

static bool lz77_short_cap(const char* who, uint64_t z, uint64_t cap) {
    if (cap >= z) return false;
    sab_set_error("%s: %llu factors, room for %llu", who, (unsigned long long)z, (unsigned long long)cap);
    return true;
}

extern "C" int32_t sab200_lz77(const uint8_t* s, uint64_t n, uint32_t* pos, uint32_t* len, uint64_t cap, uint64_t* z) {
    if (lz77_bad_args("sab200_lz77", s, n, pos, len, cap, z)) return SAB_ERR_ARGS;
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    SabContext* c = u.c;
    char* d_work;
    u8* d_s;
    u32* d_sa;
    SAB_TRY(sab_arena_carve(c, {{&d_work, sab_saca_workspace_bytes(n)}, {&d_s, (size_t)n + 64}, {&d_sa, ((size_t)n + 1) * sizeof(u32)}}));
    SAB_TRY(sab_copy_h2d(c, d_s, s, n));
    u32 *d_pos = nullptr, *d_len = nullptr;
    SAB_TRY(lz77_forward(c, d_s, n, d_sa, d_work, &d_pos, &d_len, z));
    if (lz77_short_cap("sab200_lz77", *z, cap)) return SAB_ERR_ARGS;
    SAB_TRY(sab_copy_d2h(c, pos, d_pos, *z * sizeof(u32)));
    return sab_copy_d2h(c, len, d_len, *z * sizeof(u32));
}

extern "C" int32_t sab200_lz77_device(const uint8_t* d_s, uint64_t n, uint32_t* d_pos, uint32_t* d_len, uint64_t cap, uint64_t* z,
                                      int32_t device) {
    if (lz77_bad_args("sab200_lz77_device", d_s, n, d_pos, d_len, cap, z)) return SAB_ERR_ARGS;
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    SabContext* c = u.c;
    char* d_work;
    u32* d_sa;
    SAB_TRY(sab_arena_carve(c, {{&d_work, sab_saca_workspace_bytes(n)}, {&d_sa, ((size_t)n + 1) * sizeof(u32)}}));
    u32 *w_pos = nullptr, *w_len = nullptr;
    SAB_TRY(lz77_forward(c, d_s, n, d_sa, d_work, &w_pos, &w_len, z));
    if (lz77_short_cap("sab200_lz77_device", *z, cap)) return SAB_ERR_ARGS;
    if (*z) {
        SAB_CUDA_TRY(cudaMemcpyAsync(d_pos, w_pos, *z * sizeof(u32), cudaMemcpyDeviceToDevice, c->stream));
        SAB_CUDA_TRY(cudaMemcpyAsync(d_len, w_len, *z * sizeof(u32), cudaMemcpyDeviceToDevice, c->stream));
    }
    SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return SAB_OK;
}

// the checks the host can make before any device work
static bool lz77_decode_bad_args(const char* who, const void* pos, const void* len, uint64_t z, uint64_t n, const void* s) {
    if ((z > 0 && (!pos || !len)) || (n > 0 && !s)) {
        sab_set_error("%s: bad arguments (z=%llu, n=%llu)", who, (unsigned long long)z, (unsigned long long)n);
        return true;
    }
    if (n > SAB200_MAX_LENGTH) {
        sab_set_error("%s: n = %llu exceeds SAB200_MAX_LENGTH", who, (unsigned long long)n);
        return true;
    }
    if (z > n) {
        sab_set_error("%s: %llu factors cannot parse %llu bytes (z > n)", who, (unsigned long long)z, (unsigned long long)n);
        return true;
    }
    if (z == 0 && n > 0) {
        sab_set_error("%s: the factor lengths (max(1, len) each) sum to 0, not to n = %llu", who, (unsigned long long)n);
        return true;
    }
    return false;
}

static int lz77_decode_run(SabContext* c, const u32* d_pos, const u32* d_len, u64 z, u64 n, u8* d_s) {
    const int rc = sab_lz77_decode_run(c, d_pos, d_len, z, n, d_s);
    if (rc != SAB_OK && rc != SAB_ERR_ARGS) sab_reset_after_failure(c);
    return rc;
}

extern "C" int32_t sab200_lz77_decode(const uint32_t* pos, const uint32_t* len, uint64_t z, uint64_t n, uint8_t* s) {
    if (lz77_decode_bad_args("sab200_lz77_decode", pos, len, z, n, s)) return SAB_ERR_ARGS;
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    if (n == 0) return SAB_OK;
    SabContext* c = u.c;
    u32 *d_pos, *d_len;
    u8* d_s;
    SAB_TRY(sab_arena_carve(c, {{nullptr, sab_lz77_decode_workspace_bytes(z, n)}, {&d_pos, (size_t)z * 4}, {&d_len, (size_t)z * 4},
                                {&d_s, (size_t)n + 64}}));
    SAB_TRY(sab_copy_h2d(c, d_pos, pos, z * 4));
    SAB_TRY(sab_copy_h2d(c, d_len, len, z * 4));
    SAB_TRY(lz77_decode_run(c, d_pos, d_len, z, n, d_s));
    return sab_copy_d2h(c, s, d_s, n);
}

extern "C" int32_t sab200_lz77_decode_device(const uint32_t* d_pos, const uint32_t* d_len, uint64_t z, uint64_t n, uint8_t* d_s,
                                             int32_t device) {
    if (lz77_decode_bad_args("sab200_lz77_decode_device", d_pos, d_len, z, n, d_s)) return SAB_ERR_ARGS;
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    if (n == 0) return SAB_OK;
    return lz77_decode_run(u.c, d_pos, d_len, z, n, d_s);
}

// ---- pack serialisation ---------------------------------------------------------------------
extern "C" uint64_t sab200_pack_bound(uint64_t sa_len) { return 16 + ((sa_len + 127) / 128) * 512; }

extern "C" int32_t sab200_pack(const uint32_t* sa, uint64_t sa_len, uint8_t* out, uint64_t out_cap, uint64_t* out_len) {
    if (!sa || !out || !out_len || sa_len == 0 || sa_len > 0xffffffffull) {  // src/packed_sa.rs:18
        sab_set_error("sab200_pack: bad arguments");
        return SAB_ERR_ARGS;
    }
    const unsigned bits = sab_pack_bits(sa_len);
    const u64 blocks = (sa_len + 127) / 128;
    const u64 words = blocks * 4ull * bits;
    if (out_cap < 16 + words * 4) {
        sab_set_error("sab200_pack: output buffer too small (need %llu bytes)", (unsigned long long)(16 + words * 4));
        return SAB_ERR_ARGS;
    }
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    u32 *d_sa, *d_out;
    SAB_TRY(sab_arena_carve(u.c, {{&d_sa, (size_t)sa_len * 4 + 64}, {&d_out, (size_t)words * 4}}));
    cudaStream_t st = u.c->stream;
    SAB_CUDA_TRY(cudaMemcpyAsync(d_sa, sa, sa_len * 4, cudaMemcpyHostToDevice, st));
    if (words) {
        SAB_LAUNCH(pack_blocks_kernel, (unsigned)div_up64(words, 256), 256, 0, st, (const u32*)d_sa, sa_len, bits, words, d_out);
        SAB_LAUNCH_CHECK();
        SAB_CUDA_TRY(cudaMemcpyAsync(out + 16, d_out, words * 4, cudaMemcpyDeviceToHost, st));
    }
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    u64 data_len = words * 4;
    if (sa_len % 128 != 0) {  // src/packed_sa.rs:41-45: trailing zero bytes of the padded last block are dropped
        const u64 chunk = 16ull * bits, start = data_len - chunk;
        u64 t = chunk;
        while (t > 0 && out[16 + start + t - 1] == 0) --t;
        data_len = start + t;
    }
    const u32 magic = SAB_PACK_MAGIC, length = (u32)sa_len;
    memcpy(out, &magic, 4);
    memcpy(out + 4, &length, 4);
    memcpy(out + 8, &data_len, 8);
    *out_len = 16 + data_len;
    return SAB_OK;
}

extern "C" int32_t sab200_unpack(const uint8_t* bytes, uint64_t nbytes, uint32_t* sa, uint64_t sa_cap, uint64_t* sa_len) {
    if (!bytes || !sa || !sa_len || nbytes < 16) {
        sab_set_error("sab200_unpack: bad arguments");
        return SAB_ERR_ARGS;
    }
    u32 magic, length;
    u64 dlen;
    memcpy(&magic, bytes, 4);
    memcpy(&length, bytes + 4, 4);
    memcpy(&dlen, bytes + 8, 8);
    const unsigned bits = sab_pack_bits(length);
    const u64 blocks = ((u64)length + 127) / 128, words = blocks * 4ull * bits;
    if (magic != SAB_PACK_MAGIC || dlen != nbytes - 16 || dlen > words * 4 || length == 0 || length > sa_cap) {
        sab_set_error("sab200_unpack: not a packed suffix array (magic %08x, length %u, %llu data bytes)", magic, length,
                      (unsigned long long)dlen);
        return SAB_ERR_ARGS;
    }
    SabUse u;
    SAB_TRY(sab_use(0, &u));
    const size_t in_bytes = sab_align_up((size_t)words * 4 + 64, 256);
    u32 *d_in, *d_sa;
    SAB_TRY(sab_arena_carve(u.c, {{&d_in, in_bytes}, {&d_sa, (size_t)length * 4}}));
    cudaStream_t st = u.c->stream;
    SAB_CUDA_TRY(cudaMemsetAsync(d_in, 0, in_bytes, st));  // re-pads the trimmed tail (src/packed_sa.rs:80-85)
    if (dlen) SAB_CUDA_TRY(cudaMemcpyAsync(d_in, bytes + 16, dlen, cudaMemcpyHostToDevice, st));
    SAB_LAUNCH(unpack_blocks_kernel, (unsigned)div_up64(length, 256), 256, 0, st, (const u32*)d_in, (u64)length, bits, d_sa);
    SAB_LAUNCH_CHECK();
    SAB_CUDA_TRY(cudaMemcpyAsync(sa, d_sa, (size_t)length * 4, cudaMemcpyDeviceToHost, st));
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    *sa_len = length;
    return SAB_OK;
}

extern "C" {

int32_t sab200_get_stats(sab200_stats* out) {
    if (!out) return SAB_ERR_ARGS;
    memcpy(out, &g_last_stats, sizeof(*out));
    return SAB_OK;
}

void sab200_set_profiling(int32_t on) { g_profiling = on != 0; }

const char* sab200_last_error(void) { return g_err; }

int32_t sab200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char* sab200_version(void) {
#ifdef SAB_EMU
    return "sab200 0.1.0 (SIMT emulator build -- tests only)";
#else
    return "sab200 0.1.0 (sm_100a)";
#endif
}

void sab200_shutdown(void) {
    sab_multi_shutdown();
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    for (int d = 0; d < SAB_MAX_DEVICES; ++d) {
        if (g_ctx[d]) {
            sab_context_destroy(g_ctx[d]);
            g_ctx[d] = nullptr;
        }
    }
}

}  // extern "C"

#include "sab_index.cuh"
#include "sab_dist.cuh"
