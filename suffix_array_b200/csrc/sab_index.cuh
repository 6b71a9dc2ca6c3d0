// sab_index.cuh -- the resident index of include/sab200.h and its batched queries.  Every replica GPU holds the text,
// the suffix array, the bucket table (if given) and a prefix directory over them, and carves the buffers of a call
// (patterns, offsets, results) from an arena of its own.  The host forms enqueue on every replica, pipelining their
// chunks over the replica's two streams, and then drain them all.
#pragma once
#include "sab_ms.cuh"

struct SabReplica {
    SabContext* ctx = nullptr;
    u8* d_text = nullptr;
    u32* d_sa = nullptr;
    u32* d_bkt = nullptr;
    // prefix directory (sab_search.cuh PrefixDir): built here, never leaves the library
    u32* d_pdir = nullptr;
    u16* d_plut = nullptr;
    unsigned long long* d_probes = nullptr;
    SearchArgs search = {};  // the resident fields: text, n, sa, bkt and the prefix directory
    cudaStream_t stream2 = nullptr;  // second stream: the copies of one chunk of patterns run under the kernel of another
    SabArena scratch;  // the buffers of one call
    // matching-statistics extension, built by the first sab200_matching_statistics_batch* call on the index
    u32* d_isa = nullptr;
    u32* d_lcp = nullptr;
    u32* d_lmin = nullptr;  // the levels of block minima above the LCP array, one after the other
    MsArgs ms = {};         // the resident fields: those of `search`, the extension and its level layout
};
struct sab200_index {
    u64 n = 0;
    bool has_bkt = false;
    bool count_probes = false;
    bool has_ms = false;  // every replica holds the matching-statistics extension
    std::vector<SabReplica> rep;
    std::mutex mu;
};

static void replica_free(SabReplica& r) {
    if (!r.ctx) return;
    cudaSetDevice(r.ctx->device);
    cudaFree(r.d_text);
    cudaFree(r.d_sa);
    cudaFree(r.d_bkt);
    cudaFree(r.d_pdir);
    cudaFree(r.d_plut);
    cudaFree(r.d_probes);
    cudaFree(r.scratch.base);
    cudaFree(r.d_isa);
    cudaFree(r.d_lcp);
    cudaFree(r.d_lmin);
    if (r.stream2) cudaStreamDestroy(r.stream2);
    r = SabReplica();
}

// The prefix directory over the resident text and suffix array, under the context's lock: alphabet from a byte
// histogram on the device, depth = the most symbols whose codes number at most n / 8 (between 2^16 and 2^27 entries),
// one sweep over the suffix array.  Running out of memory for it is not an error: the queries then bisect the bucket.
static int replica_build_prefix_dir(SabReplica& r, u64 n) {
    SabContext* c = r.ctx;
    cudaStream_t st = c->stream;
    SAB_TRY(sab_launch_alphabet_hist(c, r.d_text, n, c->scratch->hist));
    u32 hist[256];
    SAB_TRY(sab_read_u32(c, c->scratch->hist, 256, hist));
    u16* lut = c->staging->lut;  // pinned: the upload below is asynchronous
    u32 sigma = 0;
    for (int ch = 0; ch < 256; ++ch) {
        const bool present = hist[ch] != 0;
        lut[ch] = (u16)(sigma | (present ? 0x8000u : 0u));
        if (present) ++sigma;
    }
    const u32 base = sigma < 2 ? 2 : sigma;
    u64 limit = n / 8;
    if (limit < (1ull << 16)) limit = 1ull << 16;
    if (limit > (1ull << 27)) limit = 1ull << 27;
    u32 depth = 1;
    u64 entries = base;
    while (depth < SAB_PDIR_MAXD && entries * base <= limit) {
        entries *= base;
        ++depth;
    }
    if (cudaMalloc(&r.d_pdir, (entries + 1) * sizeof(u32)) != cudaSuccess) {
        cudaGetLastError();
        r.d_pdir = nullptr;
        return SAB_OK;
    }
    SAB_CUDA_TRY(cudaMalloc(&r.d_plut, sizeof(c->staging->lut)));
    SAB_CUDA_TRY(cudaMemcpyAsync(r.d_plut, lut, sizeof(c->staging->lut), cudaMemcpyHostToDevice, st));
    SAB_LAUNCH(fill_u32_kernel, sab_grid(c, entries + 1, 256 * 8, 16), 256, 0, st, r.d_pdir, entries + 1, (u32)(n + 1));
    SAB_LAUNCH_CHECK();
    SAB_LAUNCH(prefix_dir_kernel, (unsigned)div_up64(n + 1, 256), 256, 0, st, (const u8*)r.d_text, n, (const u32*)r.d_sa, n + 1,
               (const u16*)r.d_plut, base, depth, r.d_pdir);
    SAB_LAUNCH_CHECK();
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    PrefixDir& pd = r.search.pd;
    pd.dir = r.d_pdir;
    pd.lut = r.d_plut;
    pd.sigma = base;
    pd.depth = depth;
    pd.pw[0] = 1;
    for (u32 t = 1; t <= SAB_PDIR_MAXD; ++t) pd.pw[t] = t <= depth ? pd.pw[t - 1] * base : 0;
    return SAB_OK;
}

static int replica_init(SabReplica& r, int device, const u8* s, u64 n, const u32* sa, const u32* bkt) {
    SabUse u;
    SAB_TRY(sab_use(device, &u));
    r.ctx = u.c;
    cudaStream_t st = r.ctx->stream;
    const size_t text_bytes = sab_align_up((size_t)n + 64, 256);
    SAB_CUDA_TRY(cudaMalloc(&r.d_text, text_bytes));
    SAB_CUDA_TRY(cudaMalloc(&r.d_sa, ((size_t)n + 1) * sizeof(u32)));
    SAB_CUDA_TRY(cudaMemsetAsync(r.d_text, 0, text_bytes, st));
    if (n) SAB_CUDA_TRY(cudaMemcpyAsync(r.d_text, s, n, cudaMemcpyHostToDevice, st));
    SAB_CUDA_TRY(cudaMemcpyAsync(r.d_sa, sa, ((size_t)n + 1) * sizeof(u32), cudaMemcpyHostToDevice, st));
    if (bkt) {
        SAB_CUDA_TRY(cudaMalloc(&r.d_bkt, SAB200_BKT_LEN * sizeof(u32)));
        SAB_CUDA_TRY(cudaMemcpyAsync(r.d_bkt, bkt, SAB200_BKT_LEN * sizeof(u32), cudaMemcpyHostToDevice, st));
    }
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    r.search.text = r.d_text;
    r.search.n = n;
    r.search.sa = r.d_sa;
    r.search.bkt = r.d_bkt;
    SAB_CUDA_TRY(cudaStreamCreateWithFlags(&r.stream2, cudaStreamNonBlocking));
    SAB_CUDA_TRY(cudaMalloc(&r.d_probes, sizeof(unsigned long long)));
    SAB_CUDA_TRY(cudaMemsetAsync(r.d_probes, 0, sizeof(unsigned long long), st));
    const char* off = getenv("SAB_SEARCH_DIR");
    if (n > 0 && !(off && off[0] == '0')) SAB_TRY(replica_build_prefix_dir(r, n));
    return SAB_OK;
}

extern "C" sab200_index* sab200_index_create(const uint8_t* s, uint64_t n, const uint32_t* sa, uint64_t sa_len,
                                             const uint32_t* bkt_or_null, int32_t ngpus) {
    if (!sa || (n > 0 && !s) || n > SAB200_MAX_LENGTH || ngpus < 1 || ngpus > SAB_MAX_DEVICES) {
        sab_set_error("sab200_index_create: bad arguments");
        return nullptr;
    }
    if (sa_len != n + 1) {
        sab_set_error("sab200_index_create: the suffix array has %llu entries, the text needs %llu",
                      (unsigned long long)sa_len, (unsigned long long)(n + 1));
        return nullptr;
    }
    if (ngpus > sab200_device_count()) {
        sab_set_error("sab200_index_create: %d GPUs requested, %d visible", (int)ngpus, (int)sab200_device_count());
        return nullptr;
    }
    sab200_index* ix = new (std::nothrow) sab200_index();
    if (!ix) return nullptr;
    ix->n = n;
    ix->has_bkt = bkt_or_null != nullptr;
    ix->rep.resize(ngpus);
    for (int d = 0; d < ngpus; ++d) {
        if (replica_init(ix->rep[d], d, s, n, sa, bkt_or_null) != SAB_OK) {
            for (auto& r : ix->rep) replica_free(r);
            delete ix;
            return nullptr;
        }
    }
    return ix;
}

extern "C" void sab200_index_destroy(sab200_index* ix) {
    if (!ix) return;
    for (auto& r : ix->rep) replica_free(r);
    delete ix;
}

// The checks every batched entry point makes; `bufs`: the caller's other buffers are given (needed when nq > 0).
static int index_batch_args(const char* who, const char* what, const sab200_index* ix, u64 nq, const u64* offs, bool bufs) {
    if (!ix || (nq > 0 && (!offs || !bufs))) {
        sab_set_error("%s: bad arguments", who);
        return SAB_ERR_ARGS;
    }
    if (nq > 0x7fffffffull) {
        sab_set_error("%s: at most 2^31-1 %s per call", who, what);
        return SAB_ERR_ARGS;
    }
    return SAB_OK;
}

static cudaStream_t replica_stream(const SabReplica& r, int which) { return which ? r.stream2 : r.ctx->stream; }

// waits for both streams of every replica
static int index_drain(sab200_index* ix) {
    for (auto& r : ix->rep) {
        SAB_CUDA_TRY(cudaSetDevice(r.ctx->device));
        SAB_CUDA_TRY(cudaStreamSynchronize(r.ctx->stream));
        SAB_CUDA_TRY(cudaStreamSynchronize(r.stream2));
    }
    return SAB_OK;
}

template <int MODE>
static int launch_search(const SabReplica& r, bool count_probes, const u8* d_pats_adj, const u64* d_offs, u64 np, u32* d_out0,
                         u32* d_out1, cudaStream_t st) {
    SearchArgs a = r.search;
    a.probes = count_probes ? r.d_probes : nullptr;
    a.pats = d_pats_adj;
    a.offs = d_offs;
    a.np = np;
    a.out0 = d_out0;
    a.out1 = d_out1;
    const u64 threads = np * SAB_SEARCH_G;
    SAB_LAUNCH((search_kernel<SAB_SEARCH_G, MODE>), (unsigned)div_up64(threads, SAB_SEARCH_THREADS), SAB_SEARCH_THREADS, 0, st, a);
    SAB_LAUNCH_CHECK();
    return SAB_OK;
}

#ifndef SAB_SEARCH_CHUNK
#define SAB_SEARCH_CHUNK (1ull << 20)  // patterns per pipelined chunk
#endif

// mode 0 search_all (out0 = lo, out1 = hi), 1 contains (out0 = u8 flags), 2 search_lcp (start, end)
static int search_batch(sab200_index* ix, int mode, const u8* pats, const u64* offs, u64 np, void* out0, void* out1) {
    SAB_TRY(index_batch_args("batched search", "patterns", ix, np, offs, out0 && (mode == 1 || out1)));
    if (np == 0) return SAB_OK;
    std::lock_guard<std::mutex> lk(ix->mu);
    const int P = (int)ix->rep.size();
    const u64 per = div_up64(np, (u64)P);
    // enqueue on every replica, then drain
    for (int d = 0; d < P; ++d) {
        const u64 q0 = (u64)d * per, q1 = (q0 + per < np) ? q0 + per : np;
        if (q0 >= q1) continue;
        SabReplica& r = ix->rep[d];
        SAB_CUDA_TRY(cudaSetDevice(r.ctx->device));
        const u64 b0 = offs[q0], b1 = offs[q1];
        const u64 cnt = q1 - q0;
        u8* d_pats;
        u64* d_offs0;
        u32 *d_out0, *d_out1;
        // every pipelined chunk keeps its own end offset
        SAB_TRY(sab_arena_carve(&r.scratch, r.ctx->stream,
                                {{&d_pats, (size_t)(b1 - b0) + 64}, {&d_offs0, ((size_t)cnt + cnt / SAB_SEARCH_CHUNK + 2) * sizeof(u64)},
                                 {&d_out0, (size_t)cnt * sizeof(u32)}, {&d_out1, (size_t)cnt * sizeof(u32)}}));
        // Chunks of SAB_SEARCH_CHUNK patterns alternate between two streams: the pattern upload of one chunk and
        // the result download of another run under the kernel of a third (pinned caller buffers; PCIe is full
        // duplex).  Every chunk owns its sub-ranges of the scratch buffers, so the streams never meet.
        const u8* adj = d_pats - b0;  // the kernel indexes patterns by their absolute offsets
        int which = 0;
        for (u64 c0 = 0; c0 < cnt; c0 += SAB_SEARCH_CHUNK, which ^= 1) {
            const u64 c1 = c0 + SAB_SEARCH_CHUNK < cnt ? c0 + SAB_SEARCH_CHUNK : cnt;
            const u64 cc = c1 - c0;
            const u64 cb0 = offs[q0 + c0], cb1 = offs[q0 + c1];
            cudaStream_t st = replica_stream(r, which);
            if (cb1 > cb0) SAB_CUDA_TRY(cudaMemcpyAsync(d_pats + (cb0 - b0), pats + cb0, cb1 - cb0, cudaMemcpyHostToDevice, st));
            // chunk c reads offs[c0 .. c1]; entry c1 is also the first of the next chunk, which lives one slot further
            u64* d_offs = d_offs0 + c0 + c0 / SAB_SEARCH_CHUNK;
            SAB_CUDA_TRY(cudaMemcpyAsync(d_offs, offs + q0 + c0, (cc + 1) * sizeof(u64), cudaMemcpyHostToDevice, st));
            u32* o0 = d_out0 + c0;
            u32* o1 = d_out1 + c0;
            if (mode == 0) SAB_TRY(launch_search<0>(r, ix->count_probes, adj, d_offs, cc, o0, o1, st));
            else if (mode == 1) SAB_TRY(launch_search<1>(r, false, adj, d_offs, cc, (u32*)((u8*)d_out0 + c0), o1, st));
            else SAB_TRY(launch_search<2>(r, false, adj, d_offs, cc, o0, o1, st));
            if (mode == 1) {
                SAB_CUDA_TRY(cudaMemcpyAsync((u8*)out0 + q0 + c0, (u8*)d_out0 + c0, cc, cudaMemcpyDeviceToHost, st));
            } else {
                SAB_CUDA_TRY(cudaMemcpyAsync((u32*)out0 + q0 + c0, o0, cc * sizeof(u32), cudaMemcpyDeviceToHost, st));
                SAB_CUDA_TRY(cudaMemcpyAsync((u32*)out1 + q0 + c0, o1, cc * sizeof(u32), cudaMemcpyDeviceToHost, st));
            }
        }
    }
    return index_drain(ix);
}

extern "C" int32_t sab200_search_all_batch(sab200_index* ix, const uint8_t* pats, const uint64_t* offs, uint64_t np, uint32_t* lo,
                                uint32_t* hi) {
    return search_batch(ix, 0, pats, offs, np, lo, hi);
}
extern "C" int32_t sab200_contains_batch(sab200_index* ix, const uint8_t* pats, const uint64_t* offs, uint64_t np, uint8_t* out) {
    return search_batch(ix, 1, pats, offs, np, out, nullptr);
}
extern "C" int32_t sab200_search_lcp_batch(sab200_index* ix, const uint8_t* pats, const uint64_t* offs, uint64_t np,
                                uint32_t* start, uint32_t* end) {
    return search_batch(ix, 2, pats, offs, np, start, end);
}

// Device-resident variant for timing the kernel alone: d_pats / d_offs / d_lo / d_hi live on the
// device of replica 0; d_pats must be followed by >= 8 readable bytes.
extern "C" int32_t sab200_search_all_batch_device(sab200_index* ix, const uint8_t* d_pats, const uint64_t* d_offs, uint64_t np,
                                       uint32_t* d_lo, uint32_t* d_hi) {
    if (!ix || !d_offs || !d_lo || !d_hi) return SAB_ERR_ARGS;
    if (np == 0) return SAB_OK;
    std::lock_guard<std::mutex> lk(ix->mu);
    SabReplica& r = ix->rep[0];
    SAB_CUDA_TRY(cudaSetDevice(r.ctx->device));
    SAB_TRY(launch_search<0>(r, ix->count_probes, d_pats, d_offs, np, d_lo, d_hi, r.ctx->stream));
    SAB_CUDA_TRY(cudaStreamSynchronize(r.ctx->stream));
    return SAB_OK;
}

// Probe counting for the roofline of the search kernel (bench.py): while on, search_all adds the suffix comparisons
// of every pattern to a device counter (one atomic per pattern -- not for timed runs); returns the sum over the
// replicas since the index was created.
extern "C" uint64_t sab200_index_probes(sab200_index* ix, int32_t count_on) {
    if (!ix) return 0;
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->count_probes = count_on != 0;
    u64 total = 0;
    for (auto& r : ix->rep) {
        unsigned long long v = 0;
        cudaSetDevice(r.ctx->device);
        cudaStreamSynchronize(r.ctx->stream);
        if (cudaMemcpy(&v, r.d_probes, sizeof(v), cudaMemcpyDeviceToHost) == cudaSuccess) total += v;
    }
    return total;
}

// Layout of the prefix directory of replica 0: *sigma = base, *depth = symbols per code; returns the number of
// entries (0: no directory).
extern "C" uint64_t sab200_index_directory(sab200_index* ix, uint32_t* sigma, uint32_t* depth) {
    if (!ix || ix->rep.empty() || !ix->rep[0].search.pd.dir) return 0;
    const PrefixDir& pd = ix->rep[0].search.pd;
    if (sigma) *sigma = pd.sigma;
    if (depth) *depth = pd.depth;
    return pd.pw[pd.depth];
}

// ---- matching statistics ----------------------------------------------------------------------
static void replica_free_ms(SabReplica& r) {
    cudaFree(r.d_isa);
    cudaFree(r.d_lcp);
    cudaFree(r.d_lmin);
    r.d_isa = r.d_lcp = r.d_lmin = nullptr;
}

// isa by the integrity check (a wrong suffix array is refused here, before anything scatters through it), the LCP
// array by Kasai from that isa, then the block minima level by level up to the first level of at most 256 entries.
static int replica_build_ms_run(SabReplica& r, u64 n) {
    SabUse u;
    SAB_TRY(sab_use(r.ctx->device, &u));
    SabContext* c = u.c;
    MsArgs a = {};
    a.s = r.search;
    u64 extra = 0;  // entries of the levels above the LCP array
    a.cnt[0] = n + 1;
    while (a.cnt[a.top] > 256) {
        a.cnt[a.top + 1] = div_up64(a.cnt[a.top], 256);
        extra += a.cnt[++a.top];
    }
    const size_t arr = ((size_t)n + 2) * sizeof(u32);
    if (cudaMalloc(&r.d_isa, arr) != cudaSuccess || cudaMalloc(&r.d_lcp, arr) != cudaSuccess ||
        cudaMalloc(&r.d_lmin, (size_t)(extra + 1) * sizeof(u32)) != cudaSuccess) {
        cudaGetLastError();
        sab_set_error("matching statistics: the index extension (%zu bytes) does not fit on device %d",
                      2 * arr + (size_t)(extra + 1) * sizeof(u32), c->device);
        return SAB_ERR_OOM;
    }
    u32 bad;
    SAB_TRY(sab_isa_check(c, r.d_text, n, r.d_sa, n + 1, r.d_isa, &bad));
    if (bad) {
        sab_set_error("matching statistics: the index's suffix array is not the suffix array of its text");
        return SAB_ERR_ARGS;
    }
    SAB_TRY(sab_launch_kasai(c, r.d_text, n, r.d_sa, r.d_isa, r.d_lcp));
    a.isa = r.d_isa;
    a.lvl[0] = r.d_lcp;
    u32* out = r.d_lmin;
    for (u32 k = 1; k <= a.top; out += a.cnt[k], ++k) {
        SAB_LAUNCH(lcp_block_min_kernel, (unsigned)div_up64(a.cnt[k] * 32, 256), 256, 0, c->stream, a.lvl[k - 1], a.cnt[k - 1], out,
                   a.cnt[k]);
        SAB_LAUNCH_CHECK();
        a.lvl[k] = out;
    }
    // the directory narrows a from-scratch search to ~16 suffixes; below its depth a carried interval is no narrower
    a.fresh_below = r.search.pd.dir ? r.search.pd.depth : 1;
    SAB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    r.ms = a;
    return SAB_OK;
}

// The extension on every replica, built once per index (under ix->mu); on failure none is kept.
static int ms_prepare(sab200_index* ix) {
    if (ix->has_ms) return SAB_OK;
    for (auto& r : ix->rep) {
        const int rc = replica_build_ms_run(r, ix->n);
        if (rc != SAB_OK) {
            for (auto& q : ix->rep) replica_free_ms(q);
            return rc;
        }
    }
    ix->has_ms = true;
    return SAB_OK;
}

static MsArgs ms_args(const SabReplica& r, const u8* d_qs_adj, const u64* d_offs, u64 nq) {
    MsArgs a = r.ms;
    a.s.pats = d_qs_adj;
    a.s.offs = d_offs;
    a.s.np = nq;
    return a;
}

static int launch_ms(MsArgs a, u64 p0, u64 p1, u32* len_adj, u32* lo_adj, u32* hi_adj, cudaStream_t st) {
    a.p0 = p0;
    a.p1 = p1;
    a.len = len_adj;
    a.lo = lo_adj;
    a.hi = hi_adj;
    const u64 warps = div_up64(p1 - p0, SAB_MS_CHUNK);
    SAB_LAUNCH(ms_kernel, (unsigned)div_up64(warps * 32, SAB_MS_THREADS), SAB_MS_THREADS, 0, st, a);
    SAB_LAUNCH_CHECK();
    return SAB_OK;
}

#ifndef SAB_MS_SUB
#define SAB_MS_SUB ((u64)SAB_MS_CHUNK << 12)  // positions per pipelined launch (4 Mi: 48 MiB of results)
#endif

extern "C" int32_t sab200_matching_statistics_batch(sab200_index* ix, const uint8_t* qs, const uint64_t* offs, uint64_t nq,
                                                    uint32_t* len, uint32_t* lo, uint32_t* hi) {
    SAB_TRY(index_batch_args("matching statistics", "queries", ix, nq, offs, true));
    if (nq == 0) return SAB_OK;
    for (u64 q = 0; q < nq; ++q)
        if (offs[q + 1] < offs[q]) {
            sab_set_error("matching statistics: the offsets decrease at query %llu", (unsigned long long)q);
            return SAB_ERR_ARGS;
        }
    const u64 b0 = offs[0], b1 = offs[nq];
    if (b1 > b0 && (!qs || !len || !lo || !hi)) {
        sab_set_error("matching statistics: bad arguments");
        return SAB_ERR_ARGS;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    SAB_TRY(ms_prepare(ix));
    if (b1 == b0) return SAB_OK;
    // every replica holds the whole concatenation (a match may run past its share) and walks an equal share of the
    // positions, cut at chunk boundaries
    const int P = (int)ix->rep.size();
    const u64 per = div_up64(div_up64(b1 - b0, SAB_MS_CHUNK), (u64)P) * SAB_MS_CHUNK;
    u8* d_qs[SAB_MAX_DEVICES];
    u64* d_offs[SAB_MAX_DEVICES];
    u32* d_ms[SAB_MAX_DEVICES];  // len / lo / hi of the replica's share, one after the other
    for (int d = 0; d < P; ++d) {
        const u64 s0 = b0 + (u64)d * per;
        if (s0 >= b1) continue;
        const u64 share = b1 - s0 < per ? b1 - s0 : per;
        SabReplica& r = ix->rep[d];
        SAB_CUDA_TRY(cudaSetDevice(r.ctx->device));
        SAB_TRY(sab_arena_carve(&r.scratch, r.ctx->stream,
                                {{&d_qs[d], (size_t)(b1 - b0) + 64}, {&d_offs[d], ((size_t)nq + 1) * sizeof(u64)},
                                 {&d_ms[d], (size_t)share * 3 * sizeof(u32)}}));
        SAB_CUDA_TRY(cudaMemcpyAsync(d_qs[d], qs + b0, b1 - b0, cudaMemcpyHostToDevice, r.ctx->stream));
        SAB_CUDA_TRY(cudaMemcpyAsync(d_offs[d], offs, (nq + 1) * sizeof(u64), cudaMemcpyHostToDevice, r.ctx->stream));
    }
    for (int d = 0; d < P; ++d) {
        const u64 s0 = b0 + (u64)d * per;
        if (s0 >= b1) continue;
        const u64 s1 = b1 - s0 < per ? b1 : s0 + per;
        SabReplica& r = ix->rep[d];
        SAB_CUDA_TRY(cudaSetDevice(r.ctx->device));
        SAB_CUDA_TRY(cudaStreamSynchronize(r.ctx->stream));
        const MsArgs a = ms_args(r, d_qs[d] - b0, d_offs[d], nq);
        u32 *dl = d_ms[d] - s0, *dlo = dl + (s1 - s0), *dhi = dlo + (s1 - s0);  // indexed by absolute position
        // Sub-ranges alternate between two streams: the download of one runs under the kernel of the next, which is
        // launched first so that a pageable destination (a synchronous copy) does not leave the device idle.
        auto download = [&](u64 p0, u64 p1, cudaStream_t st) -> int {
            SAB_CUDA_TRY(cudaMemcpyAsync(len + p0, dl + p0, (p1 - p0) * sizeof(u32), cudaMemcpyDeviceToHost, st));
            SAB_CUDA_TRY(cudaMemcpyAsync(lo + p0, dlo + p0, (p1 - p0) * sizeof(u32), cudaMemcpyDeviceToHost, st));
            SAB_CUDA_TRY(cudaMemcpyAsync(hi + p0, dhi + p0, (p1 - p0) * sizeof(u32), cudaMemcpyDeviceToHost, st));
            return SAB_OK;
        };
        u64 prev0 = 0, prev1 = 0;
        cudaStream_t prev_st = nullptr;
        int which = 0;
        for (u64 p0 = s0; p0 < s1; p0 += SAB_MS_SUB, which ^= 1) {
            const u64 p1 = s1 - p0 < SAB_MS_SUB ? s1 : p0 + SAB_MS_SUB;
            cudaStream_t st = replica_stream(r, which);
            SAB_TRY(launch_ms(a, p0, p1, dl, dlo, dhi, st));
            if (prev1 > prev0) SAB_TRY(download(prev0, prev1, prev_st));
            prev0 = p0;
            prev1 = p1;
            prev_st = st;
        }
        SAB_TRY(download(prev0, prev1, prev_st));
    }
    return index_drain(ix);
}

// Device-resident form on the GPU of replica 0: d_qs is indexed by the absolute offsets and followed by at least
// 8 readable bytes; d_len / d_lo / d_hi are indexed by absolute position.
extern "C" int32_t sab200_matching_statistics_batch_device(sab200_index* ix, const uint8_t* d_qs, const uint64_t* d_offs, uint64_t nq,
                                                           uint32_t* d_len, uint32_t* d_lo, uint32_t* d_hi) {
    SAB_TRY(index_batch_args("matching statistics", "queries", ix, nq, d_offs, d_qs && d_len && d_lo && d_hi));
    if (nq == 0) return SAB_OK;
    std::lock_guard<std::mutex> lk(ix->mu);
    SAB_TRY(ms_prepare(ix));
    SabReplica& r = ix->rep[0];
    SabUse u;
    SAB_TRY(sab_use(r.ctx->device, &u));
    cudaStream_t st = u.c->stream;
    u32* flag = &u.c->scratch->ms_offs;
    SAB_CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(u32), st));
    SAB_LAUNCH(ms_offs_check_kernel, (unsigned)div_up64(nq, 256), 256, 0, st, (const u64*)d_offs, nq, flag);
    SAB_LAUNCH_CHECK();
    u64 ends[2];
    SAB_CUDA_TRY(cudaMemcpyAsync(&ends[0], d_offs, sizeof(u64), cudaMemcpyDeviceToHost, st));
    SAB_CUDA_TRY(cudaMemcpyAsync(&ends[1], d_offs + nq, sizeof(u64), cudaMemcpyDeviceToHost, st));
    u32 bad;
    SAB_TRY(sab_read_u32(u.c, flag, 1, &bad));
    if (bad) {
        sab_set_error("matching statistics: the offsets decrease");
        return SAB_ERR_ARGS;
    }
    if (ends[1] == ends[0]) return SAB_OK;
    SAB_TRY(launch_ms(ms_args(r, d_qs, d_offs, nq), ends[0], ends[1], d_len, d_lo, d_hi, st));
    SAB_CUDA_TRY(cudaStreamSynchronize(st));
    return SAB_OK;
}
