// sab_sort.cuh -- host driver of the LSD radix sort over a double buffer.
#pragma once
#include "sab_context.cuh"
#include "sab_radix.cuh"

template <typename KeyT>
struct SortBuffers {
    KeyT* k[2];
    u32* v[2];
    int cur;  // index of the buffers holding the live data
};

// tile shape of the pass kernel (see DESIGN.md "onesweep tile")
template <typename KeyT>
struct PassShape;
#ifndef SAB_PASS_THREADS
#define SAB_PASS_THREADS 256
#endif
// 18 items: 4608-record tiles (longer per-bin runs, fewer partial sectors), 64 KB of shared memory, still
// 3 CTAs/SM and 80 registers (8 bytes of spill).  Measured on the 1 GiB text: 14 items 3263 GB/s, 16: 3401,
// 18: 3547, 20: 3217 (profiles/r02_ab_radix_variants*.txt).
#ifndef SAB_PASS_ITEMS
#define SAB_PASS_ITEMS 18
#endif
template <>
struct PassShape<u64> {
    static constexpr int THREADS = SAB_PASS_THREADS, ITEMS = SAB_PASS_ITEMS;
};
template <>
struct PassShape<u32> {
    static constexpr int THREADS = SAB_PASS_THREADS, ITEMS = SAB_PASS_ITEMS;
};

template <typename KeyT, bool IOTA, typename DigitOp, bool PEER = false>
static int sab_launch_pass_op(SabContext* c, const KeyT* kin, KeyT* kout, const u32* vin, u32* vout, u64 n, DigitOp dop,
                              const u64* gbase, const PeerOut* peer = nullptr, u32 iota_base = 0) {
    constexpr int THREADS = PassShape<KeyT>::THREADS, ITEMS = PassShape<KeyT>::ITEMS;
    typedef OnesweepCfg<KeyT, true, IOTA, THREADS, ITEMS> Cfg;
    const u64 tiles = div_up64(n, (u64)Cfg::TILE);
    if (c->lb_epoch >= SAB_LB_EPOCH_MAX) {
        SAB_CUDA_TRY(cudaMemsetAsync(c->d_lookback, 0, c->lookback_tiles * SAB_RADIX_BINS * sizeof(u64), c->stream));
        c->lb_epoch = 0;
    }
    const u32 epoch = ++c->lb_epoch;
    auto kern = onesweep_kernel<KeyT, DigitOp, true, IOTA, PEER, THREADS, ITEMS>;
    PeerOut po;
    memset(&po, 0, sizeof(po));
    if (PEER && peer) po = *peer;
#ifndef SAB_EMU
    SAB_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));  // per device
#endif
    sab_prof_begin(c, SAB_PROF_RADIX_PASS);
    SAB_LAUNCH(kern, (unsigned)tiles, THREADS, Cfg::SMEM, c->stream, kin, kout, vin, vout, n, dop, gbase,
               c->d_lookback, c->d_ticket, c->ticket_host, epoch, po, iota_base);
    sab_prof_end(c);
    SAB_LAUNCH_CHECK();
    c->ticket_host += (u32)tiles;
    c->stats.radix_pass_launches += 1;
    c->stats.radix_pass_records += n;
    // algorithmic bytes (SURVEY.md 8d): read K+V, write K+V -- the first pass of a sort generates its payload
    // (iota) instead of reading it
    c->stats.radix_pass_bytes += ((IOTA ? 1ull : 2ull) * sizeof(u32) + 2ull * sizeof(KeyT)) * n;
    c->stats.kernel_launches += 1;
    return SAB_OK;
}

template <typename KeyT, bool IOTA>
static int sab_launch_pass(SabContext* c, const KeyT* kin, KeyT* kout, const u32* vin, u32* vout, u64 n, int shift,
                           const u64* gbase) {
    ShiftDigit<KeyT> dop;
    dop.shift = shift;
    return sab_launch_pass_op<KeyT, IOTA, ShiftDigit<KeyT> >(c, kin, kout, vin, vout, n, dop, gbase);
}

// Sorts the n records (k[cur], v[cur]) by key bits [begin_bit, end_bit), stable, ascending.  When
// `iota` is set the incoming payload is ignored and taken to be 0..n-1.  On return buf.cur names
// the buffers holding the result.  *passes_out receives the number of passes actually executed
// (digit places where all keys agree are skipped).  Synchronises the stream once (skip flags).
// final_v (optional): the LAST executed pass writes its payload there instead of into the double buffer (the
// suffix array itself: the sorted indices need no copy afterwards); *final_used tells whether a pass did.
template <typename KeyT>
static int sab_radix_sort(SabContext* c, SortBuffers<KeyT>& buf, u64 n, int begin_bit, int end_bit, bool iota,
                          u32* passes_out, u32* final_v = nullptr, bool* final_used = nullptr) {
    if (passes_out) *passes_out = 0;
    if (final_used) *final_used = false;
    if (n == 0) return SAB_OK;
    const int npass = (end_bit - begin_bit + SAB_RADIX_BITS - 1) / SAB_RADIX_BITS;
    if (npass < 0 || npass > SAB_MAX_PASSES) {
        sab_set_error("radix sort: bad bit range [%d,%d)", begin_bit, end_bit);
        return SAB_ERR_INTERNAL;
    }
    constexpr int TILE = PassShape<KeyT>::THREADS * PassShape<KeyT>::ITEMS;
    SAB_TRY(sab_ensure_lookback(c, (size_t)div_up64(n, TILE)));
    bool payload_ready = !iota;
    if (npass > 0) {
        SAB_CUDA_TRY(cudaMemsetAsync(c->d_ghist, 0, sizeof(u64) * SAB_MAX_PASSES * SAB_RADIX_BINS, c->stream));
        const u64 htile = (u64)SAB_HIST_THREADS * SAB_HIST_ITEMS;
        u64 hblocks = div_up64(n, htile);
        const u64 hmax = (u64)c->sm_count * 4;
        if (hblocks > hmax) hblocks = hmax;
        sab_prof_begin(c, SAB_PROF_HIST);
        SAB_LAUNCH(radix_hist_kernel<KeyT>, (unsigned)hblocks, SAB_HIST_THREADS, 0, c->stream, (const KeyT*)buf.k[buf.cur], n,
                   begin_bit, npass, c->d_ghist);
        SAB_LAUNCH_CHECK();
        SAB_LAUNCH(radix_scan_kernel, 1, SAB_RADIX_BINS, 0, c->stream, (const u64*)c->d_ghist, n, npass, c->d_gbase,
                   c->scratch->skip);
        sab_prof_end(c);
        SAB_LAUNCH_CHECK();
        c->stats.kernel_launches += 2;
        u32 skip[SAB_MAX_PASSES];
        SAB_TRY(sab_read_u32(c, c->scratch->skip, SAB_MAX_PASSES, skip));
        int last = -1;
        for (int p = 0; p < npass; ++p)
            if (!skip[p]) last = p;
        const u32* vsrc = buf.v[buf.cur];
        for (int p = 0; p < npass; ++p) {
            if (skip[p]) continue;
            const int shift = begin_bit + p * SAB_RADIX_BITS;
            const int in = buf.cur, out = buf.cur ^ 1;
            u32* vdst = (p == last && final_v) ? final_v : buf.v[out];
            if (p == last && final_v && final_used) *final_used = true;
            if (!payload_ready) {
                SAB_TRY((sab_launch_pass<KeyT, true>(c, buf.k[in], buf.k[out], nullptr, vdst, n, shift,
                                                     c->d_gbase + p * SAB_RADIX_BINS)));
                payload_ready = true;
            } else {
                SAB_TRY((sab_launch_pass<KeyT, false>(c, buf.k[in], buf.k[out], vsrc, vdst, n, shift,
                                                      c->d_gbase + p * SAB_RADIX_BINS)));
            }
            vsrc = vdst;
            buf.cur = out;
            if (passes_out) *passes_out += 1;
        }
    }
    if (!payload_ready) {
        SAB_LAUNCH(iota_kernel, (unsigned)div_up64(n, 256), 256, 0, c->stream, buf.v[buf.cur], n);
        SAB_LAUNCH_CHECK();
        c->stats.kernel_launches += 1;
    }
    return SAB_OK;
}
