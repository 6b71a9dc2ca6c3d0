// sab_group_sort.cuh -- sorting the records of a doubling round without a full radix sort.
//
// In a round the records arrive grouped by their first rank r1 (the high word of the 64-bit key) and only
// have to be ordered by the second rank INSIDE each group.  Eight radix passes over every record (192 B of
// traffic per record) are wasted work when the groups are small (1 GiB DNA-like text: mean < 3 records) or
// of moderate size (256 MiB repetitive text: the ~256 copies of one block offset):
//
//   group_sort_kernel   one sweep (24 B per record).  A tile of 2048 records is staged in shared memory and
//                       cut into groups by a ballot scan of the head flags.  A tile OWNS the groups whose
//                       head lies inside it: the tail of a group that runs over the tile border is fetched
//                       by the owner (<= SAB_GSORT_MID records) and skipped by the next tile; both tiles
//                       decide "fits" from the same total size, each by scanning outwards from the border.
//                         size <= SAB_GSORT_MAX (32): every record takes its slot by counting the group
//                           members that precede it in (key, position) order -- O(s) shared-memory reads;
//                         size <= SAB_GSORT_MID (512): one warp sorts the group as (r2, index) words in
//                           registers -- a bitonic network, strides >= 32 inside a lane, < 32 by shuffles
//                           (the order of records with equal keys is irrelevant: they stay one group);
//                         larger groups: the records are compacted in list order (chained scan) into spare
//                           buffers together with their positions.
//   scatter_back_kernel after the radix sort of those "big" records: the j-th sorted record returns to the
//                       j-th recorded position (sorting by (r1, r2) keeps every group in its own range; on a
//                       list that is not ascending in r1 the positions are first sorted by the r1 of their
//                       record, see sab_group_sort).
//
// Measured and rejected (profiles/r02_ab_round2_group_sort.txt): publishing the big-record counts before the sorting
// so that the look-back runs beside the sorting warps -- 256 MiB repetitive text 45.4 -> 49.6 ms, 1 GiB DNA-like
// text 1.8 -> 2.0 ms (the spinning look-back warp costs more issue slots than the barrier it removes).
//
// No reference counterpart: it replaces part of the work of divsufsort's group refinement
// (third-party crate behind /root/reference/src/saca.rs:14).
#pragma once
#include "sab_scan_kernels.cuh"
#include "sab_sort.cuh"

#ifndef SAB_GSORT_MAX
#define SAB_GSORT_MAX 32  // largest group ordered by the counting rank
#endif
#ifndef SAB_GSORT_MID
#define SAB_GSORT_MID 512  // largest group ordered by one warp in registers (64, 128, 256 or 512)
#endif
#define SAB_GSORT_THREADS 256
#define SAB_GSORT_ITEMS 8
#define SAB_GSORT_TILE (SAB_GSORT_THREADS * SAB_GSORT_ITEMS)
#define SAB_GSORT_CAP (SAB_GSORT_TILE + SAB_GSORT_MID)  // tile + the tail of its last group
#define SAB_GSORT_MIDLIST 96  // more than SAB_GSORT_CAP / (SAB_GSORT_MAX + 1) groups of moderate size per tile
// keys + payloads as they arrive, second ranks + payloads in output order (the first rank of a slot does not change:
// a record only moves inside its group), head positions, list of the groups of moderate size: 54.7 KB, 4 CTAs / SM
#define SAB_GSORT_SMEM ((SAB_GSORT_CAP + 2) * 8 + SAB_GSORT_CAP * 4 * 3 + (SAB_GSORT_TILE + 8) * 2 + SAB_GSORT_MIDLIST * 2)
#define SAB_GSORT_NOGROUP 0xffffffffu  // never a rank (ranks are <= n <= 2^32 - 2)
static_assert(SAB_GSORT_MID < SAB_GSORT_TILE && SAB_GSORT_MID >= SAB_GSORT_MAX, "a group the owner completes is shorter than a tile");
static_assert(SAB_GSORT_CAP / (SAB_GSORT_MAX + 1) < SAB_GSORT_MIDLIST, "list of the groups of moderate size");
static_assert(SAB_GSORT_THREADS == SAB_SCAN_THREADS, "warp_aggregates is sized for the scan kernels' block");

struct CountOp {
    __device__ __forceinline__ u32 operator()(u32 a, u32 b) const { return a + b; }
};

// One warp orders `size` (<= 32 * IPL) records of one group, staged at s_in/s_vin, by (second rank, index) and
// writes second ranks and indices to s_out/s_vout.  Element e of the group lives in register e / 32 of lane e % 32, so a
// compare-exchange at distance >= 32 stays inside the lane and one at distance < 32 is a shuffle.
template <int IPL>
__device__ __forceinline__ void warp_sort_group(const u64* s_in, const u32* s_vin, u32* s_out, u32* s_vout, u32 size, u32 lane) {
    u64 x[IPL];
#pragma unroll
    for (int j = 0; j < IPL; ++j) {
        const u32 e = (u32)j * 32u + lane;
        x[j] = e < size ? ((s_in[e] << 32) | (u64)s_vin[e]) : ~0ull;  // padding sorts behind every record
    }
#pragma unroll
    for (int k = 2; k <= 32 * IPL; k <<= 1) {
#pragma unroll
        for (int s = k >> 1; s > 0; s >>= 1) {
            if (s >= 32) {
#pragma unroll
                for (int j = 0; j < IPL; ++j) {
                    if ((j & (s >> 5)) == 0) {
                        const int jp = j | (s >> 5);
                        const bool asc = ((j << 5) & k) == 0;
                        const u64 a = x[j], b = x[jp];
                        const bool sw = (a > b) == asc;
                        x[j] = sw ? b : a;
                        x[jp] = sw ? a : b;
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < IPL; ++j) {
                    const u64 y = __shfl_xor_sync(SAB_FULL, x[j], s);
                    const bool asc = ((((u32)j << 5) | lane) & (u32)k) == 0;
                    const bool lower = (lane & (u32)s) == 0;
                    const bool take_min = lower == asc;
                    x[j] = ((x[j] < y) == take_min) ? x[j] : y;  // the words are distinct (they carry the index)
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < IPL; ++j) {
        const u32 e = (u32)j * 32u + lane;
        if (e < size) {
            s_out[e] = (u32)(x[j] >> 32);
            s_vout[e] = (u32)x[j];
        }
    }
}

// Record p of the staged tile, member of group g (an index into s_heads; < 0: the group began in an earlier
// tile): a record of a small group takes its output slot, a record of a big group keeps its place.  Returns
// whether the record belongs to a big group.
__device__ __forceinline__ bool gsort_place(const u64* s_key, const u32* s_val, u32* s_or2, u32* s_oval, const u16* s_heads, u32 p,
                                            int g, u32 G, u32 tail_big, u32 lead_big) {
    const u64 key = s_key[p + 1];
    bool big = false;
    if (g < 0) {
        big = lead_big != 0;  // else: ordered and written by the tile that owns the head
    } else {
        const u32 a = s_heads[g], b = s_heads[g + 1];
        if (((u32)g + 1 == G && tail_big) || b - a > SAB_GSORT_MID) {
            big = true;
        } else if (b - a <= SAB_GSORT_MAX) {
            u32 before = 0;
            for (u32 q = a; q < b; ++q) {
                const u64 o = s_key[q + 1];
                before += (o < key || (o == key && q < p)) ? 1u : 0u;
            }
            s_or2[a + before] = (u32)key;
            s_oval[a + before] = s_val[p];
        }
    }
    if (big) {
        s_or2[p] = (u32)key;
        s_oval[p] = s_val[p];
    }
    return big;
}

__global__ void __launch_bounds__(SAB_GSORT_THREADS)
group_sort_kernel(const u64* __restrict__ kin, const u32* __restrict__ vin, u64 m, u64* __restrict__ kout,
                  u32* __restrict__ vout, u64* __restrict__ big_k, u32* __restrict__ big_v, u32* __restrict__ big_pos,
                  u32 big_cap, u32* __restrict__ d_nbig, TileState<u32> st) {
    SAB_DYN_SMEM(smem);
    u64* s_key = (u64*)smem;                    // [0] the record before the tile, [1 + p] record p of the tile (+ tail)
    u32* s_val = (u32*)(s_key + SAB_GSORT_CAP + 2);
    u32* s_or2 = s_val + SAB_GSORT_CAP;         // second ranks and payloads in output order
    u32* s_oval = s_or2 + SAB_GSORT_CAP;
    u16* s_heads = (u16*)(s_oval + SAB_GSORT_CAP);  // positions of the group heads inside the tile, then the end
    u16* s_mid = s_heads + SAB_GSORT_TILE + 8;      // groups of moderate size (all but the tile's last group)
    SAB_SHARED_ARRAY(u32, s_edge, 4);           // tail length, tail group is big, leading records to skip, ... are big
    SAB_SHARED_VAR(u32, s_nmid);
    const u32 tile = blockIdx.x, tid = threadIdx.x, lane = lane_id(), w = warp_id();
    const u64 base = (u64)tile * SAB_GSORT_TILE;
    const u32 valid = (m - base < (u64)SAB_GSORT_TILE) ? (u32)(m - base) : (u32)SAB_GSORT_TILE;
    const u64 none = (u64)SAB_GSORT_NOGROUP << 32;
#pragma unroll
    for (int k = 0; k < SAB_GSORT_ITEMS; ++k) {
        const u32 p = tid + k * SAB_GSORT_THREADS;
        if (p < valid) {
            s_key[p + 1] = kin[base + p];
            s_val[p] = vin[base + p];
        }
    }
    if (tid == 0) {
        s_key[0] = base > 0 ? kin[base - 1] : none;
        s_nmid = 0;
    }
    // the 32 records behind the tile (warp 0) and the 32 keys in front of it (warp 1) are requested together with
    // the tile: step 2 below normally needs no more than these, so it adds no round trip of its own
    u64 edge_key = none;
    u32 edge_val = 0;
    if (w == 0 && base + valid + lane < m) {
        edge_key = kin[base + valid + lane];
        edge_val = vin[base + valid + lane];
    } else if (w == 1 && base >= (u64)lane + 1) {
        edge_key = kin[base - 1 - lane];
    }
    __syncthreads();

    // 1. group heads.  Warp w owns records [w*256, (w+1)*256) of the tile; item k of lane l is record w*256 + k*32 + l.
    u32 hb[SAB_GSORT_ITEMS];
    u32 mine = 0;
#pragma unroll
    for (int k = 0; k < SAB_GSORT_ITEMS; ++k) {
        const u32 p = w * (32 * SAB_GSORT_ITEMS) + k * 32 + lane;
        const bool head = p < valid && (u32)(s_key[p + 1] >> 32) != (u32)(s_key[p] >> 32);
        hb[k] = __ballot_sync(SAB_FULL, head);
        mine += (u32)__popc(hb[k]);
    }
    u32 hpre, G;
    warp_aggregates<u32, CountOp>(mine, CountOp(), 0u, hpre, G);
    int gidx[SAB_GSORT_ITEMS];  // group of my item k: index into s_heads, -1 = the group began in an earlier tile
    {
        u32 run = hpre;
#pragma unroll
        for (int k = 0; k < SAB_GSORT_ITEMS; ++k) {
            const u32 p = w * (32 * SAB_GSORT_ITEMS) + k * 32 + lane;
            if ((hb[k] >> lane) & 1u) s_heads[run + (u32)__popc(hb[k] & lanemask_lt())] = (u16)p;
            gidx[k] = (int)(run + (u32)__popc(hb[k] & lanemask_le())) - 1;
            run += (u32)__popc(hb[k]);
        }
    }
    __syncthreads();

    // 2. the groups on the tile borders: warp 0 looks past the end, warp 1 before the start
    if (w == 0) {
        u32 ext = 0, tail_big = 0;
        if (G > 0 && base + valid < m) {
            const u32 T = valid - (u32)s_heads[G - 1];
            const u32 r1t = (u32)(s_key[valid] >> 32);
            if (T > SAB_GSORT_MID) {
                tail_big = 1;
            } else {
                const u32 budget = SAB_GSORT_MID - T + 1;  // one more equal record than fits means "too large"
                bool found = false;
                for (u32 off = 0; off < budget; off += 32) {
                    const u32 j = off + lane;
                    const u64 g = base + valid + j;
                    bool eq = j < budget && g < m;
                    if (eq) {
                        const u64 key = off == 0 ? edge_key : kin[g];
                        eq = (u32)(key >> 32) == r1t;
                        if (eq && valid + j < SAB_GSORT_CAP) {
                            s_key[valid + 1 + j] = key;
                            s_val[valid + j] = off == 0 ? edge_val : vin[g];
                        }
                    }
                    const u32 bal = __ballot_sync(SAB_FULL, eq);
                    if (bal != SAB_FULL) {
                        const u32 jf = off + (u32)(__ffs((int)~bal) - 1);
                        if (jf >= budget) tail_big = 1;
                        else ext = jf;
                        found = true;
                        break;
                    }
                }
                if (!found) tail_big = 1;
            }
        }
        if (lane == 0) {
            s_edge[0] = ext;
            s_edge[1] = tail_big;
            s_heads[G] = (u16)(valid + ext);
        }
    } else if (w == 1) {
        u32 skip = 0, lead_big = 0;
        const u32 L = G > 0 ? (u32)s_heads[0] : valid;  // records of a group that began before this tile
        if (L > 0) {
            const u32 r1f = (u32)(s_key[1] >> 32);
            if (L > SAB_GSORT_MID) {
                lead_big = 1;
            } else {
                const u32 budget = SAB_GSORT_MID - L + 1;
                bool found = false;
                for (u32 off = 0; off < budget; off += 32) {
                    const u32 j = off + lane;
                    bool eq = j < budget && base >= (u64)j + 1;
                    if (eq) eq = (u32)((off == 0 ? edge_key : kin[base - 1 - j]) >> 32) == r1f;
                    const u32 bal = __ballot_sync(SAB_FULL, eq);
                    if (bal != SAB_FULL) {
                        const u32 jf = off + (u32)(__ffs((int)~bal) - 1);
                        if (jf >= budget) lead_big = 1;
                        else skip = L;  // jf + L records in all: the tile of the head completes and writes the group
                        found = true;
                        break;
                    }
                }
                if (!found) lead_big = 1;
            }
        }
        if (lane == 0) {
            s_edge[2] = skip;
            s_edge[3] = lead_big;
        }
    } else {
        // meanwhile the other warps list the groups of moderate size (the tile's last group is not complete yet)
        for (u32 g = (w - 2) * 32 + lane; g + 1 < G; g += (SAB_SCAN_WARPS - 2) * 32) {
            const u32 size = (u32)s_heads[g + 1] - (u32)s_heads[g];
            if (size > SAB_GSORT_MAX && size <= SAB_GSORT_MID) s_mid[atomicAdd(&s_nmid, 1u)] = (u16)g;
        }
    }
    __syncthreads();
    const u32 ext = s_edge[0], tail_big = s_edge[1], skip = s_edge[2], lead_big = s_edge[3];
    const u32 cnt = valid + ext;

    // 3. small groups by the counting rank; records of big groups keep their place (the scatter-back overwrites it)
    u32 bigb[SAB_GSORT_ITEMS];
    mine = 0;
#pragma unroll
    for (int k = 0; k < SAB_GSORT_ITEMS; ++k) {
        const u32 p = w * (32 * SAB_GSORT_ITEMS) + k * 32 + lane;
        const bool big = p < valid && gsort_place(s_key, s_val, s_or2, s_oval, s_heads, p, gidx[k], G, tail_big, lead_big);
        bigb[k] = __ballot_sync(SAB_FULL, big);
        mine += (u32)__popc(bigb[k]);
    }
    // the fetched tail of the last group (a group that is small or of moderate size: never "big")
    if (tid < ext) gsort_place(s_key, s_val, s_or2, s_oval, s_heads, valid + tid, (int)G - 1, G, tail_big, lead_big);

    // 4. groups of moderate size: one warp each, in registers (taking them from a shared counter instead of
    // striding by warp measured neutral, r02_ab_final_1gpu.txt _dyn)
    const u32 nmid = s_nmid;
    for (u32 t = w; t <= nmid; t += SAB_SCAN_WARPS) {
        u32 g;
        if (t < nmid) {
            g = s_mid[t];
        } else {  // the tile's last group, now that its tail is known
            if (G == 0 || tail_big) break;
            g = G - 1;
        }
        const u32 a = s_heads[g], size = (u32)s_heads[g + 1] - a;
        if (size <= SAB_GSORT_MAX || size > SAB_GSORT_MID) continue;
        if (size <= 64) warp_sort_group<2>(s_key + 1 + a, s_val + a, s_or2 + a, s_oval + a, size, lane);
        else if (size <= 128) warp_sort_group<4>(s_key + 1 + a, s_val + a, s_or2 + a, s_oval + a, size, lane);
#if SAB_GSORT_MID > 128
        else if (size <= 256) warp_sort_group<8>(s_key + 1 + a, s_val + a, s_or2 + a, s_oval + a, size, lane);
#endif
#if SAB_GSORT_MID > 256
        else warp_sort_group<16>(s_key + 1 + a, s_val + a, s_or2 + a, s_oval + a, size, lane);
#endif
    }

    // 5. records of big groups, compacted in list order
    u32 wpre, total;
    warp_aggregates<u32, CountOp>(mine, CountOp(), 0u, wpre, total);
    const u32 prefix = tile_exclusive_prefix<u32, CountOp>(st, tile, total, CountOp(), 0u);
    u32 run = prefix + wpre;
#pragma unroll
    for (int k = 0; k < SAB_GSORT_ITEMS; ++k) {
        const u32 p = w * (32 * SAB_GSORT_ITEMS) + k * 32 + lane;
        if ((bigb[k] >> lane) & 1u) {
            const u32 j = run + (u32)__popc(bigb[k] & lanemask_lt());
            if (j < big_cap) {
                big_k[j] = s_key[p + 1];
                big_v[j] = s_val[p];
                big_pos[j] = (u32)(base + p);
            }
        }
        run += (u32)__popc(bigb[k]);
    }
    if (tid == 0 && base + SAB_GSORT_TILE >= m) *d_nbig = prefix + total;  // last tile
    __syncthreads();
    for (u32 p = skip + tid; p < cnt; p += SAB_GSORT_THREADS) {
        kout[base + p] = (s_key[p + 1] & 0xffffffff00000000ull) | (u64)s_or2[p];  // a slot keeps its first rank
        vout[base + p] = s_oval[p];
    }
}

__global__ void __launch_bounds__(256)
scatter_back_kernel(const u64* __restrict__ big_k, const u32* __restrict__ big_v, const u32* __restrict__ big_pos, u32 nbig,
                    u64* __restrict__ kout, u32* __restrict__ vout) {
    const u32 j = blockIdx.x * 256u + threadIdx.x;
    if (j < nbig) {
        const u32 pos = big_pos[j];
        kout[pos] = big_k[j];
        vout[pos] = big_v[j];
    }
}

// Spare memory for the records of big groups: two key and two payload buffers (radix ping-pong) and the
// position list, `cap` records each.
struct GroupSortSpare {
    u64* k[2];
    u32* v[2];
    u32* pos;
    u64 cap;
};

// Sorts the cnt records of (sb.k[0], sb.v[0]) -- grouped by the high key word -- by the full key.
// `ascending`: the groups arrive in ascending order of the high word, so the j-th radix-sorted large-group record
// belongs at the j-th recorded position.  Otherwise (a list of two ascending runs after a split-filter round) the
// recorded positions are first sorted by the high word of their record (a stable radix sort of a second copy of
// the keys with the positions as payload), which needs twice the spare room.
// Returns 1 with the result in (sb.k[1], sb.v[1]) and sb.cur = 1; returns 0 with the input untouched when
// the records of big groups do not fit the spare buffers (the caller falls back to the radix sort); < 0 on error.
// *nbig_out = number of records that needed the radix sort.
static int sab_group_sort(SabContext* c, SortBuffers<u64>& sb, u64 cnt, int key_bits, const GroupSortSpare& sp,
                          u32* passes_out, u64* nbig_out, bool ascending = true) {
    const u64 tiles = div_up64(cnt, SAB_GSORT_TILE);
    SAB_TRY(sab_ensure_scan(c, (size_t)tiles));
    TileState<u32> ts = sab_tile_state<u32>(c, tiles);
    const u32 cap = sp.cap > 0xffffffffull ? 0xffffffffu : (u32)sp.cap;
#ifndef SAB_EMU
    SAB_CUDA_TRY(cudaFuncSetAttribute(group_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SAB_GSORT_SMEM));
#endif
    sab_prof_begin(c, SAB_PROF_GROUP_SORT);
    SAB_LAUNCH(group_sort_kernel, (unsigned)tiles, SAB_GSORT_THREADS, SAB_GSORT_SMEM, c->stream, (const u64*)sb.k[0],
               (const u32*)sb.v[0], cnt, sb.k[1], sb.v[1], sp.k[0], sp.v[0], sp.pos, cap, &c->scratch->big, ts);
    sab_prof_end(c);
    SAB_LAUNCH_CHECK();
    c->stats.kernel_launches++;
    u32 nbig;
    SAB_TRY(sab_read_u32(c, &c->scratch->big, 1, &nbig));
    c->stats.group_sort_records += cnt;
    c->stats.group_big_records += nbig;
    *nbig_out = nbig;
    if (passes_out) *passes_out = 0;
    if (nbig > sp.cap) return 0;
    if (nbig > 0) {
        const u32* sorted_pos = sp.pos;
        const u64 half = (sp.cap / 2) & ~(u64)63;
        if (!ascending) {
            if (nbig > half) return 0;
            SAB_CUDA_TRY(cudaMemcpyAsync(sp.k[0] + half, sp.k[0], nbig * sizeof(u64), cudaMemcpyDeviceToDevice, c->stream));
        }
        SortBuffers<u64> bb;
        bb.k[0] = sp.k[0];
        bb.k[1] = sp.k[1];
        bb.v[0] = sp.v[0];
        bb.v[1] = sp.v[1];
        bb.cur = 0;
        SAB_TRY(sab_radix_sort<u64>(c, bb, nbig, 0, key_bits, /*iota=*/false, passes_out));
        if (!ascending) {
            SortBuffers<u64> pb;  // (key copy, position) by the high word only: the positions in the order of their groups
            pb.k[0] = sp.k[0] + half;
            pb.k[1] = sp.k[1] + half;
            pb.v[0] = sp.pos;
            pb.v[1] = sp.v[0] + half;
            pb.cur = 0;
            u32 pos_passes = 0;
            SAB_TRY(sab_radix_sort<u64>(c, pb, nbig, 32, key_bits, /*iota=*/false, &pos_passes));
            sorted_pos = pb.v[pb.cur];
        }
        sab_prof_begin(c, SAB_PROF_GROUP_SORT);
        SAB_LAUNCH(scatter_back_kernel, (unsigned)div_up64(nbig, 256), 256, 0, c->stream, (const u64*)bb.k[bb.cur],
                   (const u32*)bb.v[bb.cur], sorted_pos, (u32)nbig, sb.k[1], sb.v[1]);
        sab_prof_end(c);
        SAB_LAUNCH_CHECK();
        c->stats.kernel_launches++;
    }
    sb.cur = 1;
    return 1;
}
