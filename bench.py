#!/usr/bin/env python3
"""bench.py -- headline benchmark of the hot path (BASELINE.json): suffix-array construction
throughput in MB/s of text, next to the CPU baseline, with the roofline of the dominant kernel.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c1|c3|c4]

A "step" = one construction of the suffix array of one synthetic text.  At N=1 the workload is
BASELINE.json configs[1]: 1 GiB DNA-like text (sigma=4) on one B200.  N>1 (launched by torchrun, one
process per GPU): the SAME text block-sharded over the N GPUs (strong scaling), built by the distributed
driver inside libsab200 (NCCL all-to-all per round); the line also carries a `c4` sub-record (the 3.9 GiB
text of configs[3]) and the batched search of configs[4] sharded over N replicas.  ONE JSON line on rank 0.

  value  = whole-job MB/s with the text already resident in HBM
  e2e    = the same metric through the reference-facing C ABI call with HOST buffers
           (sab200_saca / sab200_saca_sharded: host text -> device -> host SA inside the timed region)
  roofline     = the onesweep radix pass: algorithmic bytes (2*(K+V)*m; (2K+V)*m for the first pass of a sort,
                 whose payload is generated) / CUDA-event time on the library's stream, against
                 MEASURED_PEAKS.json hbm_gbs
  cpu_baseline = the oracle port (single thread, like divsufsort) on a bounded prefix of the text
  verified     = the benchmarked output checked once, outside the timed region (sab200_check on the GPU,
                 oracle sufcheck on the CPU for the 1 GiB text)

--dump-outputs DIR writes what the timed path returned in its last step as DIR/<name>.npy (float64, exact for
32-bit values), so that two builds can be compared output for output on the same inputs (the texts and patterns
are pure functions of their seeds):
  suffix_array                      the suffix array (n + 1 entries) at sampled positions
  search_<set>_lo / search_<set>_hi the batched search_all ranges of each pattern set, at sampled queries
A sample is the sorted distinct positions np.unique(gen.splitmix64(DUMP_SEED, 0, k) % size); an output of at most
k entries is written whole.  At most 48 MiB in all.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C4_BYTES = int(3.9 * (1 << 30))  # 4 187 593 113: the u32 index limit configuration

WORKLOADS = {
    "c4": ("3.9 GiB mixed text (first half uniform bytes, second half English-like), BASELINE.json configs[3]",
           C4_BYTES, "mixed"),
    "c2": ("1 GiB DNA-like text (sigma=4, planted repeats), BASELINE.json configs[1]", 1 << 30, "dna_like"),
    "c1": ("64 MiB uniform-random bytes (sigma=256), BASELINE.json configs[0]", 64 << 20, "uniform_bytes"),
    "c3": ("256 MiB repetitive text (1 MiB block, 1e-4 mutations), BASELINE.json configs[2]", 256 << 20, "repetitive"),
}
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only if MEASURED_PEAKS.json is absent
METRIC = "sa_construction_throughput"
DTYPE = "u8 text / u64 keys / u32 ranks"
DUMP_SEED = 0xD0D0
DUMP_SA_ENTRIES = 4 << 20       # 32 MiB of float64
DUMP_SEARCH_QUERIES = 1 << 19   # 4 MiB per array, four arrays


def make_text(workload, n, seed_shift=0):
    from suffix_array_b200 import gen
    fn = getattr(gen, WORKLOADS[workload][2])
    seed = {"c1": gen.SEED_C1, "c2": gen.SEED_C2, "c3": gen.SEED_C3, "c4": gen.SEED_C4}[workload] + seed_shift
    return fn(n, seed)


def load_profile(name):
    try:
        with open(os.path.join(ROOT, "profiles", name)) as f:
            return json.load(f)
    except Exception:
        return None


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def dump_positions(size, k):
    """The fixed sample of an output of `size` entries that --dump-outputs writes (see the module docstring)."""
    from suffix_array_b200 import gen
    if size <= k:
        return np.arange(size, dtype=np.int64)
    return np.unique(gen.splitmix64(DUMP_SEED, 0, k) % np.uint64(size)).astype(np.int64)


def write_outputs(path, outputs):
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


def pinned(n, dtype):
    import torch
    t = torch.empty(int(n), dtype=dtype, pin_memory=True)
    return t, t.numpy()


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (the recipe's clocks line).

    ONE long-lived `nvidia-smi -lms` process, started before the warm-up steps: a fresh nvidia-smi per sample
    initialises NVML on every GPU of the box each time and was seen to stall short multi-GPU steps.  Only the
    rows between begin() and end() are reported."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.all_rows = []
        self.t_begin = self.t_end = None
        self.proc = None

    def begin(self):
        self.t_begin = time.perf_counter()

    def end(self):
        self.t_end = time.perf_counter()
        self.stop_flag.set()
        if self.proc is not None:
            self.proc.terminate()

    @property
    def rows(self):
        lo = self.t_begin if self.t_begin is not None else 0.0
        hi = self.t_end if self.t_end is not None else float("inf")
        inside = [r for t, r in self.all_rows if lo <= t <= hi]
        return inside if inside else [r for _, r in self.all_rows[-1:]]  # region shorter than one period

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 7:
                    self.all_rows.append((time.perf_counter(), parts))
                if self.stop_flag.is_set():
                    break
        except Exception:
            pass

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_baseline_run(text, sample_bytes):
    """Times the oracle port (oracle/sa_oracle.c, single thread) on the first sample_bytes of text."""
    from oracle import oracle
    sample = np.ascontiguousarray(text[:sample_bytes])
    oracle.lib()
    t0 = time.perf_counter()
    sa = oracle.saca(sample)
    dt = time.perf_counter() - t0
    assert int(sa[0]) == sample.size
    return sample.size / 1e6 / dt, dt


def cpu_all_cores_run(text, sample_bytes):
    """The "all cores" column (north_star names psacak, which is not available here): the OpenMP prefix-doubling
    port of oracle/sa_parallel.cpp with every host thread, on the same prefix as the single-thread figure."""
    from oracle import oracle
    sample = np.ascontiguousarray(text[:sample_bytes])
    try:
        t0 = time.perf_counter()
        sa, threads = oracle.saca_parallel(sample)
        dt = time.perf_counter() - t0
    except Exception as e:  # noqa: BLE001 -- a box without the OpenMP runtime reports it instead of failing the line
        return {"unavailable": str(e)[:200]}
    assert int(sa[0]) == sample.size
    return {"value": round(sample.size / 1e6 / dt, 3), "unit": "MB/s", "cores": threads, "kind": "port",
            "sample": "first %d MiB of the same text (%.1f s)" % (sample_bytes >> 20, dt),
            "note": "OpenMP prefix doubling (oracle/sa_parallel.cpp); psacak, the all-cores SACA north_star names, "
                    "is not a dependency of the reference and not installable here"}


def config_of(workload, n, n_mib):
    desc = WORKLOADS[workload][0]
    return {"workload": desc if not n_mib else "%s at %d MiB" % (workload, n_mib), "text_bytes": n}


def run_reference(args, rank, world):
    """`--impl reference`: the reference's CPU path.  The reference cannot be compiled here (Rust crate; its SACA
    is the un-vendored cdivsufsort 2.0 = libdivsufsort, single-threaded), so this times the oracle port on the
    host cores -- one thread, as the reference uses -- on the SAME text as the GPU arm.  Each step sorts a
    bounded prefix of that text (the whole run must end within minutes: 25 full-size constructions would take
    ~40 minutes); `--ref-full` adds ONE full-size construction, reported as cpu_baseline.full_size."""
    if rank != 0:
        return
    desc, n_full, _ = WORKLOADS[args.workload]
    if args.n_mib:
        n_full = args.n_mib << 20
    sample_bytes = min(n_full, args.ref_sample_mib << 20)
    text = make_text(args.workload, n_full if (args.ref_full or args.workload == "c2") else sample_bytes)
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_baseline_run(text, min(sample_bytes, 1 << 20))
    times = []
    for _ in range(args.steps):
        _, dt = cpu_baseline_run(text, sample_bytes)
        times.append(dt)
    ms = 1e3 * float(np.mean(times))
    v = sample_bytes / 1e6 / (ms / 1e3)
    sample = "first %d MiB of the same text per step, oracle SA-IS port, 1 thread" % (sample_bytes >> 20)
    cpu = {"value": round(v, 3), "unit": "MB/s", "cores": 1, "kind": "port", "sample": sample,
           "note": "the reference's libdivsufsort (single thread) is not buildable here (no Rust / crate sources)"}
    cpu["all_cores"] = cpu_all_cores_run(text, sample_bytes)
    if args.ref_full:
        vf, dtf = cpu_baseline_run(text, n_full)
        cpu["full_size"] = {"value": round(vf, 3), "unit": "MB/s", "seconds": round(dtf, 1), "text_bytes": n_full}
    else:
        cpu["full_size"] = (load_profile("r02_reference_full_size.json") or {}).get("full_size")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": "MB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": config_of(args.workload, n_full, args.n_mib), "cpu_baseline": cpu,
        "e2e": {"value": round(v, 3), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------ search (C5)
def search_bytes(bkt, pats, offs, n):
    """SURVEY.md 8d: algorithmic bytes of a batch = sum over queries of 2*ceil(log2(hi0-lo0)) * (4 + min(|pat|, 32)),
    (lo0, hi0) = the bucket range of the query; sector-level = the same probes * 32 B * (1 + ceil(|pat|/32))."""
    lens = (offs[1:] - offs[:-1]).astype(np.int64)
    o = offs[:-1].astype(np.int64)
    two = lens >= 2
    last = max(pats.size - 1, 0)
    c0 = pats[np.minimum(o, last)].astype(np.int64)
    c1 = pats[np.minimum(o + 1, last)].astype(np.int64)
    idx = c0 * 257 + c1 + 2
    lo0 = np.where(two, bkt[np.maximum(idx - 1, 0)], 0).astype(np.int64)
    hi0 = np.where(two, bkt[idx], n + 1).astype(np.int64)
    width = np.maximum(hi0 - lo0, 1)
    probes = 2 * np.ceil(np.log2(width)).astype(np.int64)
    algo = int((probes * (4 + np.minimum(lens, 32))).sum())
    sector = int((probes * 32 * (1 + (lens + 31) // 32)).sum())
    return algo, sector, int(probes.sum())


def bench_search(L, _lib, torch, dev, text, sa, n, ngpus, npat, outputs, sample=1_000_000):
    """BASELINE.json configs[4]: batched search_all of `npat` patterns (len 8..64) on the finished index with
    enable_buckets, sharded over `ngpus` replicas (one process, no collective).  Two pattern sets (SURVEY.md 8d):
    half substrings + half hybrids whose second half is random symbols of the text's alphabet, and the
    reference's own hybrid (raw random bytes, benches/utils.rs:193-197).  (lo, hi) of a sample is compared
    with the oracle's restatement of src/sa.rs:173-204.  The host-ABI ranges of the last call go to `outputs`
    (None: not kept)."""
    from suffix_array_b200 import gen
    from oracle import oracle
    bkt = np.empty(_lib.BKT_LEN, dtype=np.uint32)
    _lib.check(L.sab200_enable_buckets(text.ctypes.data, n, bkt.ctypes.data), "sab200_enable_buckets")
    t0 = time.perf_counter()
    ix = L.sab200_index_create(text.ctypes.data, n, sa.ctypes.data, n + 1, bkt.ctypes.data, ngpus)
    create_ms = (time.perf_counter() - t0) * 1e3
    if not ix:
        return {"error": L.sab200_last_error().decode()}
    peak, _ = hbm_peak()
    out = {"patterns": npat, "len": "8..64", "replicas": ngpus, "buckets": True,
           "index_create_ms": round(create_ms, 1),
           "index_create_note": "upload of text + suffix array + bucket table from pageable memory and the prefix directory, per replica; not in the timed region"}
    for name, alphabet in (("alphabet_hybrid", None), ("raw_byte_hybrid", np.arange(256, dtype=np.uint8))):
        pats, offs = gen.patterns(text, npat, alphabet=alphabet)
        _, hp = pinned(pats.size + 64, torch.uint8)
        hp[:pats.size] = pats
        _, ho = pinned(offs.size, torch.int64)
        ho[:] = offs.view(np.int64)
        _, lo = pinned(npat, torch.int32)
        _, hi = pinned(npat, torch.int32)
        lo, hi = lo.view(np.uint32), hi.view(np.uint32)
        host_s = 1e9
        for _ in range(3):  # the first call also allocates the device-side pattern / result buffers
            t0 = time.perf_counter()
            _lib.check(L.sab200_search_all_batch(ix, hp.ctypes.data, ho.ctypes.data, npat, lo.ctypes.data, hi.ctypes.data), "search")
            host_s = min(host_s, time.perf_counter() - t0)
        if outputs is not None:
            q = dump_positions(npat, DUMP_SEARCH_QUERIES)
            outputs["search_%s_lo" % name] = lo[q]
            outputs["search_%s_hi" % name] = hi[q]
        rec = {"hit_fraction": round(float((hi > lo).mean()), 3), "queries_per_s_host_abi": round(npat / host_s, 1),
               "h2d_bytes": int(pats.size + 8 * offs.size), "d2h_bytes": 8 * npat}
        if ngpus == 1:
            d_p = torch.zeros(pats.size + 64, dtype=torch.uint8, device=dev)
            d_p[:pats.size] = torch.from_numpy(pats).to(dev)
            d_o = torch.from_numpy(offs.view(np.int64)).to(dev)
            d_lo = torch.empty(npat, dtype=torch.int32, device=dev)
            d_hi = torch.empty(npat, dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            best = 1e9
            for _ in range(4):
                t0 = time.perf_counter()
                _lib.check(L.sab200_search_all_batch_device(ix, d_p.data_ptr(), d_o.data_ptr(), npat, d_lo.data_ptr(), d_hi.data_ptr()), "search_dev")
                best = min(best, time.perf_counter() - t0)
            ref_algo, ref_sector, ref_probes = search_bytes(bkt, pats, offs, n)
            # probes the kernel really makes (it starts from the prefix directory of the resident index, not from the
            # whole bucket): counted by the kernel itself in one extra, untimed pass
            p0 = L.sab200_index_probes(ix, 1)
            _lib.check(L.sab200_search_all_batch_device(ix, d_p.data_ptr(), d_o.data_ptr(), npat, d_lo.data_ptr(), d_hi.data_ptr()), "search_dev")
            probes = int(L.sab200_index_probes(ix, 0) - p0)
            lens = (offs[1:] - offs[:-1]).astype(np.int64)
            per_probe = float((4 + np.minimum(lens, 32)).mean())
            per_probe_sector = float((32 * (1 + (lens + 31) // 32)).mean())
            algo = int(probes * per_probe + 16 * npat)        # + two bucket and two directory entries per query
            sector = int(probes * per_probe_sector + 3 * 32 * npat)
            rec.update({"queries_per_s_kernel": round(npat / best, 1), "kernel_ms": round(best * 1e3, 3),
                        "device_equals_host": bool(np.array_equal(d_lo.cpu().numpy().view(np.uint32), lo)),
                        "roofline": {"bound": "hbm (dependent random 32-byte sectors)", "kernel": "search_kernel<4, search_all> (4 lanes per pattern)",
                                     "probes": probes, "probes_per_query": round(probes / npat, 2),
                                     "algorithmic_bytes": algo, "sector_bytes": sector,
                                     "achieved": round(algo / 1e9 / best, 1), "achieved_sector": round(sector / 1e9 / best, 1),
                                     "peak": peak, "unit": "GB/s", "frac": round(algo / 1e9 / best / peak, 4),
                                     "frac_sector": round(sector / 1e9 / best / peak, 4),
                                     "formula": "probes counted by the kernel * (4 + min(|pat|,32)) B (SURVEY.md 8d per-probe bytes) "
                                                "+ 16 B of bucket / directory entries per query; sector-level 32 B*(1+ceil(|pat|/32)) "
                                                "per probe + 3 sectors per query",
                                     "reference_bisection": {"probes": ref_probes, "algorithmic_bytes": ref_algo, "sector_bytes": ref_sector,
                                                             "note": "SURVEY.md 8d as written: 2*ceil(log2(bucket)) probes per query -- what "
                                                                     "bisecting the whole two-byte bucket (src/sa.rs:181-201) would read"}}})
            sg, dp = ctypes.c_uint32(), ctypes.c_uint32()
            ent = int(L.sab200_index_directory(ix, ctypes.byref(sg), ctypes.byref(dp)))
            out["prefix_directory"] = {"entries": ent, "base": int(sg.value), "depth": int(dp.value)}
            del d_p, d_o, d_lo, d_hi
        ns = min(sample, npat)
        so = offs[:ns + 1]
        elo, ehi = oracle.search_all_batch(text, sa, bkt, pats[:int(so[-1])], so)
        rec["oracle_equal_on_sample"] = bool(np.array_equal(lo[:ns], elo) and np.array_equal(hi[:ns], ehi))
        rec["oracle_sample"] = ns
        out[name] = rec
    L.sab200_index_destroy(ix)
    return out


# ------------------------------------------------------------------------------------------------ N = 1
def verify_host(L, _lib, text, sa, n, with_oracle):
    """The benchmarked output, checked once outside the timed region."""
    ok = L.sab200_check(text.ctypes.data, n, sa.ctypes.data, n + 1) == 1
    rec = {"verified": bool(ok), "verifier": "sab200_check (GPU, linear-time equivalent of check_integrity, src/sa.rs:72-84)"}
    if with_oracle:
        from oracle import oracle
        t0 = time.perf_counter()
        okc = bool(oracle.sufcheck(text, sa))
        rec["oracle_sufcheck"] = okc
        rec["oracle_sufcheck_s"] = round(time.perf_counter() - t0, 1)
        rec["verified"] = bool(ok and okc)
    return rec


def run_single_c4(args, L, _lib, torch, dev):
    """BASELINE.json configs[3] on ONE GPU: the 3.9 GiB text needs 156 GB of the 180 GB for the construction, so
    there is no device-resident leg: host-buffer entry only, `value` from the library's own CUDA events around
    the device pipeline (stats.total_ms), e2e = the whole call."""
    desc, n, _ = WORKLOADS["c4"]
    if args.n_mib:
        n = args.n_mib << 20
    from suffix_array_b200 import gen
    text_t, text = pinned(n, torch.uint8)
    text[:] = gen.mixed_range(n, 0, n)
    sa_t, sa = pinned(n + 1, torch.int32)
    sa = sa.view(np.uint32)
    L.sab200_set_profiling(0)
    sampler = ClockSampler(dev.index)
    sampler.start()
    wu = min(args.warmup, 1)
    for _ in range(wu):
        _lib.check(L.sab200_saca(text.ctypes.data, n, sa.ctypes.data, 1), "sab200_saca")
    sampler.begin()
    dev_ms, e2e_ms, launches = [], [], 0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        _lib.check(L.sab200_saca(text.ctypes.data, n, sa.ctypes.data, 1), "sab200_saca")
        e2e_ms.append((time.perf_counter() - t0) * 1e3)
        st = _lib.last_stats()
        dev_ms.append(st["total_ms"])
        launches += st["kernel_launches"]
    sampler.end()
    sampler.join(timeout=2)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"suffix_array": sa[dump_positions(n + 1, DUMP_SA_ENTRIES)]})
    ver = verify_host(L, _lib, text, sa, n, with_oracle=False)
    d, e = float(np.mean(dev_ms)), float(np.mean(e2e_ms))
    print(json.dumps({
        "metric": METRIC, "value": round(n / 1e6 / (d / 1e3), 2), "unit": "MB/s", "n_gpus": 1, "steps": args.steps,
        "warmup": wu, "ms_per_step": round(d, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": DTYPE, "data": "synthetic",
        "config": dict(config_of("c4", n, args.n_mib), per_gpu="single GPU, host-buffer entry only (156 GB of HBM)",
                       l2="inputs larger than L2 (no flush needed)", rounds=st["rounds"], active=st["active"], sigma=st["sigma"],
                       symbols_per_key=st["symbols_per_key"], timing="value: CUDA events around the device pipeline inside sab200_saca"),
        "e2e": {"value": round(n / 1e6 / (e / 1e3), 2), "unit": "MB/s", "ms_per_step": round(e, 3), "h2d_bytes_per_step": n,
                "d2h_bytes_per_step": 4 * (n + 1), "api": "sab200_saca (host buffers, pinned)"},
        "roofline": None, "cpu_baseline": None, "gpu_launches": int(launches), "verification": ver, "verified": ver["verified"],
        "clocks": sampler.summary()}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: c2 (BASELINE.json configs[1]) at every N; c4 = the 3.9 GiB text of configs[3]")
    ap.add_argument("--n-mib", type=int, default=0, help="override the text size (MiB); 0 = the named config")
    ap.add_argument("--ref-sample-mib", type=int, default=64)
    ap.add_argument("--ref-full", action="store_true", help="reference arm: also time ONE full-size construction")
    ap.add_argument("--cpu-sample-mib", type=int, default=128)
    ap.add_argument("--patterns", type=int, default=10_000_000, help="C5: batched search_all patterns")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-search", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="N>1: skip the 3.9 GiB sub-record")
    ap.add_argument("--no-oracle-verify", action="store_true")
    ap.add_argument("--api-gpus", type=int, default=1,
                    help="N=1 process: the ngpus argument of the host-buffer leg, sab200_saca(s, n, sa, ngpus) -- "
                         "one process driving several GPUs through the reference seam")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of what the timed path returned in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload is None:
        # the same text at every N, so that the driver's 1 -> 8 GPU ratio is a strong-scaling figure of one workload
        args.workload = "c2"
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from suffix_array_b200 import _lib
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L = _lib.require_gpu()
    if world > 1:
        run_distributed(args, L, _lib, torch, dist, rank, local_rank, world)
        dist.destroy_process_group()
        return
    dev = torch.device("cuda", local_rank)
    desc, n, _ = WORKLOADS[args.workload]
    if args.n_mib:
        n = args.n_mib << 20
    if args.workload == "c4" and n > (3 << 30):
        run_single_c4(args, L, _lib, torch, dev)
        return
    text = make_text(args.workload, n)
    h_text_t, h_text = pinned(n, torch.uint8)
    h_text[:] = text
    h_sa_t, h_sa = pinned(n + 1, torch.int32)
    h_sa = h_sa.view(np.uint32)
    d_text = h_text_t.to(dev)
    d_sa = torch.empty(n + 1, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    def step_device():
        _lib.check(L.sab200_saca_device(d_text.data_ptr(), n, d_sa.data_ptr(), local_rank), "sab200_saca_device")

    def step_e2e(t_ptr, s_ptr):
        _lib.check(L.sab200_saca(t_ptr, n, s_ptr, args.api_gpus), "sab200_saca")

    # ---- device-resident timing (value) + roofline of the radix pass
    sampler = ClockSampler(local_rank)
    sampler.start()
    L.sab200_set_profiling(0)
    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    sampler.begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    e0.record()
    for _ in range(args.steps):
        step_device()   # blocks until the library's stream has drained
        launches += _lib.last_stats()["kernel_launches"]
    e1.record()
    torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1) / args.steps
    outputs = None
    if args.dump_outputs:
        pos = torch.from_numpy(dump_positions(n + 1, DUMP_SA_ENTRIES)).to(dev)
        outputs = {"suffix_array": d_sa.index_select(0, pos).cpu().numpy().view(np.uint32)}
    # per-launch CUDA events of the radix passes: separate steps (the events cost a few %)
    L.sab200_set_profiling(1)
    pass_ms = pass_bytes = pass_launches = 0
    prof_steps = min(3, args.steps)
    for _ in range(prof_steps):
        step_device()
        st = _lib.last_stats()
        pass_ms += st["radix_pass_ms"]
        pass_bytes += st["radix_pass_bytes"]
        pass_launches += st["radix_pass_launches"]
    stats = _lib.last_stats()
    prof_total_ms = stats["total_ms"]
    L.sab200_set_profiling(0)
    # ---- end-to-end through the C ABI with host buffers: pinned, then pageable (what a Rust Vec<u32> is)
    for _ in range(min(args.warmup, 2)):
        step_e2e(h_text.ctypes.data, h_sa.ctypes.data)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e(h_text.ctypes.data, h_sa.ctypes.data)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    e2e_stats = _lib.last_stats()
    sampler.end()
    sampler.join(timeout=2)
    assert int(h_sa[0]) == n
    ver = verify_host(L, _lib, text, h_sa, n, with_oracle=(args.workload == "c2" and not args.n_mib and not args.no_oracle_verify))
    p_sa = np.zeros(n + 1, dtype=np.uint32)
    p_sa[::1024] = 1  # touch the pages: the reference allocates vec![0u32; n + 1] (src/sa.rs:24)
    pg = []
    for _ in range(min(3, args.steps)):
        t0 = time.perf_counter()
        step_e2e(text.ctypes.data, p_sa.ctypes.data)
        pg.append((time.perf_counter() - t0) * 1e3)
    pageable_ms = float(np.mean(pg))
    pageable_ok = bool(np.array_equal(p_sa, h_sa))
    del p_sa
    total_mb = n / 1e6
    value = total_mb / (dev_ms / 1e3)
    e2e = total_mb / (e2e_ms / 1e3)
    peak, peak_src = hbm_peak()
    achieved = (pass_bytes / 1e9) / (pass_ms / 1e3) if pass_ms > 0 else 0.0
    traffic = load_profile("r02_traffic.json") or load_profile("r01_traffic.json") or {}

    search = None
    if not args.no_search:
        del d_sa
        torch.cuda.empty_cache()
        search = bench_search(L, _lib, torch, dev, text, h_sa, n, 1, args.patterns, outputs)
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)

    cpu = None
    if not args.no_cpu_baseline:
        sb = min(n, args.cpu_sample_mib << 20)
        v, dt = cpu_baseline_run(text, sb)
        cpu = {"value": round(v, 3), "unit": "MB/s", "cores": 1, "kind": "port",
               "sample": "first %d MiB of the same text, oracle SA-IS port, 1 thread (%.1f s)" % (sb >> 20, dt),
               "full_size": (load_profile("r02_reference_full_size.json") or {}).get("full_size"),
               "all_cores": cpu_all_cores_run(text, sb)}
    print(json.dumps({
        "metric": METRIC, "value": round(value, 2), "unit": "MB/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dev_ms, 3), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": dict(config_of(args.workload, n, args.n_mib), per_gpu="single GPU",
                       l2="inputs larger than L2 (no flush needed)" if n > (126 << 20) else "working set 36n bytes > L2",
                       rounds=stats["rounds"], radix_passes=stats["passes"], active=stats["active"],
                       sigma=stats["sigma"], symbols_per_key=stats["symbols_per_key"]),
        "roofline": {"bound": "hbm", "kernel": "onesweep_kernel<u64,u32> (LSD radix pass)", "achieved": round(achieved, 1),
                     "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                     "traffic": traffic.get("traffic") if args.workload == "c2" and not args.n_mib else None,
                     "traffic_note": traffic.get("note"),
                     "peak_source": peak_src, "bytes_per_record": "24 (20 for the first pass of a sort: generated payload)",
                     "launches": int(pass_launches), "avg_launch_ms": round(pass_ms / max(1, pass_launches), 4),
                     "share_of_step": round(pass_ms / prof_steps / prof_total_ms, 3) if prof_total_ms else None,
                     "timing": "CUDA events around every pass launch on the library stream, %d separate steps with "
                               "profiling on; the headline steps run with profiling off" % prof_steps},
        "e2e": {"value": round(e2e, 2), "unit": "MB/s", "ms_per_step": round(e2e_ms, 3), "h2d_bytes_per_step": n,
                "d2h_bytes_per_step": 4 * (n + 1), "api": "sab200_saca (host buffers, pinned, ngpus=%d)" % args.api_gpus,
                "h2d_ms": round(e2e_stats["h2d_ms"], 2), "device_ms": round(e2e_stats["total_ms"], 2), "d2h_ms": round(e2e_stats["d2h_ms"], 2),
                "pageable": {"value": round(total_mb / (pageable_ms / 1e3), 2), "ms_per_step": round(pageable_ms, 3),
                             "equals_pinned_result": pageable_ok,
                             "note": "plain malloc'ed text and suffix array, as the Rust seam hands them over"}},
        "cpu_baseline": cpu, "gpu_launches": int(launches), "search": search,
        "verification": ver, "verified": ver["verified"],
        "breakdown_ms": {k: round(stats[k], 3) for k in ("total_ms", "radix_pass_ms", "hist_ms", "pack_ms", "rank_ms", "gather_ms", "group_sort_ms")},
        "group_sort": {"records": stats["group_sort_records"], "in_large_groups": stats["group_big_records"]},
        "clocks": sampler.summary()}))


# ------------------------------------------------------------------------------------------------ N > 1
def gather_to_rank0(dist, gloo, rank, world, arr, total_len, off, dtype):
    """Host-side gather over a gloo group (verification only): rank 0 returns an array of total_len entries with
    every rank's `arr` at its offset `off`."""
    import torch
    arr = np.ascontiguousarray(arr)
    meta = torch.tensor([int(off), int(arr.size)], dtype=torch.int64)
    metas = [torch.empty_like(meta) for _ in range(world)]
    dist.all_gather(metas, meta, group=gloo)
    out = None
    if rank == 0:
        out = np.empty(total_len, dtype=dtype)
        out[int(off):int(off) + arr.size] = arr
        for r in range(1, world):
            o, c = int(metas[r][0]), int(metas[r][1])
            if c:
                dist.recv(torch.from_numpy(out[o:o + c]), src=r, group=gloo)
    elif arr.size:
        dist.send(torch.from_numpy(arr), dst=0, group=gloo)
    return out


def dist_case(L, _lib, torch, dist, gloo, comm, rank, local_rank, world, workload, n, steps, warmup, sampler, oracle_verify):
    """Device-resident and host-buffer timing of one text sharded over the ranks + verification of the output."""
    from suffix_array_b200 import dist as sdist, gen
    dev = torch.device("cuda", local_rank)
    B, lo, hi = sdist.shard_bounds(n, rank, world)
    end = min(n, hi + sdist.HALO)
    if workload == "c4":
        shard = gen.mixed_range(n, lo, end)      # every rank generates only its own shard
    else:
        shard = make_text(workload, n)[lo:end]
    h_shard_t, h_shard = pinned(shard.size, torch.uint8)
    h_shard[:] = shard
    d_shard = h_shard_t.to(dev)
    torch.cuda.synchronize()

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def allred(x, op):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    L.sab200_set_profiling(0)
    for _ in range(warmup):
        comm.saca(d_shard, n)
    barrier()
    if sampler is not None:
        sampler.begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    lib_ms = 0.0
    host = {"wall_ms": 0.0, "host_setup_ms": 0.0, "host_finish_ms": 0.0}
    e0.record()
    for _ in range(steps):
        comm.saca(d_shard, n)       # blocks until this rank's library stream has drained
        launches += _lib.last_stats()["kernel_launches"]
        cs = comm.stats()
        lib_ms += cs["total_ms"]
        for k_ in host:
            host[k_] += cs[k_] / steps
    e1.record()
    barrier()
    dev_ms = allred(e0.elapsed_time(e1) / steps, dist.ReduceOp.MAX)
    st = comm.stats()
    # radix-pass roofline: one extra step with per-launch events
    L.sab200_set_profiling(1)
    comm.saca(d_shard, n)
    ls = _lib.last_stats()
    L.sab200_set_profiling(0)
    achieved = (ls["radix_pass_bytes"] / 1e9) / (ls["radix_pass_ms"] / 1e3) if ls["radix_pass_ms"] > 0 else 0.0
    achieved = -allred(-achieved, dist.ReduceOp.MAX)
    pass_share = allred(ls["radix_pass_ms"] / ls["total_ms"] if ls["total_ms"] else 0.0, dist.ReduceOp.MAX)
    # end to end: pinned host shard in, pinned host slice of the suffix array out
    slice_len = st["slice_len"]
    _, h_out = pinned(slice_len + 1024, torch.int32)
    h_out = h_out.view(np.uint32)
    comm.saca(h_shard, n, out=h_out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        sl, off = comm.saca(h_shard, n, out=h_out)
    barrier()
    e2e_ms = allred((time.perf_counter() - t0) * 1e3 / steps, dist.ReduceOp.MAX)
    es = comm.stats()
    e2e_parts = {"h2d_ms": round(es["phase_ms"][14], 2), "stream_ms": round(es["total_ms"], 2), "d2h_ms": round(es["phase_ms"][15], 2),
                 "wall_ms": round(es["wall_ms"], 2)}
    if sampler is not None:
        sampler.end()
    # verification, outside the timed region: slices and shards to rank 0, GPU verifier (+ CPU oracle)
    sa_full = gather_to_rank0(dist, gloo, rank, world, sl, n + 1, off, np.uint32)
    text_full = gather_to_rank0(dist, gloo, rank, world, shard[:hi - lo], n, lo, np.uint8)
    ver = None
    if rank == 0:
        sa_full[0] = n
        ver = verify_host(L, _lib, text_full, sa_full, n, with_oracle=oracle_verify)
    a2a = allred(st["all_to_all_bytes"], dist.ReduceOp.SUM)
    tot_launches = allred(launches, dist.ReduceOp.SUM)
    max_slice = allred(slice_len, dist.ReduceOp.MAX)
    phases = {nm: round(st["phase_ms"][i], 2) for i, nm in enumerate(sdist.PHASES) if st["phase_ms"][i] > 0}
    rec = {"text_bytes": n, "ms_per_step": round(dev_ms, 3), "value": round(n / 1e6 / (dev_ms / 1e3), 2),
           "e2e_ms_per_step": round(e2e_ms, 3), "e2e_value": round(n / 1e6 / (e2e_ms / 1e3), 2), "e2e_parts_rank0": e2e_parts,
           "rounds": st["rounds"], "active": st["active"], "lazy_isa": bool(st["lazy_isa"]),
           "rank_layout": "block-cyclic" if st["rank_layout"] else "block", "collectives_per_step": st["collectives"],
           "all_to_all_bytes_per_step": int(a2a), "largest_slice": int(max_slice), "phase_ms_rank0": phases,
           "lib_stream_ms_rank0": round(lib_ms / steps, 3), "host_ms_rank0": {k_: round(v_, 3) for k_, v_ in host.items()},
           "radix_pass_gbs_slowest_rank": round(achieved, 1),
           "radix_pass_share_max": round(pass_share, 3), "gpu_launches": int(tot_launches), "verification": ver,
           "verified": bool(ver and ver["verified"])}
    return rec, (text_full, sa_full)


def run_distributed(args, L, _lib, torch, dist, rank, local_rank, world):
    """N > 1: ONE text sharded over the N GPUs (strong scaling: the total work is fixed as N grows).  Distributed
    sample sort + prefix doubling inside libsab200 (csrc/sab_dist.cuh); collectives = NCCL, created from a unique
    id this script broadcasts (suffix_array_b200.dist.Comm)."""
    from suffix_array_b200 import dist as sdist
    dev = torch.device("cuda", local_rank)
    gloo = dist.new_group(backend="gloo")
    comm = sdist.Comm("nccl", device=dev)
    desc, n, _ = WORKLOADS[args.workload]
    if args.n_mib:
        n = args.n_mib << 20
    sampler = ClockSampler(local_rank)
    if rank == 0:  # one nvidia-smi poller per box, started before the warm-up (see ClockSampler)
        sampler.start()
    main_rec, (text_full, sa_full) = dist_case(L, _lib, torch, dist, gloo, comm, rank, local_rank, world, args.workload, n,
                                               args.steps, args.warmup, sampler if rank == 0 else None,
                                               oracle_verify=(args.workload == "c2" and not args.n_mib and not args.no_oracle_verify))
    if rank == 0:
        sampler.join(timeout=2)
    outputs = None
    if rank == 0 and args.dump_outputs:  # the suffix array assembled from the slices of the last host-buffer step
        outputs = {"suffix_array": sa_full[dump_positions(n + 1, DUMP_SA_ENTRIES)]}
    c4 = None
    if args.workload != "c4" and not args.no_c4 and not args.n_mib:
        c4, _ = dist_case(L, _lib, torch, dist, gloo, comm, rank, local_rank, world, "c4", C4_BYTES, 2, 1, None, False)
        n1 = load_profile("r02_c4_1gpu.json") or {}
        n1_ms = n1.get("ms_per_step")
        if n1_ms:
            c4["single_gpu_ms"] = n1_ms
            c4["single_gpu_source"] = "profiles/r02_c4_1gpu.json (bench.py --workload c4 at N=1, same build)"
            c4["speedup_vs_single_gpu"] = round(n1_ms / c4["ms_per_step"], 2)
        c4["workload"] = WORKLOADS["c4"][0]
    # batched search sharded over N replicas: one process (rank 0) drives all GPUs; the others release theirs first
    comm.close()
    L.sab200_shutdown()
    torch.cuda.empty_cache()
    dist.barrier()
    search = None
    if rank == 0 and not args.no_search and args.workload == "c2":
        search = bench_search(L, _lib, torch, dev, text_full, sa_full, n, world, args.patterns, outputs)
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    dist.barrier()
    peak, peak_src = hbm_peak()
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": main_rec["value"], "unit": "MB/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_rec["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": dict(config_of(args.workload, n, args.n_mib),
                           per_gpu="one text block-sharded over %d GPUs: sample sort of the packed keys, then prefix "
                                   "doubling; NCCL all-to-all (inside libsab200) for keys, rank requests/answers and rank updates" % world,
                           l2="inputs larger than L2 (no flush needed)", rounds=main_rec["rounds"], active=main_rec["active"],
                           lazy_isa=main_rec["lazy_isa"], rank_layout=main_rec["rank_layout"],
                           collectives_per_step=main_rec["collectives_per_step"], phase_ms_rank0=main_rec["phase_ms_rank0"],
                           lib_stream_ms_rank0=main_rec["lib_stream_ms_rank0"], host_ms_rank0=main_rec["host_ms_rank0"],
                           largest_slice=main_rec["largest_slice"],
                           all_to_all_bytes_per_step=main_rec["all_to_all_bytes_per_step"]),
            "roofline": {"bound": "hbm", "kernel": "onesweep_kernel (LSD radix pass, slowest rank)",
                         "achieved": main_rec["radix_pass_gbs_slowest_rank"], "peak": peak, "unit": "GB/s",
                         "frac": round(main_rec["radix_pass_gbs_slowest_rank"] / peak, 4), "traffic": None, "peak_source": peak_src,
                         "share_of_step": main_rec["radix_pass_share_max"]},
            "e2e": {"value": main_rec["e2e_value"], "unit": "MB/s", "ms_per_step": main_rec["e2e_ms_per_step"],
                    "h2d_bytes_per_step": n + world * sdist.HALO, "d2h_bytes_per_step": 4 * n, "parts_rank0": main_rec["e2e_parts_rank0"],
                    "api": "sab200_saca_sharded (pinned host shard in, pinned host SA slice out, one PCIe link per rank)"},
            "cpu_baseline": None, "gpu_launches": main_rec["gpu_launches"], "verification": main_rec["verification"],
            "verified": main_rec["verified"], "c4": c4, "search": search, "clocks": sampler.summary()}))


if __name__ == "__main__":
    main()
