"""Timing of the matching statistics (sab200_matching_statistics_batch*) on the 1 GiB DNA-like text of
BASELINE.json configs[1].  One JSON line per query set, then one for the index extension.

    python tools/ms_bench.py [--mib 1024] [--reps 3]

Query sets: 64 MiB of random DNA (matches of about log4 n bytes), 64 MiB of excerpts of the text with 1 % byte
substitutions, and one 16 MiB excerpt (every position matches to the end of the query: the longest runs, where a
quadratic path would show first).  Times are host clocks around calls that synchronise before they return (median of
--reps after one warm-up call of the same shape).  The host form takes pageable numpy buffers; the device form takes
device buffers (no PCIe).  For scale, search_all (device form) on as many 32-byte patterns as the set has positions.
The extension's build time is the first call on a fresh index minus a second call of the same one-byte query.
Outputs are checked on a sample of positions outside the timed region with the library's own search_all and contains.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from suffix_array_b200 import SuffixArray, _lib, gen  # noqa: E402
from tests.test_matching_statistics import check_sample, excerpt, pack  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception:
        return None, "unknown"


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def query_sets(s, rng):
    dna = np.frombuffer(b"ACGT", np.uint8)
    rand = [rng.choice(dna, 64 << 20).tobytes()]
    exc = []
    while sum(map(len, exc)) < 64 << 20:
        exc.append(excerpt(rng, s, int(rng.integers(1000, 100000)), subs=0.01))
    return [("random_dna_64mib", rand), ("excerpts_1pct_64mib", exc), ("excerpt_16mib", [excerpt(rng, s, 16 << 20)])]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    L = _lib.require_gpu()
    name, limit = card()
    gpu = {"gpu": name or torch.cuda.get_device_name(0), "power_limit": limit}
    s = gen.dna_like(args.mib << 20)
    n = s.size
    sa = SuffixArray(s)
    ix = sa._get_index()
    t0 = time.perf_counter()
    sa.matching_statistics(b"A")
    t1 = time.perf_counter()
    sa.matching_statistics(b"A")
    t2 = time.perf_counter()
    extra = 0
    c = n + 1
    while c > 256:
        c = -(-c // 256)
        extra += c
    ext = {"what": "index_extension", "n": n, "build_s": round((t1 - t0) - (t2 - t1), 4),
           "bytes": 8 * (n + 2) + 4 * (extra + 1), **gpu}
    rng = np.random.default_rng(2026)
    d_text = torch.from_numpy(s).cuda()
    for label, queries in query_sets(s, rng):
        qs, offs = pack(queries)
        m = qs.size
        host_s = timed(lambda: sa.matching_statistics_batch(qs, offs), args.reps)
        d_qs = torch.from_numpy(np.concatenate([qs, np.zeros(64, np.uint8)])).cuda()
        d_offs = torch.from_numpy(offs.view(np.uint8)).cuda()
        d_out = torch.empty(3 * m * 4, dtype=torch.uint8, device="cuda")
        p = d_out.data_ptr()
        torch.cuda.synchronize()

        def dev():
            _lib.check(L.sab200_matching_statistics_batch_device(ix, d_qs.data_ptr(), d_offs.data_ptr(), offs.size - 1,
                                                                  p, p + 4 * m, p + 8 * m), "ms device")
        dev_s = timed(dev, args.reps)
        del d_out, d_qs
        # search_all on m 32-byte windows of the text, device form
        starts = torch.randint(0, n - 32, (m,), device="cuda")
        pats = d_text[(starts[:, None] + torch.arange(32, device="cuda")).reshape(-1)]
        pats = torch.cat([pats, torch.zeros(64, dtype=torch.uint8, device="cuda")])
        del starts
        p_offs = (torch.arange(m + 1, device="cuda", dtype=torch.int64) * 32)
        lo_hi = torch.empty(2 * m, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

        def sall():
            _lib.check(L.sab200_search_all_batch_device(ix, pats.data_ptr(), p_offs.data_ptr(), m, lo_hi.data_ptr(),
                                                        lo_hi.data_ptr() + 4 * m), "search_all device")
        sall_s = timed(sall, args.reps)
        del pats, p_offs, lo_hi
        torch.cuda.empty_cache()
        got = sa.matching_statistics_batch(qs, offs)
        sample = np.sort(rng.choice(m - 4096, 100000, replace=False)) if m > 200000 else np.arange(m)
        if label == "excerpt_16mib":  # each match runs to the query's end: sample few long ones, many short ones
            assert np.array_equal(got[0], np.arange(m, 0, -1, dtype=np.uint32))
            sample = np.concatenate([np.sort(rng.choice(m - 4096, 16, replace=False)), np.arange(m - 4096, m)])
        check_sample(sa, qs, offs, got, sample)
        print(json.dumps({"what": label, "query_bytes": int(m), "queries": int(offs.size - 1),
                          "mean_len": round(float(got[0].mean()), 2), "max_len": int(got[0].max()),
                          "host_s": round(host_s, 4), "host_gbytes_per_s": round(m / host_s / 1e9, 4),
                          "device_s": round(dev_s, 4), "device_gbytes_per_s": round(m / dev_s / 1e9, 4),
                          "search_all_32b_same_count_s": round(sall_s, 4), "sample_checked": int(sample.size), **gpu}),
              flush=True)
    print(json.dumps(ext), flush=True)


if __name__ == "__main__":
    main()
