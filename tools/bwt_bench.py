"""Timing of the Burrows-Wheeler transform and its inverse (sab200_bwt*, sab200_inverse_bwt*) on the gen.py texts at
user sizes, next to sab200_saca end to end on the same text.  One JSON line per text.

    python tools/bwt_bench.py [--texts dna:1024,rep:256,uni:64] [--reps 3] [--no-cpu]

Times are host clocks around calls that synchronise before they return (median of --reps after one warm-up call of
the same shape).  The device forms take device buffers (no PCIe); the host forms take pageable numpy buffers, as a
caller's plain allocation would be.  Every output is checked against the library's own suffix array and by the round
trip, outside the timed region.  cpu_inverse_ms is the sequential LF walk of tests/bwt_checker.c on one core.  The
card's name and power limit are read in the same run: a time means nothing without them."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from suffix_array_b200 import _lib, gen  # noqa: E402
from tests import bwt_checker  # noqa: E402

TEXTS = {
    "dna": gen.dna_like,                 # DNA-like, the 1 GiB flagship text
    "rep": gen.repetitive,               # long repeats with sparse mutations (long LCPs)
    "uni": gen.uniform_bytes,            # uniform bytes, sigma = 256
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as e:  # the name still comes from torch below
        return None, "unknown (%s)" % e


def timed(f, reps):
    f()  # warm-up of the same shape: arena, look-back and scan status arrays, bounce buffers
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def run_text(L, name, mib, reps, cpu):
    import torch
    n = mib << 20
    s = TEXTS[name](n)
    d_s = torch.from_numpy(s).cuda()
    d_u = torch.empty(n, dtype=torch.uint8, device="cuda")
    d_back = torch.empty(n, dtype=torch.uint8, device="cuda")
    d_sa = torch.empty(n + 1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    u = np.empty(n, dtype=np.uint8)
    back = np.empty(n, dtype=np.uint8)
    sa = np.empty(n + 1, dtype=np.uint32)
    p = C.c_uint64()
    r = {"text": name, "n": n}

    def ok(rc, what):
        _lib.check(rc, what)

    r["saca_host_ms"] = timed(lambda: ok(L.sab200_saca(s.ctypes.data, n, sa.ctypes.data, 1), "sab200_saca"), reps)
    r["saca_device_ms"] = timed(lambda: ok(L.sab200_saca_device(d_s.data_ptr(), n, d_sa.data_ptr(), 0), "sab200_saca_device"), reps)
    r["fwd_host_ms"] = timed(lambda: ok(L.sab200_bwt(s.ctypes.data, n, u.ctypes.data, C.byref(p)), "sab200_bwt"), reps)
    # checks, untimed: the transform is the gather from the library's own suffix array, and it inverts to s
    pf = int(p.value)
    assert sa[pf] == 0 and np.array_equal(u, s[np.delete(sa, pf) - 1]), "forward transform differs from the gather"
    r["fwd_device_ms"] = timed(lambda: ok(L.sab200_bwt_device(d_s.data_ptr(), n, d_u.data_ptr(), C.byref(p), 0), "sab200_bwt_device"), reps)
    assert int(p.value) == pf and np.array_equal(d_u.cpu().numpy(), u), "device form differs from the host form"
    r["inv_host_ms"] = timed(lambda: ok(L.sab200_inverse_bwt(u.ctypes.data, n, pf, back.ctypes.data), "sab200_inverse_bwt"), reps)
    assert np.array_equal(back, s), "round trip failed"
    r["inv_device_ms"] = timed(lambda: ok(L.sab200_inverse_bwt_device(d_u.data_ptr(), n, pf, d_back.data_ptr(), 0),
                                          "sab200_inverse_bwt_device"), reps)
    assert np.array_equal(d_back.cpu().numpy(), s), "device round trip failed"
    for k in ("saca_host", "saca_device", "fwd_host", "fwd_device", "inv_host", "inv_device"):
        r[k + "_GBps"] = round(n / (r[k + "_ms"] * 1e6), 3)  # text bytes per second
    if cpu:
        t0 = time.perf_counter()
        text = bwt_checker.inverse_bwt(u, pf)
        r["cpu_inverse_ms"] = (time.perf_counter() - t0) * 1e3
        assert text is not None and np.array_equal(text, s)
    del d_s, d_u, d_back, d_sa
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--texts", default="dna:1024,rep:256,uni:64", help="name:MiB,... with names from %s" % sorted(TEXTS))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true", help="skip the single-core LF walk")
    args = ap.parse_args()
    import torch
    L = _lib.require_gpu()
    name, limit = card()
    gpu = {"gpu": name or torch.cuda.get_device_name(0), "power_limit": limit}
    for item in args.texts.split(","):
        t, mib = item.split(":")
        r = run_text(L, t, int(mib), args.reps, not args.no_cpu)
        r.update(gpu)
        print(json.dumps(r), flush=True)
    L.sab200_shutdown()


if __name__ == "__main__":
    main()
