"""Timing of the LZ77 factorization and its decoder (sab200_lz77*, sab200_lz77_decode*) on the gen.py texts at user
sizes, next to sab200_saca on the same text.  One JSON line per text.

    python tools/lz77_bench.py [--texts dna:1024,rep:256,a:64] [--reps 3] [--no-check]

Times are host clocks around calls that synchronise before they return (median of --reps after one warm-up call of
the same shape).  The device forms take device buffers (no PCIe); the host forms take pageable numpy buffers, as a
caller's plain allocation would be.  The phase breakdown of the device form comes from one more call under
torch.profiler, its kernels grouped by name (construction / ISA+LCP / LPF / parse / compaction / copy).  Every output
is checked outside the timed region: the factors against tests/lz77_checker.c over the library's own suffix array
(after sab200_check accepts it), and the decoder by the round trip.  The card's name and power limit are read in the
same run: a time means nothing without them."""
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
from tests import lz77_checker  # noqa: E402

TEXTS = {
    "dna": gen.dna_like,                                   # DNA-like, the 1 GiB flagship text
    "rep": gen.repetitive,                                 # long repeats with sparse mutations (long factors)
    "a": lambda n: np.full(n, 97, dtype=np.uint8),         # one symbol: a decreasing suffix array, z = 2
}

# kernel name prefixes of each phase after the construction; every other kernel is the construction's
PHASES = (("isa_lcp", ("lcp_isa_kernel", "lz_plcp")),
          ("lpf", ("lcp_block_min_kernel", "lz_lpf_kernel")),
          ("parse", ("lz_exit", "lz_walk")),
          ("compaction", ("lz_compact_kernel",)))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as e:  # the name still comes from torch below
        return None, "unknown (%s)" % e


def timed(f, reps):
    f()  # warm-up of the same shape: arena, scan status arrays, bounce buffers
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def phases(f):
    """device time per phase (ms) of one call of f, from the CUDA kernels and copies torch.profiler records"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        f()
    out = {k: 0.0 for k, _ in PHASES}
    out["construction"] = out["copy"] = 0.0
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        ms = ev.device_time / 1e3 if hasattr(ev, "device_time") else ev.cuda_time / 1e3
        name = ev.name
        if "memcpy" in name.lower() or "memset" in name.lower():
            out["copy"] += ms
            continue
        for k, prefixes in PHASES:
            if name.startswith(prefixes):
                out[k] += ms
                break
        else:
            out["construction"] += ms
    return {k + "_ms": round(v, 3) for k, v in out.items()}


def run_text(L, name, mib, reps, check):
    import torch
    n = mib << 20
    s = TEXTS[name](n)
    d_s = torch.from_numpy(s).cuda()
    d_pos = torch.empty(n, dtype=torch.int32, device="cuda")
    d_len = torch.empty(n, dtype=torch.int32, device="cuda")
    d_back = torch.empty(n, dtype=torch.uint8, device="cuda")
    d_sa = torch.empty(n + 1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    pos = np.empty(n, dtype=np.uint32)
    ln = np.empty(n, dtype=np.uint32)
    back = np.empty(n, dtype=np.uint8)
    sa = np.empty(n + 1, dtype=np.uint32)
    z = C.c_uint64()
    r = {"text": name, "n": n}

    def ok(rc, what):
        _lib.check(rc, what)

    r["saca_host_ms"] = timed(lambda: ok(L.sab200_saca(s.ctypes.data, n, sa.ctypes.data, 1), "sab200_saca"), reps)
    r["saca_device_ms"] = timed(lambda: ok(L.sab200_saca_device(d_s.data_ptr(), n, d_sa.data_ptr(), 0), "sab200_saca_device"), reps)
    r["lz_host_ms"] = timed(lambda: ok(L.sab200_lz77(s.ctypes.data, n, pos.ctypes.data, ln.ctypes.data, n, C.byref(z)), "sab200_lz77"), reps)
    zh = int(z.value)
    r["z"] = zh
    if check:  # untimed: the definition over the library's own suffix array
        assert L.sab200_check(s.ctypes.data, n, sa.ctypes.data, n + 1) == 1, "sab200_saca's suffix array is refused"
        epos, eln = lz77_checker.lz77(s, sa)
        assert np.array_equal(pos[:zh], epos) and np.array_equal(ln[:zh], eln), "factors differ from the definition"
        del epos, eln
    dev = lambda: ok(L.sab200_lz77_device(d_s.data_ptr(), n, d_pos.data_ptr(), d_len.data_ptr(), n, C.byref(z), 0), "sab200_lz77_device")
    r["lz_device_ms"] = timed(dev, reps)
    assert int(z.value) == zh
    assert np.array_equal(d_pos[:zh].cpu().numpy().view(np.uint32), pos[:zh]), "device form differs from the host form"
    assert np.array_equal(d_len[:zh].cpu().numpy().view(np.uint32), ln[:zh]), "device form differs from the host form"
    r["dec_host_ms"] = timed(lambda: ok(L.sab200_lz77_decode(pos.ctypes.data, ln.ctypes.data, zh, n, back.ctypes.data), "sab200_lz77_decode"), reps)
    assert np.array_equal(back, s), "round trip failed"
    r["dec_device_ms"] = timed(lambda: ok(L.sab200_lz77_decode_device(d_pos.data_ptr(), d_len.data_ptr(), zh, n, d_back.data_ptr(), 0),
                                          "sab200_lz77_decode_device"), reps)
    assert np.array_equal(d_back.cpu().numpy(), s), "device round trip failed"
    for k in ("saca_host", "saca_device", "lz_host", "lz_device", "dec_host", "dec_device"):
        r[k + "_GBps"] = round(n / (r[k + "_ms"] * 1e6), 3)  # text bytes per second
    try:
        r["lz_device_phases"] = phases(dev)
    except Exception as e:  # the timings above stand without it
        r["lz_device_phases"] = "not measured (%s)" % e
    del d_s, d_pos, d_len, d_back, d_sa
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--texts", default="dna:1024,rep:256,a:64", help="name:MiB,... with names from %s" % sorted(TEXTS))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-check", action="store_true", help="skip the CPU checker of the factors")
    args = ap.parse_args()
    import torch
    L = _lib.require_gpu()
    name, limit = card()
    gpu = {"gpu": name or torch.cuda.get_device_name(0), "power_limit": limit}
    for item in args.texts.split(","):
        t, mib = item.split(":")
        r = run_text(L, t, int(mib), args.reps, not args.no_check)
        r.update(gpu)
        print(json.dumps(r), flush=True)
    L.sab200_shutdown()


if __name__ == "__main__":
    main()
