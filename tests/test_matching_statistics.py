"""Matching statistics of batched queries (sab200_matching_statistics_batch, include/sab200.h).

All three outputs (len, lo, hi) are compared with the CPU checkers of tests/ms_checker.c: the definition by brute
force on small inputs, a per-position bisection over the oracle's suffix array on larger ones.  The large GPU cases
check a sample with the library's own search_all / contains.  The emulator tests run the CUDA sources on the CPU; the
gpu-marked ones run libsab200.so on the device."""
import numpy as np
import pytest

from suffix_array_b200 import SuffixArray, gen
from tests import ms_checker

CHUNK = 1024  # SAB_MS_CHUNK (csrc/sab_ms.cuh): positions per warp


def pack(queries):
    qs = [bytes(q) for q in queries]
    offs = np.zeros(len(qs) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(q) for q in qs])
    return np.frombuffer(b"".join(qs), dtype=np.uint8), offs


def check(oracle, s, queries, sa_obj=None, naive=None):
    """matching_statistics_batch against the bisection checker (and the brute-force one on small inputs)"""
    s = np.ascontiguousarray(s, dtype=np.uint8)
    qs, offs = pack(queries)
    sa_obj = sa_obj if sa_obj is not None else SuffixArray(s)
    got = sa_obj.matching_statistics_batch(qs, offs)
    exp = ms_checker.bisect(s, oracle.saca(s), qs, offs)
    if (s.size * qs.size <= 4 << 20) if naive is None else naive:
        for e, x in zip(exp, ms_checker.naive(s, qs, offs)):
            assert np.array_equal(e, x), "the checkers differ"
    for name, g, e in zip(("len", "lo", "hi"), got, exp):
        if not np.array_equal(g, e):
            bad = np.nonzero(g != e)[0][:5]
            raise AssertionError("%s differs at %s: %s, expected %s (n=%d)" % (name, bad, g[bad], e[bad], s.size))
    return got


def excerpt(rng, s, m, subs=0.0):
    """m bytes of s from a random start, with a fraction `subs` of its bytes replaced"""
    i = int(rng.integers(0, s.size - m + 1))
    q = s[i:i + m].copy()
    k = int(m * subs)
    if k:
        q[rng.integers(0, m, k)] = rng.integers(0, 256, k, dtype=np.uint8)
    return q.tobytes()


def random_texts(seed, count):
    """n in [0, 6000) with n = 0 and n = 1 among them, sigma in {1, 2, 4, 256}, periodic texts with one flipped byte"""
    rng = np.random.default_rng(seed)
    out = [np.zeros(0, dtype=np.uint8), np.array([7], dtype=np.uint8)]
    for trial in range(count):
        n = int(rng.integers(2, 6000))
        s = rng.integers(0, int(rng.choice([1, 2, 4, 256])), n, dtype=np.uint8)
        if trial % 2 == 0 and n > 100:
            per = int(rng.integers(1, 300))
            s = np.tile(s[:per], n // per + 1)[:n].copy()
            s[int(rng.integers(0, n))] ^= 1
        out.append(s)
    return out


def mixed_queries(rng, s):
    """excerpts with sparse substitutions, a query inside the text, bytes absent from the text, empty queries, short
    queries back to back (a match must stop at its query's end)"""
    n = s.size
    qs = [b"", b"\xff\xfe\xfd", b""]
    if n:
        qs.append(excerpt(rng, s, min(n, 700)))
        qs.append(excerpt(rng, s, min(n, 500), subs=0.01))
        qs.append(excerpt(rng, s, min(n, 300), subs=0.05))
        qs += [excerpt(rng, s, int(rng.integers(1, min(n, 12) + 1))) for _ in range(40)]
    qs.append(rng.integers(0, 256, 200, dtype=np.uint8).tobytes())
    qs.append(b"")
    return qs


def chunk_queries(rng, s):
    """query lengths at C-1, C, C+1 and around multiples of C, so that chunk starts fall inside long matches"""
    return [excerpt(rng, s, m, subs=0.002 if k % 2 else 0.0)
            for k, m in enumerate((CHUNK - 1, CHUNK, CHUNK + 1, 2 * CHUNK - 1, 2 * CHUNK + 1, 3 * CHUNK, 3 * CHUNK + 7))]


def golden_cases(golden):
    rng = np.random.default_rng(8)
    for v in golden["vectors"]:
        s = np.frombuffer(bytes.fromhex(v["text_hex"]), dtype=np.uint8)
        yield s, mixed_queries(rng, s)


def check_basic(oracle, golden):
    for s, qs in golden_cases(golden):
        check(oracle, s, qs)
    rng = np.random.default_rng(21)
    for s in random_texts(5, 10):
        check(oracle, s, mixed_queries(rng, s))


def check_chunk_boundaries(oracle):
    rng = np.random.default_rng(22)
    for s in (gen.dna_like(12000), gen.repetitive(9000, block=500, mut_rate=1e-3), np.tile(np.frombuffer(b"ab", np.uint8), 5000)):
        got = check(oracle, s, chunk_queries(rng, s), naive=False)
        assert got[0].max() > 2 * CHUNK  # matches that run across chunk starts


def check_index_variants(oracle, monkeypatch):
    """buckets, and no prefix directory: the from-scratch search then bisects the whole array"""
    rng = np.random.default_rng(23)
    s = gen.dna_like(20000)
    qs = mixed_queries(rng, s) + chunk_queries(rng, s)[:3]
    check(oracle, s, qs, sa_obj=SuffixArray.new_with_buckets(s))
    monkeypatch.setenv("SAB_SEARCH_DIR", "0")
    sa = SuffixArray(s)
    assert _lib().sab200_index_directory(sa._get_index(), None, None) == 0
    check(oracle, s, qs, sa_obj=sa)
    sa = SuffixArray.new_with_buckets(s)
    check(oracle, s, qs, sa_obj=sa)


def check_wrong_array(oracle):
    """an index over a suffix array that is not the text's: ValueError, and the index still answers search_all"""
    rng = np.random.default_rng(24)
    s = rng.integers(0, 4, 3000, dtype=np.uint8)
    good = oracle.saca(s)
    oob = good.copy()
    oob[1000] = s.size + 5
    perm = good.copy()
    perm[[100, 101]] = perm[[101, 100]]
    pats = [excerpt(rng, s, 8) for _ in range(50)]
    for bad in (oob, perm):
        sa = SuffixArray.unchecked_from_parts(s, bad)
        before = sa.search_all_batch(pats)
        for _ in range(2):  # no extension is kept: the second call checks again
            with pytest.raises(ValueError, match="not the suffix array of its text"):
                sa.matching_statistics(s[:100].tobytes())
        after = sa.search_all_batch(pats)
        assert all(np.array_equal(a, b) for a, b in zip(before, after))


def check_arguments():
    s = gen.dna_like(5000)
    sa = SuffixArray(s)
    with pytest.raises(ValueError, match="offsets decrease"):
        sa.matching_statistics_batch(np.frombuffer(b"ACGTACGT", np.uint8), np.array([0, 5, 3, 8], dtype=np.uint64))
    L = _lib()
    assert L.sab200_matching_statistics_batch(sa._get_index(), None, None, 0, None, None, None) == 0
    ln, lo, hi = sa.matching_statistics(b"")
    assert ln.size == 0
    ln, lo, hi = sa.matching_statistics(b"\x00")  # a byte the text lacks
    assert (ln[0], lo[0], hi[0]) == (0, 0, s.size + 1)
    # offsets that do not start at 0: the outputs are indexed by the absolute offset
    qs = np.frombuffer(s[:300].tobytes(), np.uint8)
    offs = np.array([100, 150, 300], dtype=np.uint64)
    out = [np.zeros(300, dtype=np.uint32) for _ in range(3)]
    assert L.sab200_matching_statistics_batch(sa._get_index(), qs.ctypes.data, offs.ctypes.data, 2,
                                              *[o.ctypes.data for o in out]) == 0
    assert not out[0][:100].any() and list(out[0][100:150]) == list(range(50, 0, -1))


def _lib():
    from suffix_array_b200 import _lib as m
    return m.lib()


def check_device_form(oracle, s, queries, to_dev, from_dev):
    """sab200_matching_statistics_batch_device against the host form"""
    sa = SuffixArray(s)
    qs, offs = pack(queries)
    exp = sa.matching_statistics_batch(qs, offs)
    total = int(offs[-1])
    d_qs, d_offs = to_dev(np.concatenate([qs, np.zeros(64, np.uint8)])), to_dev(offs)
    outs = [to_dev(np.zeros(total, dtype=np.uint32)) for _ in range(3)]
    rc = _lib().sab200_matching_statistics_batch_device(sa._get_index(), d_qs[1], d_offs[1], offs.size - 1,
                                                        *[o[1] for o in outs])
    assert rc == 0, _lib().sab200_last_error()
    for o, e in zip(outs, exp):
        assert np.array_equal(from_dev(o), e)
    bad = to_dev(np.array([0, 5, 3], dtype=np.uint64))
    assert _lib().sab200_matching_statistics_batch_device(sa._get_index(), d_qs[1], bad[1], 2, *[o[1] for o in outs]) == -1


# ---------------------------------------------------------------- emulator (CPU)
def test_emu_ms_golden_and_random(emu_backend, oracle, golden):
    check_basic(oracle, golden)


def test_emu_ms_chunk_boundaries(emu_backend, oracle):
    check_chunk_boundaries(oracle)


def test_emu_ms_index_variants(emu_backend, oracle, monkeypatch):
    check_index_variants(oracle, monkeypatch)


def test_emu_ms_wrong_array(emu_backend, oracle):
    check_wrong_array(oracle)


def test_emu_ms_arguments(emu_backend):
    check_arguments()


def test_emu_ms_device_form(emu_backend, oracle):
    """the emulator's device memory is host memory"""
    rng = np.random.default_rng(25)
    s = gen.dna_like(8000)
    check_device_form(oracle, s, mixed_queries(rng, s), lambda a: (a, a.ctypes.data), lambda t: t[0])


# ---------------------------------------------------------------- GPU (libsab200.so)
@pytest.mark.gpu
def test_ms_against_checker(gpu_lib, oracle, golden, monkeypatch):
    check_basic(oracle, golden)
    check_chunk_boundaries(oracle)
    check_arguments()
    check_index_variants(oracle, monkeypatch)
    rng = np.random.default_rng(26)
    s = gen.dna_like(3 << 20)  # ~3000 chunks, long planted repeats
    check(oracle, s, [excerpt(rng, s, 1 << 20, subs=0.01), excerpt(rng, s, 200000), rng.choice(np.frombuffer(b"ACGT", np.uint8), 300000)])


@pytest.mark.gpu
def test_ms_wrong_array(gpu_lib, oracle):
    check_wrong_array(oracle)


def slices(qs, starts, lens):
    """the concatenation of qs[starts[k] : starts[k] + lens[k]] and its offsets"""
    starts, lens = starts.astype(np.int64), lens.astype(np.int64)
    offs = np.zeros(lens.size + 1, dtype=np.uint64)
    offs[1:] = np.cumsum(lens)
    idx = np.repeat(starts - offs[:-1].astype(np.int64), lens) + np.arange(int(offs[-1]), dtype=np.int64)
    return qs[idx], offs


def check_sample(sa, qs, offs, got, positions):
    """(lo, hi) equals search_all of the match, and the match extended by one byte does not occur"""
    ln, lo, hi = got
    qend = offs[np.searchsorted(offs, positions, side="right")]
    pl = ln[positions].astype(np.int64)
    flat, po = slices(qs, positions, pl)
    elo, ehi = sa.search_all_batch(flat, po)
    assert np.array_equal(lo[positions], elo) and np.array_equal(hi[positions], ehi)
    ext = positions + pl < qend.astype(np.int64)
    flat, po = slices(qs, positions[ext], pl[ext] + 1)
    assert not sa.contains_batch(flat, po).any()


@pytest.mark.gpu
def test_ms_dna_64mib(gpu_lib):
    s = gen.dna_like(64 << 20)
    sa = SuffixArray(s)
    rng = np.random.default_rng(27)
    qs = [rng.choice(np.frombuffer(b"ACGT", np.uint8), 8 << 20).tobytes()]
    while sum(map(len, qs)) < 16 << 20:
        qs.append(excerpt(rng, s, int(rng.integers(100, 20000)), subs=0.01))
    flat, offs = pack(qs)
    got = sa.matching_statistics_batch(flat, offs)
    assert np.median(got[0]) >= 8 and got[0].max() > 1000
    check_sample(sa, flat, offs, got, np.sort(rng.choice(flat.size, 1 << 20, replace=False)))


@pytest.mark.gpu
def test_ms_repetitive_256mib(gpu_lib):
    """a 4 MiB query taken from the text: every position matches to the end of the query"""
    s = gen.repetitive(256 << 20)
    sa = SuffixArray(s)
    rng = np.random.default_rng(28)
    q = excerpt(rng, s, 4 << 20)
    flat, offs = pack([q])
    got = sa.matching_statistics_batch(flat, offs)
    m = flat.size
    assert np.array_equal(got[0], np.arange(m, 0, -1, dtype=np.uint32))
    positions = np.concatenate([np.sort(rng.choice(m - 4096, 24, replace=False)), np.arange(m - 4096, m)])
    check_sample(sa, flat, offs, got, positions)


@pytest.mark.gpu
def test_ms_pageable_pinned_and_device(gpu_lib, oracle):
    import torch
    rng = np.random.default_rng(29)
    s = gen.dna_like((2 << 20) + 3)
    queries = [excerpt(rng, s, 300000, subs=0.01), rng.choice(np.frombuffer(b"ACGT", np.uint8), 200000).tobytes()] + mixed_queries(rng, s)
    qs, offs = pack(queries)
    exp = ms_checker.bisect(s, oracle.saca(s), qs, offs)
    sa = SuffixArray(s)
    L = _lib()
    for pinned in (False, True):
        def buf(a):
            b = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=pinned).numpy().view(a.dtype)
            b[:] = a
            return b
        q, o = buf(qs), buf(offs)
        outs = [buf(np.zeros(qs.size, dtype=np.uint32)) for _ in range(3)]
        assert L.sab200_matching_statistics_batch(sa._get_index(), q.ctypes.data, o.ctypes.data, o.size - 1,
                                                  *[x.ctypes.data for x in outs]) == 0
        for x, e in zip(outs, exp):
            assert np.array_equal(x, e), pinned

    def to_dev(a):
        t = torch.from_numpy(a.view(np.uint8)).cuda()
        torch.cuda.synchronize()
        return t, t.data_ptr(), a.dtype

    def from_dev(t):
        return t[0].cpu().numpy().view(t[2])
    check_device_form(oracle, s, queries, to_dev, from_dev)


@pytest.mark.gpu
def test_ms_multi_gpu_identical(gpu_lib):
    if gpu_lib.sab200_device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    rng = np.random.default_rng(30)
    s = gen.dna_like(16 << 20)
    queries = [excerpt(rng, s, int(rng.integers(1, 50000)), subs=0.01) for _ in range(200)] + [b""] * 3
    qs, offs = pack(queries)
    one = SuffixArray(s)
    exp = one.matching_statistics_batch(qs, offs)
    for ngpus in sorted({2, gpu_lib.sab200_device_count()}):
        many = SuffixArray(s, _sa=one.sa)
        many.use_gpus(ngpus)
        for g, e in zip(many.matching_statistics_batch(qs, offs), exp):
            assert np.array_equal(g, e), ngpus
