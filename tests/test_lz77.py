"""LZ77 factorization and its decoder (sab200_lz77 / sab200_lz77_decode, include/sab200.h).

The factorization is compared bit for bit with the definition applied to a suffix array (tests/lz77_checker.c), its
lengths with a brute-force greedy parse on small texts, and every factor is property-checked (tiling, literal bytes,
matching copies with earlier sources, maximal lengths).  The decoder is checked on round trips, on non-greedy valid
parses, and on every rule it must refuse.  The emulator tests run the CUDA sources on the CPU, with chunks of 8
positions so that small texts cross many chunks and blocks of the parse; the gpu-marked ones run libsab200.so."""
import ctypes as C

import numpy as np
import pytest

from suffix_array_b200 import SuffixArray, gen, lz77, lz77_decode
from tests import lz77_checker
from tests import parity_cases as pc
from tests.test_bwt import golden_texts, random_texts


def check_lz77(oracle, s, sa=None, props=True):
    """lz77(s) against the definition over the oracle's (or the given) suffix array, properties, and the round trip"""
    s = np.ascontiguousarray(s, dtype=np.uint8)
    pos, ln = lz77(s)
    epos, eln = lz77_checker.lz77(s, oracle.saca(s) if sa is None else sa)
    assert pos.dtype == np.uint32 and ln.dtype == np.uint32
    assert np.array_equal(ln, eln) and np.array_equal(pos, epos), "factors differ from the definition (n=%d)" % s.size
    if props:
        assert lz77_checker.verify(s, pos, ln) == 0, "not a greedy parse (n=%d)" % s.size
    if s.size <= 2000:
        bpos, bln = lz77_checker.lz77_brute(s)
        assert np.array_equal(ln, bln) and np.array_equal(pos[ln == 0], bpos[bln == 0])
    assert np.array_equal(lz77_decode(pos, ln, s.size), s), "round trip failed (n=%d)" % s.size
    return pos, ln


def check_examples():
    for s, exp in ((b"banana", [(98, 0), (97, 0), (110, 0), (1, 3)]), (b"aaaa", [(97, 0), (0, 3)]), (b"", [])):
        pos, ln = lz77(s)
        assert list(zip(pos.tolist(), ln.tolist())) == exp, s
        assert lz77_decode(pos, ln, len(s)).tobytes() == s


def texts():
    a = [np.full(n, 97, dtype=np.uint8) for n in (2, 63, 64, 65, 4097, 5000)]
    return a + pc.adversarial_texts() + random_texts(23, 14)


def random_parse(rng, s):
    """a valid, mostly non-greedy parse of s: literals and copies of random earlier occurrences"""
    pos, ln, b = [], [], 0
    while b < s.size:
        if b == 0 or rng.random() < 0.3:
            pos.append(int(s[b]))
            ln.append(0)
            b += 1
            continue
        p = int(rng.integers(0, b))
        l = 0
        while b + l < s.size and s[p + l] == s[b + l] and l < int(rng.integers(1, 64)):
            l += 1
        if l == 0:
            pos.append(int(s[b]))
            ln.append(0)
            b += 1
        else:
            pos.append(p)
            ln.append(l)
            b += l
    return np.array(pos, dtype=np.uint32), np.array(ln, dtype=np.uint32)


def check_decoder_valid():
    rng = np.random.default_rng(5)
    for s in [gen.dna_like(3000), np.full(2500, 97, dtype=np.uint8), gen.repetitive(4000, block=300, mut_rate=1e-2)]:
        lit = s.astype(np.uint32)
        assert np.array_equal(lz77_decode(lit, np.zeros(s.size, dtype=np.uint32), s.size), s)  # all literals
        for _ in range(3):
            pos, ln = random_parse(rng, s)
            assert np.array_equal(lz77_decode(pos, ln, s.size), s)
            assert np.array_equal(lz77_checker.decode(pos, ln, s.size), s)
    # a copy that overlaps itself: "abababab" = a, b, (0, 6)
    assert lz77_decode([97, 98, 0], [0, 0, 6], 8).tobytes() == b"abababab"


BAD_PARSES = [  # (pos, len, n, the rule sab200_last_error names)
    ([97, 0], [0, 3], 5, "sum to 4"),                  # lengths sum short of n
    ([97, 0], [0, 3], 3, "sum to 4"),                  # ... and beyond it
    ([97, 300], [0, 0], 2, "pos > 255"),               # a literal above 255
    ([97, 1], [0, 3], 4, "source at or after"),        # a copy from its own start
    ([97, 5], [0, 3], 4, "source at or after"),        # a copy from the future
    ([97, 98, 99], [0, 0, 0], 2, "z > n"),
    ([], [], 3, "sum to 0"),
]


def check_decoder_invalid(L):
    for pos, ln, n, why in BAD_PARSES:
        with pytest.raises(ValueError, match=why):
            lz77_decode(pos, ln, n)
        p, l = np.array(pos, dtype=np.uint32), np.array(ln, dtype=np.uint32)
        out = np.full(max(n, 1), 0xA5, dtype=np.uint8)
        rc = L.sab200_lz77_decode(p.ctypes.data if p.size else None, l.ctypes.data if l.size else None, p.size, n, out.ctypes.data)
        assert rc == -1 and why.encode() in L.sab200_last_error()
        assert (out == 0xA5).all(), "a refused parse wrote to the output"
    out = np.zeros(1, dtype=np.uint8)
    assert L.sab200_lz77_decode(None, None, 0, (1 << 32), out.ctypes.data) == -1
    assert b"SAB200_MAX_LENGTH" in L.sab200_last_error()


def check_capacity(L):
    s = np.frombuffer(b"abracadabra abracadabra", dtype=np.uint8)
    epos, eln = lz77(s)
    z = C.c_uint64()
    pos = np.full(s.size, 7, dtype=np.uint32)
    ln = np.full(s.size, 7, dtype=np.uint32)
    assert L.sab200_lz77(s.ctypes.data, s.size, pos.ctypes.data, ln.ctypes.data, epos.size - 1, C.byref(z)) == -1
    assert z.value == epos.size and b"room for" in L.sab200_last_error()
    assert (pos == 7).all() and (ln == 7).all()
    assert L.sab200_lz77(s.ctypes.data, s.size, None, None, 0, C.byref(z)) == -1 and z.value == epos.size
    assert L.sab200_lz77(s.ctypes.data, s.size, pos.ctypes.data, ln.ctypes.data, epos.size, C.byref(z)) == 0
    assert z.value == epos.size and np.array_equal(pos[:z.value], epos) and np.array_equal(ln[:z.value], eln)


# ---------------------------------------------------------------- emulator (CPU)
def test_emu_lz77_examples(emu_backend):
    check_examples()


def test_emu_lz77_against_checkers(emu_backend, oracle, golden):
    for s in golden_texts(golden) + texts():
        check_lz77(oracle, s)


def test_emu_lz77_many_chunks_and_blocks(emu_backend, oracle):
    # with 8-position chunks: thousands of chunks, hundreds of blocks of 64, a top walk of thousands of steps
    check_lz77(oracle, gen.dna_like(150000), props=False)
    check_lz77(oracle, gen.repetitive(60000, block=700, mut_rate=1e-3))
    check_lz77(oracle, np.tile(np.frombuffer(b"abcab", dtype=np.uint8), 9000))
    # a common prefix of 70 000 bytes: eight rounds of the parallel comparison of the LCP step
    check_lz77(oracle, np.full(70001, 97, dtype=np.uint8), props=False)


def test_emu_lz77_stats_stay_readable(emu_backend):
    from suffix_array_b200 import last_stats
    lz77(gen.dna_like(5000))
    assert last_stats()["n"] == 5000


def test_emu_lz77_decode_valid(emu_backend):
    check_decoder_valid()


def test_emu_lz77_decode_invalid(emu_backend):
    check_decoder_invalid(emu_backend)


def test_emu_lz77_capacity(emu_backend):
    check_capacity(emu_backend)


def test_emu_lz77_device_forms(emu_lib, oracle):
    """the *_device entry points (the emulator's device memory is host memory)"""
    s = gen.dna_like(20000)
    epos, eln = lz77_checker.lz77(s, oracle.saca(s))
    pos = np.empty(s.size, dtype=np.uint32)
    ln = np.empty(s.size, dtype=np.uint32)
    z = C.c_uint64()
    assert emu_lib.sab200_lz77_device(s.ctypes.data, s.size, pos.ctypes.data, ln.ctypes.data, s.size, C.byref(z), 0) == 0
    assert np.array_equal(pos[:z.value], epos) and np.array_equal(ln[:z.value], eln)
    back = np.empty(s.size, dtype=np.uint8)
    assert emu_lib.sab200_lz77_decode_device(pos.ctypes.data, ln.ctypes.data, z.value, s.size, back.ctypes.data, 0) == 0
    assert np.array_equal(back, s)
    pos[int(np.argmax(ln[:z.value] > 0))] = 0xFFFFFFF0  # a copy whose source lies after its start
    back[:] = 0xA5
    assert emu_lib.sab200_lz77_decode_device(pos.ctypes.data, ln.ctypes.data, z.value, s.size, back.ctypes.data, 0) == -1
    assert b"source at or after" in emu_lib.sab200_last_error()
    assert (back == 0xA5).all()


def test_emu_prod_lz77_production_chunk(oracle, monkeypatch):
    """the emulator build with the production chunk of 2048 positions: many chunks, one block"""
    import os
    import subprocess
    from suffix_array_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(["make", "-C", os.path.join(root, "suffix_array_b200", "csrc"), "emu-prod"], stdout=subprocess.DEVNULL)
    monkeypatch.setattr(_lib, "_lib", _lib._bind(C.CDLL(os.path.join(root, "tests", "emu", "libsab200_emu_prod.so"))))
    check_lz77(oracle, gen.repetitive(40000, block=900, mut_rate=1e-3))
    check_lz77(oracle, np.full(9000, 97, dtype=np.uint8))


# ---------------------------------------------------------------- GPU (libsab200.so)
@pytest.mark.gpu
def test_lz77_examples(gpu_lib):
    check_examples()


@pytest.mark.gpu
def test_lz77_against_checkers(gpu_lib, oracle, golden):
    for s in golden_texts(golden) + texts():
        check_lz77(oracle, s)
    check_lz77(oracle, gen.dna_like(150000), props=False)
    check_lz77(oracle, gen.repetitive(60000, block=700, mut_rate=1e-3))
    check_lz77(oracle, gen.dna_like(5 << 20), props=False)  # thousands of chunks of 2048, two blocks of 2^22


@pytest.mark.gpu
def test_lz77_decode(gpu_lib):
    check_decoder_valid()
    check_decoder_invalid(gpu_lib)
    check_capacity(gpu_lib)


def _check_large(L, s):
    """against the definition over sab200_saca's own suffix array, once sab200_check accepts it, and the round trip"""
    sa = SuffixArray(s).sa
    assert L.sab200_check(s.ctypes.data, s.size, sa.ctypes.data, sa.size) == 1
    pos, ln = lz77(s)
    epos, eln = lz77_checker.lz77(s, sa)
    assert np.array_equal(ln, eln) and np.array_equal(pos, epos)
    assert np.array_equal(lz77_decode(pos, ln, s.size), s)


@pytest.mark.gpu
def test_lz77_dna_64mib(gpu_lib):
    _check_large(gpu_lib, gen.dna_like(64 << 20))


@pytest.mark.gpu
def test_lz77_repetitive_256mib(gpu_lib):
    _check_large(gpu_lib, gen.repetitive(256 << 20))


@pytest.mark.gpu
def test_lz77_all_a_64mib(gpu_lib):
    _check_large(gpu_lib, np.full(64 << 20, 97, dtype=np.uint8))


@pytest.mark.gpu
def test_lz77_pageable_pinned_and_device_buffers(gpu_lib, oracle):
    import torch
    s = gen.dna_like((5 << 20) + 3)
    epos, eln = lz77_checker.lz77(s, oracle.saca(s))
    z = C.c_uint64()
    for pinned in (False, True):
        def buf(n, dt):
            return torch.empty(n, dtype=dt, pin_memory=pinned).numpy()
        src, back = buf(s.size, torch.uint8), buf(s.size, torch.uint8)
        pos, ln = buf(s.size, torch.int32).view(np.uint32), buf(s.size, torch.int32).view(np.uint32)
        src[:] = s
        assert gpu_lib.sab200_lz77(src.ctypes.data, s.size, pos.ctypes.data, ln.ctypes.data, s.size, C.byref(z)) == 0
        assert np.array_equal(pos[:z.value], epos) and np.array_equal(ln[:z.value], eln), pinned
        assert gpu_lib.sab200_lz77_decode(pos.ctypes.data, ln.ctypes.data, z.value, s.size, back.ctypes.data) == 0
        assert np.array_equal(back, s), pinned
    d_s = torch.from_numpy(s).cuda()
    d_pos = torch.empty(s.size, dtype=torch.int32, device="cuda")
    d_len = torch.empty(s.size, dtype=torch.int32, device="cuda")
    d_back = torch.empty(s.size, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    assert gpu_lib.sab200_lz77_device(d_s.data_ptr(), s.size, d_pos.data_ptr(), d_len.data_ptr(), s.size, C.byref(z), 0) == 0
    zz = z.value
    assert np.array_equal(d_pos[:zz].cpu().numpy().view(np.uint32), epos) and np.array_equal(d_len[:zz].cpu().numpy().view(np.uint32), eln)
    assert gpu_lib.sab200_lz77_decode_device(d_pos.data_ptr(), d_len.data_ptr(), zz, s.size, d_back.data_ptr(), 0) == 0
    assert np.array_equal(d_back.cpu().numpy(), s)
    d_pos[int(np.argmax(eln > 0))] = -16  # 0xFFFFFFF0: a copy whose source lies after its start
    d_back.fill_(0xA5)
    torch.cuda.synchronize()
    assert gpu_lib.sab200_lz77_decode_device(d_pos.data_ptr(), d_len.data_ptr(), zz, s.size, d_back.data_ptr(), 0) == -1
    assert b"source at or after" in gpu_lib.sab200_last_error()
    assert (d_back.cpu().numpy() == 0xA5).all()
