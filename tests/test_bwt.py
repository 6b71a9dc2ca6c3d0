"""Burrows-Wheeler transform and its inverse (sab200_bwt / sab200_inverse_bwt, include/sab200.h).

The forward transform is compared with the definition applied to the oracle's suffix array (tests/bwt_checker.c),
the inverse with the round trip and, on every small transform over {a, b}, with the sequential LF walk: the library
must accept exactly the pairs (U, p) the walk accepts.  The emulator tests run the CUDA sources on the CPU; the
gpu-marked ones run libsab200.so on the device."""
import ctypes as C
import itertools

import numpy as np
import pytest

from suffix_array_b200 import SuffixArray, bwt, gen, inverse_bwt
from tests import bwt_checker
from tests import parity_cases as pc


def check_bwt(oracle, s):
    """bwt(s) against the definition over the oracle's suffix array, and the round trip"""
    s = np.ascontiguousarray(s, dtype=np.uint8)
    u, p = bwt(s)
    eu, ep = bwt_checker.bwt(s, oracle.saca(s))
    assert u.dtype == np.uint8 and u.size == s.size
    assert p == ep and np.array_equal(u, eu), "transform differs from the definition (n=%d)" % s.size
    assert np.array_equal(inverse_bwt(u, p), s), "round trip failed (n=%d)" % s.size


def golden_texts(golden):
    return [np.frombuffer(bytes.fromhex(v["text_hex"]), dtype=np.uint8) for v in golden["vectors"]]


def random_texts(seed, count):
    """n in [0, 30000) with n = 0 and n = 1 among them, sigma in {1, 2, 4, 256}, periodic texts with one flipped byte"""
    rng = np.random.default_rng(seed)
    out = [np.zeros(0, dtype=np.uint8), np.array([7], dtype=np.uint8)]
    for trial in range(count):
        n = int(rng.integers(0, 30000))
        s = rng.integers(0, int(rng.choice([1, 2, 4, 256])), n, dtype=np.uint8)
        if trial % 2 == 0 and n > 100:
            per = int(rng.integers(1, 300))
            s = np.tile(s[:per], n // per + 1)[:n].copy()
            s[int(rng.integers(0, n))] ^= 1
        out.append(s)
    return out


def not_a_transform(u, p):
    """u with two different bytes swapped, such that the LF walk rejects it"""
    for j in range(11, u.size):
        if u[j] != u[10]:
            bad = u.copy()
            bad[[10, j]] = bad[[j, 10]]
            if bwt_checker.inverse_bwt(bad, p) is None:
                return bad
    raise AssertionError("no rejected swap found")


def check_definition(golden):
    u, p = bwt(b"banana")
    assert (u.tobytes(), p) == (b"annbaa", 4)
    assert inverse_bwt(b"annbaa", 4).tobytes() == b"banana"
    for v in golden["vectors"]:  # the definition over the golden suffix arrays
        s = np.frombuffer(bytes.fromhex(v["text_hex"]), dtype=np.uint8)
        sa = v["sa"]
        u, p = bwt(s)
        assert sa[p] == 0 and u.tolist() == [int(s[j - 1]) for j in sa if j > 0]


def check_validation():
    """Every (U, p) with U in {a, b}^n, 1 <= p <= n, n <= 6: accepted iff the LF walk accepts, with its text."""
    accepted = 0
    for n in range(1, 7):
        for bits in itertools.product(b"ab", repeat=n):
            u = bytes(bits)
            for p in range(1, n + 1):
                exp = bwt_checker.inverse_bwt(u, p)
                if exp is None:
                    with pytest.raises(ValueError, match="not the Burrows-Wheeler transform"):
                        inverse_bwt(u, p)
                else:
                    accepted += 1
                    assert inverse_bwt(u, p).tobytes() == exp.tobytes(), (u, p)
    assert accepted == sum(2 ** n for n in range(1, 7))  # one (U, p) per text


def check_bad_primary():
    for u, p in ((b"annbaa", 0), (b"annbaa", 7), (b"annbaa", 2 ** 40), (b"", 1)):
        with pytest.raises(ValueError, match="primary index"):
            inverse_bwt(u, p)
    assert inverse_bwt(b"", 0).size == 0
    assert bwt(b"")[1] == 0 and bwt(b"")[0].size == 0
    assert bwt(b"x")[0].tobytes() == b"x" and bwt(b"x")[1] == 1


# ---------------------------------------------------------------- emulator (CPU)
def test_emu_bwt_definition(emu_backend, golden):
    check_definition(golden)


def test_emu_bwt_against_checker(emu_backend, oracle, golden):
    for s in golden_texts(golden) + pc.adversarial_texts() + random_texts(17, 14):
        check_bwt(oracle, s)


def test_emu_bwt_many_tiles_and_samples(emu_backend, oracle):
    # > 30 onesweep tiles, > 36 scan tiles and hundreds of sample rows
    check_bwt(oracle, gen.dna_like(150000))
    check_bwt(oracle, gen.repetitive(60000, block=700, mut_rate=1e-3))


def test_emu_inverse_bwt_validation(emu_backend):
    check_validation()


def test_emu_inverse_bwt_bad_primary(emu_backend):
    check_bad_primary()


def test_emu_bwt_device_forms(emu_lib, oracle):
    """the *_device entry points (the emulator's device memory is host memory)"""
    s = gen.dna_like(20000)
    u = np.empty(s.size, dtype=np.uint8)
    p = C.c_uint64()
    assert emu_lib.sab200_bwt_device(s.ctypes.data, s.size, u.ctypes.data, C.byref(p), 0) == 0
    eu, ep = bwt_checker.bwt(s, oracle.saca(s))
    assert p.value == ep and np.array_equal(u, eu)
    back = np.empty(s.size, dtype=np.uint8)
    assert emu_lib.sab200_inverse_bwt_device(u.ctypes.data, u.size, p.value, back.ctypes.data, 0) == 0
    assert np.array_equal(back, s)
    bad = not_a_transform(u, p.value)
    assert emu_lib.sab200_inverse_bwt_device(bad.ctypes.data, bad.size, p.value, back.ctypes.data, 0) == -1
    assert b"not the Burrows-Wheeler transform" in emu_lib.sab200_last_error()


# ---------------------------------------------------------------- GPU (libsab200.so)
@pytest.mark.gpu
def test_bwt_definition(gpu_lib, golden):
    check_definition(golden)


@pytest.mark.gpu
def test_bwt_against_checker(gpu_lib, oracle, golden):
    for s in golden_texts(golden) + pc.adversarial_texts() + random_texts(17, 14):
        check_bwt(oracle, s)
    check_bwt(oracle, gen.dna_like(150000))
    check_bwt(oracle, gen.repetitive(60000, block=700, mut_rate=1e-3))
    check_bwt(oracle, gen.dna_like(3 << 20))  # ~12k sample rows: many look-back tiles and walks


@pytest.mark.gpu
def test_inverse_bwt_validation(gpu_lib):
    check_validation()
    check_bad_primary()


def _check_large(s):
    """forward against the gather from sab200_saca's own suffix array, and the round trip"""
    u, p = bwt(s)
    sa = SuffixArray(s).sa
    assert sa[p] == 0
    assert np.array_equal(u, s[np.delete(sa, p) - 1])
    assert np.array_equal(inverse_bwt(u, p), s)


@pytest.mark.gpu
def test_bwt_uniform_64mib(gpu_lib):
    _check_large(gen.uniform_bytes(64 << 20))


@pytest.mark.gpu
def test_bwt_repetitive_256mib(gpu_lib):
    _check_large(gen.repetitive(256 << 20))


@pytest.mark.gpu
def test_bwt_pageable_and_pinned_buffers(gpu_lib, oracle):
    import torch
    s = gen.dna_like((5 << 20) + 3)
    eu, ep = bwt_checker.bwt(s, oracle.saca(s))
    for pinned in (False, True):
        def buf(n):
            return torch.empty(n, dtype=torch.uint8, pin_memory=True).numpy() if pinned else np.empty(n, dtype=np.uint8)
        src, u, back = buf(s.size), buf(s.size), buf(s.size)
        src[:] = s
        p = C.c_uint64()
        assert gpu_lib.sab200_bwt(src.ctypes.data, s.size, u.ctypes.data, C.byref(p)) == 0
        assert p.value == ep and np.array_equal(u, eu), pinned
        assert gpu_lib.sab200_inverse_bwt(u.ctypes.data, u.size, p.value, back.ctypes.data) == 0
        assert np.array_equal(back, s), pinned


@pytest.mark.gpu
def test_bwt_device_forms(gpu_lib, oracle):
    import torch
    s = gen.dna_like((3 << 20) + 5)
    eu, ep = bwt_checker.bwt(s, oracle.saca(s))
    d_s = torch.from_numpy(s).cuda()
    d_u = torch.empty(s.size, dtype=torch.uint8, device="cuda")
    d_back = torch.empty(s.size, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    p = C.c_uint64()
    assert gpu_lib.sab200_bwt_device(d_s.data_ptr(), s.size, d_u.data_ptr(), C.byref(p), 0) == 0
    assert p.value == ep and np.array_equal(d_u.cpu().numpy(), eu)
    assert gpu_lib.sab200_inverse_bwt_device(d_u.data_ptr(), s.size, p.value, d_back.data_ptr(), 0) == 0
    assert np.array_equal(d_back.cpu().numpy(), s)
    d_bad = torch.from_numpy(not_a_transform(eu, ep)).cuda()
    torch.cuda.synchronize()
    assert gpu_lib.sab200_inverse_bwt_device(d_bad.data_ptr(), s.size, p.value, d_back.data_ptr(), 0) == -1
    assert b"not the Burrows-Wheeler transform" in gpu_lib.sab200_last_error()
