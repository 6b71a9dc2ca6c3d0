"""sab200::bwt / sab200::inverse_bwt of the C++ host mirror (include/sab200_suffix_array.hpp): compiles on CPU, runs
its round trips on the GPU."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "suffix_array_b200")


def _compile(out_dir):
    from suffix_array_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    exe = os.path.join(str(out_dir), "test_bwt_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_bwt_mirror.cpp"), "-L" + LIBDIR, "-lsab200", "-o", exe])
    return exe


def test_cpp_bwt_mirror_compiles(tmp_path):
    assert os.path.exists(_compile(tmp_path))


@pytest.mark.gpu
def test_cpp_bwt_mirror_runs(gpu_lib, tmp_path):
    exe = _compile(tmp_path)
    env = dict(os.environ, LD_LIBRARY_PATH=LIBDIR + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    out = subprocess.run([exe], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "all checks passed" in out.stdout, out.stdout + out.stderr
