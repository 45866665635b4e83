"""Work-decomposition arithmetic of the persistent kernels, compiled on the host (no GPU) from the header the kernels
and launchers include (csrc/crf_sched.h): `balanced_tile_rows` (fused MLP forward, fused d.LN' kernel) gives rows per
tile that are a multiple of 8, at most 128, cover the input, and never need more rounds of the grid than 128-row tiles do.
"""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "monocular_depth_estimation_b200", "csrc")

SHIM = r"""
#include "crf_sched.h"
extern "C" int tile_rows(int T, int sms) { return crf::balanced_tile_rows(T, sms); }
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("sched")
    src, so = d / "shim.cpp", d / "libsched.so"
    src.write_text(SHIM)
    subprocess.run(["g++", "-O1", "-shared", "-fPIC", "-x", "c++", "-I", CSRC, str(src), "-o", str(so)], check=True)
    lib = ctypes.CDLL(str(so))
    lib.tile_rows.argtypes = [ctypes.c_int, ctypes.c_int]
    return lib


def test_balanced_tile_rows(shim):
    sms = 148
    for T in list(range(1, 700)) + [2400, 9600, 38400, 153600, 16 * 60 * 80, 16 * 240 * 320, 123457]:
        tm = shim.tile_rows(T, sms)
        assert 8 <= tm <= 128 and tm % 8 == 0, (T, tm)
        tiles = -(-T // tm)
        tiles128 = -(-T // 128)
        rounds, rounds128 = -(-tiles // sms), -(-tiles128 // sms)
        assert rounds <= rounds128, (T, tm)                      # never more rounds than 128-row tiles
        assert rounds * tm <= rounds128 * 128, (T, tm)           # and never more row-time
    assert shim.tile_rows(38400, sms) == 88 and shim.tile_rows(153600, sms) == 120    # the two decoder scales that use it
    assert shim.tile_rows(128, sms) == 128 and shim.tile_rows(1000, sms) == 128
