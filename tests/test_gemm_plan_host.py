"""Which GEMM kernel launch_gemm runs for a problem, compiled on the host (no GPU) from the header the launcher includes
(csrc/crf_sched.h, `plan_gemm`): the CTA-pair kernel, the persistent kernel or the tiled gemm_kernel<BN>, for every
projection of a block at the widths the library accepts, in both precision modes, and at each threshold of the rule.
"""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "monocular_depth_estimation_b200", "csrc")

SHIM = r"""
#include "crf_sched.h"
extern "C" int plan(int M, int N, int K, int a_major, int epi, int split3, int* bn) {
  const crf::GemmPlan p = crf::plan_gemm(M, N, K, a_major, epi, split3);
  *bn = p.bn;
  return p.kernel;
}
extern "C" int tile_n(int N) { return crf::gemm_tile_n(N); }
"""

STORE_F32, STORE_BF16, BIAS_RES_F32, BIAS_GELU, MUL_DGELU, SPLITK_F32 = range(6)   # CRF_EPI_* (include/crf_sm100.h)
T = 2400   # tokens of a 30 x 40 map at batch 2; the rule does not depend on M


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("gemm_plan")
    src, so = d / "shim.cpp", d / "libgemmplan.so"
    src.write_text(SHIM)
    subprocess.run(["g++", "-O1", "-shared", "-fPIC", "-x", "c++", "-I", CSRC, str(src), "-o", str(so)], check=True)
    lib = ctypes.CDLL(str(so))
    lib.plan.argtypes = [ctypes.c_int] * 6 + [ctypes.POINTER(ctypes.c_int)]
    lib.tile_n.argtypes = [ctypes.c_int]
    return lib


def kernel(shim, M, N, K, a_major, epi, split3=0):
    """'P' (CTA pair), 'S' (persistent) or 'T<BN>' (tiled)"""
    bn = ctypes.c_int(-1)
    k = shim.plan(M, N, K, a_major, epi, split3, ctypes.byref(bn))
    assert k in (0, 1, 2), k
    if k == 2:
        return f"T{bn.value}"
    assert bn.value == 0, (k, bn.value)
    return "PS"[k]


def block_gemms(C, precise):
    """(name, M, N, K, a_major, epilogue) of every GEMM of one block's forward and backward at width C (crf_api.cu; the
    fp32 precision mode, crf_precise.cu, runs the same shapes with fp32 epilogues and split3)."""
    def bf16(epi):
        return STORE_F32 if precise else epi
    return [("qk", T, 2 * C, C, 0, bf16(STORE_BF16)), ("proj", T, C, C, 0, BIAS_RES_F32),
            ("fc1", T, 4 * C, C, 0, bf16(BIAS_GELU)), ("fc2", T, C, 4 * C, 0, BIAS_RES_F32),
            ("d_fc2", T, 4 * C, C, 0, bf16(MUL_DGELU)), ("d_fc1", T, C, 4 * C, 0, STORE_F32),
            ("d_proj", T, C, C, 0, bf16(STORE_BF16)), ("d_qk", T, C, 2 * C, 0, STORE_F32),
            ("w_fc2", C, 4 * C, T, 1, SPLITK_F32), ("w_fc1", 4 * C, C, T, 1, SPLITK_F32),
            ("w_proj", C, C, T, 1, SPLITK_F32), ("w_qk", 2 * C, C, T, 1, SPLITK_F32)]


# Pair: A K-major, N % 256 == 0, N >= 512, K >= 512, no split3, not split-K.  Persistent: A K-major, N % 128 == 0, no
# split3, not split-K.  Otherwise tiled, BN = 256 / 128 / 64 (the widest dividing N), at most 128 with K-major A.
BF16_MODE = {  # qk   proj  fc1  fc2   d_fc2 d_fc1 d_proj d_qk    w_fc2 w_fc1 w_proj w_qk
    64:   "S     T64   S    T64   S     T64   T64    T64     T256  T64   T64    T64",
    128:  "S     S     S    S     S     S     S      S       T256  T128  T128   T128",
    192:  "S     T64   S    T64   S     T64   T64    T64     T256  T64   T64    T64",
    256:  "S     S     S    S     S     S     S      S       T256  T256  T256   T256",
    320:  "S     T64   S    T64   S     T64   T64    T64     T256  T64   T64    T64",
    512:  "P     P     P    P     P     P     P      P       T256  T256  T256   T256",
    576:  "S     T64   P    T64   P     T64   T64    T64     T256  T64   T64    T64",
    960:  "S     T64   P    T64   P     T64   T64    T64     T256  T64   T64    T64",
    1024: "P     P     P    P     P     P     P      P       T256  T256  T256   T256",
}
FP32_MODE = {  # split3: always the tiled kernel
    64:   "T128  T64   T128 T64   T128  T64   T64    T64     T256  T64   T64    T64",
    128:  "T128  T128  T128 T128  T128  T128  T128   T128    T256  T128  T128   T128",
    192:  "T128  T64   T128 T64   T128  T64   T64    T64     T256  T64   T64    T64",
    256:  "T128  T128  T128 T128  T128  T128  T128   T128    T256  T256  T256   T256",
    320:  "T128  T64   T128 T64   T128  T64   T64    T64     T256  T64   T64    T64",
    512:  "T128  T128  T128 T128  T128  T128  T128   T128    T256  T256  T256   T256",
    576:  "T128  T64   T128 T64   T128  T64   T64    T64     T256  T64   T64    T64",
    960:  "T128  T64   T128 T64   T128  T64   T64    T64     T256  T64   T64    T64",
    1024: "T128  T128  T128 T128  T128  T128  T128   T128    T256  T256  T256   T256",
}


@pytest.mark.parametrize("precise", [0, 1], ids=["bf16", "fp32"])
@pytest.mark.parametrize("C", sorted(BF16_MODE))
def test_block_gemms(shim, C, precise):
    want = (FP32_MODE if precise else BF16_MODE)[C].split()
    got = [kernel(shim, M, N, K, am, epi, precise) for _, M, N, K, am, epi in block_gemms(C, precise)]
    names = [g[0] for g in block_gemms(C, precise)]
    assert dict(zip(names, got)) == dict(zip(names, want))


@pytest.mark.parametrize("M,N,K,a_major,epi,split3,want", [
    # pair kernel: K = 448 / 512, N = 256 / 512
    (T, 512, 448, 0, STORE_BF16, 0, "S"), (T, 512, 512, 0, STORE_BF16, 0, "P"),
    (T, 256, 512, 0, STORE_BF16, 0, "S"), (T, 512, 512, 0, MUL_DGELU, 0, "P"),
    (T, 768, 512, 0, BIAS_GELU, 0, "P"), (T, 640, 512, 0, STORE_F32, 0, "S"),   # N % 256
    (T, 1024, 1024, 0, STORE_F32, 1, "T128"),                                  # split3 never runs on the pair kernel
    (T, 1024, 1024, 0, SPLITK_F32, 0, "T128"),                                 # nor split-K, capped with K-major A
    (T, 512, 512, 1, STORE_F32, 0, "T256"),                                    # nor MN-major A
    # persistent kernel: N % 128
    (T, 384, 64, 0, STORE_BF16, 0, "S"), (T, 448, 64, 0, STORE_BF16, 0, "T64"), (T, 128, 4096, 0, BIAS_RES_F32, 0, "S"),
    (T, 64, 64, 0, STORE_BF16, 0, "T64"), (T, 384, 64, 0, STORE_F32, 1, "T128"), (T, 384, 64, 0, SPLITK_F32, 0, "T128"),
    (T, 384, 64, 1, STORE_F32, 0, "T128"),
    # tiled width: N % 256 with (K-major A) and without (MN-major A) the cap at 128
    (T, 768, 64, 0, SPLITK_F32, 0, "T128"), (768, 768, T, 1, SPLITK_F32, 0, "T256"),
    (T, 768, 64, 0, STORE_F32, 1, "T128"), (768, 768, T, 1, SPLITK_F32, 1, "T256"),
    (T, 640, 64, 0, SPLITK_F32, 0, "T128"), (640, 640, T, 1, SPLITK_F32, 0, "T128"),
    (T, 704, 64, 0, SPLITK_F32, 0, "T64"), (704, 704, T, 1, SPLITK_F32, 0, "T64"),
])
def test_boundaries(shim, M, N, K, a_major, epi, split3, want):
    assert kernel(shim, M, N, K, a_major, epi, split3) == want


def test_splitk_workspace_width_is_uncapped(shim):
    """gemm_splitk_workspace_bytes sizes its splits with the widest tile that divides N, also where plan_gemm caps the
    launch at 128 (split-K with K-major A, which no caller in the library makes)."""
    assert [shim.tile_n(n) for n in (64, 128, 192, 256, 384, 512, 640, 768, 4096)] == [64, 128, 64, 256, 128, 256, 128,
                                                                                       256, 256]
    assert kernel(shim, T, 512, 512, 0, SPLITK_F32) == "T128"
