"""CPU checks of the depthwise convolutions: the tap map of csrc/crf_dwconv.cuh (compiled with g++) against brute force,
the encoder's module swap (15 DepthwiseConv2d modules, torchvision's state_dict, the unchanged torch path on CPU) and the
C ABI's argument errors for the depthwise entry points."""
import copy
import ctypes
import os
import subprocess

import pytest
import torch
import torch.nn as nn

from monocular_depth_estimation_b200 import _lib
from monocular_depth_estimation_b200.model import DepthwiseConv2d, Encoder

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "monocular_depth_estimation_b200", "csrc")

SHIM = r"""
#define __host__
#define __device__
#include "crf_dwconv.cuh"
using namespace crf;
extern "C" int out_size(int n, int k, int s) { return dw_out_size(n, k, s); }
extern "C" int src(int o, int i, int k, int s, int n) { return dw_src(o, i, k, s, n); }
extern "C" int dst(int h, int i, int k, int s, int n_out) { return dw_dst(h, i, k, s, n_out); }
template <int K, int S> void run_maps(int* m) {
  using R = DwRun<K, S, 4>;
  m[0] = R::kIn; m[1] = R::kLo; m[2] = R::kOut;
  for (int q = 0; q < 4; ++q) {
    for (int c = 0; c < 16; ++c) m[3 + q * 16 + c] = c < R::kIn ? R::fwd_tap(q, c) : -2;
    for (int d = 0; d < 16; ++d) m[67 + q * 16 + d] = d < R::kOut ? R::dgrad_tap(q, R::kLo + d) : -2;
  }
}
// m: kIn, kLo, kOut, fwd_tap[4][16], dgrad_tap[4][16] (-2 past the table)
extern "C" void run(int k, int s, int* m) {
  if (k == 3 && s == 1) run_maps<3, 1>(m);
  if (k == 3 && s == 2) run_maps<3, 2>(m);
  if (k == 5 && s == 1) run_maps<5, 1>(m);
  if (k == 5 && s == 2) run_maps<5, 2>(m);
}
"""

GEOMS = [(k, s) for k in (3, 5) for s in (1, 2)]


@pytest.fixture(scope="module")
def taps(tmp_path_factory):
    d = tmp_path_factory.mktemp("dwconv")
    src, so = d / "shim.cpp", d / "libtaps.so"
    src.write_text(SHIM)
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-I", CSRC, str(src), "-o", str(so)],
                   check=True)
    return ctypes.CDLL(str(so))


def _brute(n, k, s):
    """Every (input, tap, output) triple of one axis: output o, tap i reads input o s - k // 2 + i inside [0, n)."""
    n_out = (n + 2 * (k // 2) - k) // s + 1
    return n_out, {(o * s - k // 2 + i, i, o) for o in range(n_out) for i in range(k) if 0 <= o * s - k // 2 + i < n}


@pytest.mark.parametrize("k,s", GEOMS)
def test_axis_maps_match_brute_force(taps, k, s):
    for n in range(1, 21):
        n_out, want = _brute(n, k, s)
        assert taps.out_size(n, k, s) == n_out == (n - 1) // s + 1
        fwd = {(taps.src(o, i, k, s, n), i, o) for o in range(n_out) for i in range(k) if taps.src(o, i, k, s, n) >= 0}
        bwd = [(h, i, taps.dst(h, i, k, s, n_out)) for h in range(n) for i in range(k) if taps.dst(h, i, k, s, n_out) >= 0]
        assert fwd == want, (n, k, s)
        assert sorted(bwd) == sorted(want) and len(set(bwd)) == len(bwd), (n, k, s)   # each triple exactly once
        # borders: a padding tap maps to nothing
        assert all(taps.src(o, i, k, s, n) == -1 for o in range(n_out) for i in range(k)
                   if not 0 <= o * s - k // 2 + i < n)


def _run_tables(taps, k, s):
    m = (ctypes.c_int * 131)()
    taps.run(k, s, m)
    kin, klo, kout = m[0], m[1], m[2]
    fwd = [[m[3 + q * 16 + c] for c in range(kin)] for q in range(4)]
    dgr = [[m[67 + q * 16 + d] for d in range(kout)] for q in range(4)]
    return kin, klo, kout, fwd, dgr


@pytest.mark.parametrize("k,s", GEOMS)
def test_run_tables_cover_every_tap_exactly_once(taps, k, s):
    """The kernels' runs of 4 pixels, with every H, W <= 20: summed over runs, the forward / weight-gradient table and
    the input-gradient table each produce every (input, tap, output) triple of an axis exactly once, with the loads past
    the axis' ends (zeros) and the pixels past it (not stored) dropped."""
    kin, klo, kout, fwd, dgr = _run_tables(taps, k, s)
    p = k // 2
    for n in range(1, 21):
        n_out, want = _brute(n, k, s)
        got_f, got_d = [], []
        for o0 in range(0, n_out, 4):              # forward and weight gradient: runs of outputs
            for q in range(4):
                for c in range(kin):
                    j, h = fwd[q][c], o0 * s - p + c
                    if j >= 0 and o0 + q < n_out and 0 <= h < n:
                        got_f.append((h, j, o0 + q))
        for h0 in range(0, n, 4):                  # input gradient: runs of inputs
            for q in range(4):
                for d in range(kout):
                    j, o = dgr[q][d], h0 // s + klo + d
                    if j >= 0 and h0 + q < n and 0 <= o < n_out:
                        got_d.append((h0 + q, j, o))
        assert sorted(got_f) == sorted(want) and len(set(got_f)) == len(got_f), (n, k, s)
        assert sorted(got_d) == sorted(want) and len(set(got_d)) == len(got_d), (n, k, s)
    # the taps an output (input) takes are in ascending (descending) order along the run's loads: a fixed sum order
    for q in range(4):
        f = [j for j in fwd[q] if j >= 0]
        d = [j for j in dgr[q] if j >= 0]
        assert f == sorted(f) and d == sorted(d, reverse=True)


def _tv():
    import torchvision.models as tvm
    return tvm.mobilenet_v3_large()


def test_swap_counts_and_shared_weights():
    import torchvision.models as tvm
    from monocular_depth_estimation_b200.model import fuse_depthwise
    feats = tvm.mobilenet_v3_large().features
    before = feats.state_dict(keep_vars=True)
    fuse_depthwise(feats)
    dw = [m for m in feats.modules() if isinstance(m, DepthwiseConv2d)]
    assert len(dw) == 15
    assert sorted({(m.kernel_size[0], m.stride[0]) for m in dw}) == [(3, 1), (3, 2), (5, 1), (5, 2)]
    after = feats.state_dict(keep_vars=True)
    assert list(after) == list(before) and all(after[n] is t for n, t in before.items())
    assert len([m for m in Encoder().modules() if isinstance(m, DepthwiseConv2d)]) == 15


def test_state_dict_is_torchvisions():
    ours, ref = Encoder().original_model.state_dict(), _tv().state_dict()
    assert list(ours) == list(ref)
    for k in ref:
        assert ours[k].shape == ref[k].shape and ours[k].dtype == ref[k].dtype, k


def test_cpu_training_step_is_bit_identical_to_torchvision():
    torch.manual_seed(0)
    ref = _tv().features.train()
    enc = Encoder().train()
    enc.original_model.features.load_state_dict(ref.state_dict())
    ours = enc.original_model.features
    x = torch.randn(2, 3, 64, 96)
    y_r, y_o = ref(x), ours(x)
    assert torch.equal(y_r, y_o)
    g = torch.randn_like(y_r)
    y_r.backward(g)
    y_o.backward(g)
    for (n, p_r), (_, p_o) in zip(ref.named_parameters(), ours.named_parameters()):
        assert torch.equal(p_r.grad, p_o.grad), n


def test_rejects_grouped_conv_that_is_not_depthwise():
    with pytest.raises(ValueError):
        DepthwiseConv2d(16, 32, 3, groups=16)
    assert isinstance(DepthwiseConv2d.from_conv(nn.Conv2d(8, 8, 5, 2, 2, groups=8, bias=False)), nn.Conv2d)


@pytest.fixture
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("extension not built")
    return _lib.lib()


def _fwd(lib, x=16, C=64, k=3, s=1, H=8, W=8, B=2):
    p = ctypes.c_void_p(4096)
    return lib.crf_dwconv_fwd(None if x is None else ctypes.c_void_p(x), p, p, B, H, W, C, k, s, 0, None)


def _bwd(lib, x=16, C=64, k=3, s=1, H=8, W=8, B=2, ws=256, tickets=512, dx=4096, dw=4096):
    p = ctypes.c_void_p(4096)
    v = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    return lib.crf_dwconv_bwd(v(x), p, p, v(dx), v(dw), B, H, W, C, k, s, v(ws), 1 << 20, v(tickets), 0, None)


@pytest.mark.parametrize("kw,msg", [({"C": 12}, b"multiple of 8"), ({"C": 0}, b"multiple of 8"),
                                    ({"k": 7}, b"kernel size 7"), ({"k": 1}, b"kernel size 1"),
                                    ({"s": 3}, b"stride 3"), ({"H": 0}, b"must be positive"),
                                    ({"B": 0}, b"must be positive"), ({"x": 18}, b"16-byte aligned"),
                                    ({"x": None}, b"null pointer")])
def test_dwconv_argument_errors(lib, kw, msg):
    assert _fwd(lib, **kw) != 0
    assert msg in lib.crf_last_error()
    assert _bwd(lib, **kw) != 0
    assert msg in lib.crf_last_error()


@pytest.mark.parametrize("kw,msg", [({"tickets": None}, b"tickets"), ({"ws": None}, b"workspace"),
                                    ({"ws": 264}, b"16-byte aligned"), ({"dx": 4104}, b"16-byte aligned"),
                                    ({"dx": None, "dw": None}, b"neither dx nor dweight")])
def test_dwconv_bwd_argument_errors(lib, kw, msg):
    assert _bwd(lib, **kw) != 0
    assert msg in lib.crf_last_error()
