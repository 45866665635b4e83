"""CPU checks of BatchNormAct2d and the encoder's module swap: layer counts, torchvision's state_dict, the unchanged torch
path on CPU, and the C ABI's argument errors for the BatchNorm entry points."""
import copy
import ctypes
import os

import pytest
import torch
import torch.nn as nn

from monocular_depth_estimation_b200 import _lib
from monocular_depth_estimation_b200.model import BatchNormAct2d, Encoder


def _tv():
    import torchvision.models as tvm
    return tvm.mobilenet_v3_large()


def test_swap_counts():
    acts = [m.act for m in Encoder().modules() if isinstance(m, BatchNormAct2d)]
    assert len(acts) == 46
    assert (acts.count("hardswish"), acts.count("relu"), acts.count(None)) == (20, 11, 15)
    from torchvision.ops.misc import Conv2dNormActivation
    cna = [m for m in Encoder().original_model.features.modules() if isinstance(m, Conv2dNormActivation)]
    assert len(cna) == 46
    assert all(isinstance(m[1], BatchNormAct2d) and (len(m) == 2 or type(m[2]) is nn.Identity) for m in cna)


def test_state_dict_is_torchvisions():
    ours, ref = Encoder().original_model.state_dict(), _tv().state_dict()
    assert list(ours) == list(ref)
    for k in ref:
        assert ours[k].shape == ref[k].shape and ours[k].dtype == ref[k].dtype, k


def test_strict_load_of_a_torchvision_state_dict():
    ref = _tv()
    with torch.no_grad():
        for t in ref.state_dict().values():
            if t.dtype.is_floating_point:
                t.copy_(torch.randn_like(t))
    enc = Encoder()
    enc.original_model.load_state_dict(ref.state_dict(), strict=True)
    for k, t in enc.original_model.state_dict().items():
        assert torch.equal(t, ref.state_dict()[k]), k


def test_swap_keeps_the_tensors():
    import torchvision.models as tvm
    from monocular_depth_estimation_b200.model import fuse_batchnorm_act
    feats = tvm.mobilenet_v3_large().features
    before = {n: t for n, t in feats.state_dict(keep_vars=True).items()}
    fuse_batchnorm_act(feats)
    after = feats.state_dict(keep_vars=True)
    assert all(after[n] is t for n, t in before.items())


def test_cpu_training_step_is_bit_identical_to_torchvision():
    torch.manual_seed(0)
    ref = _tv().features.train()
    enc = Encoder().train()
    enc.original_model.features.load_state_dict(ref.state_dict())
    ours = enc.original_model.features
    ref_c = copy.deepcopy(ref)
    x = torch.randn(2, 3, 64, 96)
    y_r, y_o = ref(x), ours(x)
    assert torch.equal(y_r, y_o)
    g = torch.randn_like(y_r)
    y_r.backward(g)
    y_o.backward(g)
    for (n, p_r), (_, p_o) in zip(ref.named_parameters(), ours.named_parameters()):
        assert torch.equal(p_r.grad, p_o.grad), n
    for (n, b_r), (_, b_o) in zip(ref.named_buffers(), ours.named_buffers()):
        assert torch.equal(b_r, b_o), n
    assert not torch.equal(ref_c[1].block[0][1].running_mean, ref[1].block[0][1].running_mean)  # the step did train


def test_eval_forward_matches_torchvision():
    ref = _tv().features.eval()
    enc = Encoder().eval()
    enc.original_model.features.load_state_dict(ref.state_dict())
    x = torch.randn(1, 3, 64, 64)
    with torch.no_grad():
        assert torch.equal(ref(x), enc.original_model.features(x))


def test_rejects_unknown_activation():
    with pytest.raises(ValueError):
        BatchNormAct2d(16, act="gelu")


@pytest.fixture
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("extension not built")
    return _lib.lib()


def _fwd(lib, x=16, T=64, C=64, act=0, ws=256, ws_bytes=1 << 20, tickets=512):
    p = ctypes.c_void_p(4096)
    return lib.crf_bn_fwd(ctypes.c_void_p(x), p, p, p, p, p, p, p, p, T, C, 1e-3, 0.01, act,
                          None if ws is None else ctypes.c_void_p(ws), ws_bytes,
                          None if tickets is None else ctypes.c_void_p(tickets), 0, None)


def _bwd(lib, x=16, T=64, C=64, act=0):
    p = ctypes.c_void_p(4096)
    return lib.crf_bn_bwd(ctypes.c_void_p(x), p, p, p, p, p, p, p, p, T, C, act, ctypes.c_void_p(256), 1 << 20,
                          ctypes.c_void_p(512), 0, None)


@pytest.mark.parametrize("kw,msg", [({"C": 12}, b"multiple of 8"), ({"C": 0}, b"multiple of 8"),
                                    ({"T": 1}, b"more than one value"), ({"act": 3}, b"unknown activation"),
                                    ({"x": 18}, b"16-byte aligned"), ({"ws": 264}, b"16-byte aligned"),
                                    ({"tickets": None}, b"tickets"), ({"x": 0}, b"null pointer")])
def test_bn_argument_errors(lib, kw, msg):
    assert _fwd(lib, **kw) != 0
    assert msg in lib.crf_last_error()
    if set(kw) <= {"C", "T", "act", "x"} and kw.get("x") != 0:
        assert _bwd(lib, **kw) != 0
        assert msg in lib.crf_last_error()
