"""BatchNormAct2d on the library's BatchNorm kernels (crf_bn_fwd / crf_bn_bwd) against torch's act(F.batch_norm) in
training mode: every BatchNorm shape of the encoder at batch 8, ragged shapes, large |mean| / std, repeatability,
CUDA-graph replay, the fallback cases and one whole-model training step."""
import json
import os

import pytest
import torch
import torch.nn as nn

from tests.helpers import fill_by_name, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF16_ULP = 2.0 ** -7     # bf16 spacing relative to the value (8 significant bits)


def _encoder_bn_shapes():
    """(C, H, W, act) of the encoder's 46 BatchNorm layers at the bench resolution (480 x 640)."""
    import torchvision.models as tvm
    from monocular_depth_estimation_b200.model import BatchNormAct2d, fuse_batchnorm_act
    m = fuse_batchnorm_act(tvm.mobilenet_v3_large().features)
    shapes = []
    hooks = [mod.register_forward_hook(lambda mod, inp, out: shapes.append((mod.num_features, inp[0].shape[2],
                                                                           inp[0].shape[3], mod.act)))
             for mod in m.modules() if isinstance(mod, BatchNormAct2d)]
    with torch.no_grad():
        m.eval()(torch.zeros(1, 3, 480, 640))
    for h in hooks:
        h.remove()
    return shapes


ENCODER_SHAPES = _encoder_bn_shapes()
RAGGED = [(1, 64, 7, 9, "relu"), (3, 40, 13, 11, "hardswish"), (2, 960, 1, 1, "hardswish"), (2, 16, 1, 1, None),
          (5, 72, 17, 3, None), (1, 24, 1, 2, "relu")]


def _stock(C, act, eps=1e-3, momentum=0.01):
    bn = nn.BatchNorm2d(C, eps=eps, momentum=momentum)
    return nn.Sequential(bn, {"relu": nn.ReLU(inplace=True), "hardswish": nn.Hardswish(inplace=True),
                              None: nn.Identity()}[act])


def _pair(C, act, seed=0):
    """(stock Sequential(BatchNorm2d, act), BatchNormAct2d) with equal, non-trivial parameters and running stats."""
    from monocular_depth_estimation_b200.model import BatchNormAct2d
    g = torch.Generator().manual_seed(seed)
    ref = _stock(C, act)
    with torch.no_grad():
        ref[0].weight.copy_(1 + 0.3 * torch.randn(C, generator=g))
        ref[0].bias.copy_(0.3 * torch.randn(C, generator=g))
        ref[0].running_mean.copy_(0.1 * torch.randn(C, generator=g))
        ref[0].running_var.copy_(1 + 0.2 * torch.rand(C, generator=g))
    ours = BatchNormAct2d(C, eps=1e-3, momentum=0.01, act=act)
    ours.load_state_dict(ref[0].state_dict())
    return ref.to(DEV).train(), ours.to(DEV).train()


def _input(B, C, H, W, seed=1, mean_scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    sd = 0.5 + torch.rand(1, C, 1, 1, device=DEV, generator=g)
    if mean_scale > 1:    # |mean| / std = mean_scale in every channel
        mu = mean_scale * sd * torch.randn(1, C, 1, 1, device=DEV, generator=g).sign()
    else:
        mu = torch.randn(1, C, 1, 1, device=DEV, generator=g)
    x = mu + sd * torch.randn(B, C, H, W, device=DEV, generator=g)
    return x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)


def _run(mod, x, dy):
    x = x.detach().clone().requires_grad_(True)
    y = mod(x)
    y.backward(dy)
    return y.detach(), x.grad


def _within_ulp(got, ref):
    """Fraction of elements within one bf16 ulp of the reference."""
    g, r = got.double(), ref.double()
    tol = BF16_ULP * r.abs().clamp_min(2.0 ** -100) * 1.0001
    return float(((g - r).abs() <= tol).double().mean())


def _compare(B, C, H, W, act, steps=1, mean_scale=1.0, record=None, ulp_check=True):
    ref, ours = _pair(C, act)
    for step in range(steps):
        x = _input(B, C, H, W, seed=step + 1, mean_scale=mean_scale)
        dy = (torch.randn(x.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(100 + step))
              .to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
        for p in list(ref.parameters()) + list(ours.parameters()):
            p.grad = None
        y_r, dx_r = _run(ref, x, dy)
        y_o, dx_o = _run(ours, x, dy)
    assert y_o.is_contiguous(memory_format=torch.channels_last) and y_o.dtype == torch.bfloat16
    assert dx_o.is_contiguous(memory_format=torch.channels_last) and dx_o.dtype == torch.bfloat16
    bn = ref[0]
    # the batch statistics of the last step, from torch in double
    xd = x.double()
    mean = xd.mean((0, 2, 3))
    var = xd.var((0, 2, 3), unbiased=False)
    std = var.sqrt()
    errs = {
        "running_mean": float(((ours.running_mean.double() - bn.running_mean.double()).abs()
                               / (0.01 * std + bn.running_mean.double().abs() * 1e-3)).max()),
        "running_var": float(((ours.running_var.double() - bn.running_var.double()).abs()
                              / bn.running_var.double()).max()),
        "y": rel_l2(y_o, y_r), "dx": rel_l2(dx_o, dx_r),
        "y_ulp": _within_ulp(y_o, y_r), "dx_ulp": _within_ulp(dx_o, dx_r),
        "dw": rel_l2(ours.weight.grad, bn.weight.grad), "db": rel_l2(ours.bias.grad, bn.bias.grad),
    }
    assert int(ours.num_batches_tracked) == int(bn.num_batches_tracked) == steps
    # the saved statistics, read back through one more library forward of the last input
    from monocular_depth_estimation_b200 import _lib as L
    from monocular_depth_estimation_b200.functional import _BatchNormActFn
    y2 = _BatchNormActFn.apply(x, ours.weight, ours.bias, ours.running_mean.clone(), ours.running_var.clone(),
                               ours.num_batches_tracked.clone(), ours._tickets, 1e-3, 0.01, L.ACT_NONE)
    stats = y2.grad_fn.saved_tensors[3]
    d_mean = (stats[0].double() - mean).abs()
    errs["save_mean"] = float(torch.where(d_mean == 0, 0.0, d_mean / std).max())   # a constant channel has std 0
    errs["save_invstd"] = float(((stats[1].double() - 1 / (var + 1e-3).sqrt()).abs() * (var + 1e-3).sqrt()).max())
    if record is not None:
        record.append({"shape": [B, C, H, W], "act": act, **errs})
    assert errs["save_mean"] < 1e-5 and errs["save_invstd"] < 1e-5, errs
    assert errs["running_mean"] < 1e-3 and errs["running_var"] < 1e-5, errs
    assert errs["dw"] < 1e-4 and errs["db"] < 1e-4, errs
    assert errs["y"] < 1e-3 and errs["dx"] < 1e-3, errs
    if ulp_check:
        assert errs["y_ulp"] > 0.999 and errs["dx_ulp"] > 0.99, errs
    return errs


_RECORD = []


@pytest.mark.parametrize("C,H,W,act", ENCODER_SHAPES, ids=[f"{c}x{h}x{w}-{a}" for c, h, w, a in ENCODER_SHAPES])
def test_encoder_layer_matches_torch(C, H, W, act):
    _compare(8, C, H, W, act, steps=3, record=_RECORD)


@pytest.mark.parametrize("B,C,H,W,act", RAGGED)
def test_ragged_shapes_match_torch(B, C, H, W, act):
    _compare(B, C, H, W, act, steps=3, record=_RECORD)


@pytest.mark.parametrize("mean_scale", [10.0, 100.0])
def test_large_mean_against_spread(mean_scale):
    # The statistics and the rel-L2 bounds hold; the one-ulp count does not: at |mean| = 100 std the fp32 mean itself is
    # only known to 0.5 ulp(100 std) ~ 4e-6 std, which moves z = w (x - mean) invstd + b by more than its bf16 ulp where
    # z is near zero -- in torch's result as in ours, by different amounts.
    _compare(8, 64, 30, 40, "hardswish", mean_scale=mean_scale, record=_RECORD, ulp_check=mean_scale < 100)


def test_write_error_record():
    """Writes the errors measured by the parity tests above (when CRF_BN_RECORD names a file)."""
    path = os.environ.get("CRF_BN_RECORD")
    if path and _RECORD:
        with open(path, "w") as f:
            json.dump(_RECORD, f, indent=1)


def test_repeated_call_is_bit_identical():
    _, ours = _pair(120, "hardswish")
    x = _input(8, 120, 60, 80)
    dy = torch.randn_like(x)
    y1, dx1 = _run(ours, x, dy)
    g1 = (ours.weight.grad.clone(), ours.bias.grad.clone())
    ours.weight.grad = ours.bias.grad = None
    y2, dx2 = _run(ours, x, dy)
    assert torch.equal(y1, y2) and torch.equal(dx1, dx2)
    assert torch.equal(g1[0], ours.weight.grad) and torch.equal(g1[1], ours.bias.grad)


def test_cuda_graph_replay_matches_eager(monkeypatch):
    monkeypatch.setenv("CRF_DEBUG_GUARD", "0")    # the guard check synchronises, which a capture does not allow
    _, ours = _pair(40, "relu")
    _, eager = _pair(40, "relu")
    x_s = _input(8, 40, 60, 80)
    dy_s = torch.randn_like(x_s)
    xg = x_s.clone().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):     # warm-up (allocates the module's counters) outside the graph
        ours(xg).backward(dy_s)
    torch.cuda.current_stream().wait_stream(side)
    eager(x_s.clone().requires_grad_(True)).backward(dy_s)
    g = torch.cuda.CUDAGraph()
    ours.weight.grad = ours.bias.grad = None
    xg.grad = None
    with torch.cuda.graph(g):
        y_g = ours(xg)
        y_g.backward(dy_s)
    n0 = int(ours.num_batches_tracked)
    for step in range(3):
        xi = _input(8, 40, 60, 80, seed=10 + step)
        xg.detach().copy_(xi)
        g.replay()
        eager.weight.grad = eager.bias.grad = None
        y_e, dx_e = _run(eager, xi, dy_s)
        torch.cuda.synchronize()
        assert torch.equal(y_g, y_e) and torch.equal(xg.grad, dx_e)
        assert torch.equal(ours.weight.grad, eager.weight.grad) and torch.equal(ours.bias.grad, eager.bias.grad)
        assert torch.equal(ours.running_mean, eager.running_mean) and torch.equal(ours.running_var, eager.running_var)
        assert int(ours.num_batches_tracked) == n0 + step + 1 == int(eager.num_batches_tracked)


@pytest.mark.parametrize("case", ["eval", "fp32", "nchw", "c12", "momentum_none"])
def test_fallback_equals_stock_batchnorm(case):
    C = 12 if case == "c12" else 64
    ref, ours = _pair(C, "hardswish")
    x = _input(4, C, 10, 12)
    if case == "eval":
        ref.eval(), ours.eval()
    if case == "fp32":
        x = x.float().contiguous(memory_format=torch.channels_last)
    if case == "nchw":
        x = x.contiguous()
    if case == "momentum_none":
        ref[0].momentum = ours.momentum = None
    dy = torch.randn_like(x)
    y_r, dx_r = _run(ref, x, dy)
    y_o, dx_o = _run(ours, x, dy)
    assert ours._tickets is None          # the library was not used
    assert torch.equal(y_r, y_o) and torch.equal(dx_r, dx_o)
    assert torch.equal(ref[0].running_mean, ours.running_mean) and torch.equal(ref[0].running_var, ours.running_var)
    assert int(ref[0].num_batches_tracked) == int(ours.num_batches_tracked)


def test_single_value_per_channel_raises_like_torch():
    _, ours = _pair(16, "relu")
    with pytest.raises(ValueError, match="more than 1 value per channel"):
        ours(_input(1, 16, 1, 1))


def _unfuse(model):
    """The same model with stock BatchNorm2d + ReLU / Hardswish modules (holding the same tensors)."""
    from torchvision.ops.misc import Conv2dNormActivation
    from monocular_depth_estimation_b200.model import BatchNormAct2d
    for mod in model.modules():
        if isinstance(mod, Conv2dNormActivation) and isinstance(mod[1], BatchNormAct2d):
            b = mod[1]
            bn = nn.BatchNorm2d(b.num_features, b.eps, b.momentum, device="meta")
            bn._parameters.update(b._parameters)
            bn._buffers.update(b._buffers)
            mod[1] = bn.train(b.training)
            if b.act is not None:
                mod[2] = {"relu": nn.ReLU, "hardswish": nn.Hardswish}[b.act](inplace=True)
    return model


def test_whole_model_step_matches_stock_batchnorm():
    """One training step (bf16 autocast, channels-last): loss and per-group gradients of the library-BN model against the
    stock model stay within a small multiple of the stock model's own spread under a change of summation order -- the
    same step on the batch in reverse order (every per-image result is the same; BatchNorm statistics, weight gradients
    and the loss sum in another order)."""
    from monocular_depth_estimation_b200.model import PTModel
    from monocular_depth_estimation_b200.training import depth_norm
    from monocular_depth_estimation_b200.functional import depth_loss

    torch.manual_seed(0)
    img = torch.rand(4, 3, 192, 256, device=DEV).contiguous(memory_format=torch.channels_last)
    dep = torch.rand(4, 1, 192, 256, device=DEV)

    def step(model, reverse=False):
        x, d = (img.flip(0).contiguous(memory_format=torch.channels_last), dep.flip(0)) if reverse else (img, dep)
        model.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            pred = model(x)
        loss = depth_loss(pred, depth_norm(d))
        loss.backward()
        groups = {}
        for n, p in model.named_parameters():
            if p.grad is None:          # the classifier head of the torchvision model is not used
                continue
            key = "encoder" if n.startswith("Unet.0") else n.split(".")[2]
            groups.setdefault(key, []).append(p.grad.detach().flatten().double())
        return float(loss), {k: torch.cat(v) for k, v in groups.items()}

    def build(fused):
        m = fill_by_name(PTModel()).to(DEV).train().to(memory_format=torch.channels_last)
        return m if fused else _unfuse(m)

    ours = build(True)
    assert sum(type(m).__name__ == "BatchNormAct2d" for m in ours.modules()) == 46
    l_o, g_o = step(ours)
    l_s, g_s = step(build(False))
    l_r, g_r = step(build(False), reverse=True)
    rec = {"loss_ours": abs(l_o - l_s) / abs(l_s), "loss_spread": abs(l_r - l_s) / abs(l_s)}
    for k in g_s:
        rec[k] = (rel_l2(g_o[k], g_s[k]), rel_l2(g_r[k], g_s[k]))
    path = os.environ.get("CRF_BN_RECORD")
    if path:
        with open(path + ".model.json", "w") as f:
            json.dump(rec, f, indent=1)
    # one scalar: its rounding difference varies more from sample to sample than a whole gradient's rel-L2
    assert rec["loss_ours"] <= 10 * max(rec["loss_spread"], 1e-6), rec
    for k in g_s:
        assert rec[k][0] <= 4 * max(rec[k][1], 1e-4), (k, rec)
