"""DepthwiseConv2d on the library's depthwise kernels (crf_dwconv_fwd / crf_dwconv_bwd) against torch's conv2d: every
depthwise layer of the encoder at batch 8, ragged shapes, repeatability, CUDA-graph replay, the gradients left out, the
fallback cases and one whole-model training step."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests.helpers import fill_by_name, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF16_ULP = 2.0 ** -7     # bf16 spacing relative to the value (8 significant bits)


def _encoder_dw_shapes():
    """(C, H, W, k, stride) of the encoder's 15 depthwise convolutions at the bench resolution (480 x 640)."""
    import torchvision.models as tvm
    from monocular_depth_estimation_b200.model import DepthwiseConv2d, fuse_depthwise
    m = fuse_depthwise(tvm.mobilenet_v3_large().features)
    shapes = []
    for mod in m.modules():
        if isinstance(mod, DepthwiseConv2d):
            mod.register_forward_hook(lambda mod, inp, out: shapes.append(
                (mod.in_channels, inp[0].shape[2], inp[0].shape[3], mod.kernel_size[0], mod.stride[0])))
    with torch.no_grad():
        m.eval()(torch.zeros(1, 3, 480, 640))
    return shapes


ENCODER_SHAPES = _encoder_dw_shapes()
# (B, C, H, W, k, stride): batch 1, odd sizes at stride 2, maps smaller than the kernel, C = 8 / 72 / 184 / 200
RAGGED = [(1, 64, 33, 47, 3, 1), (2, 72, 15, 21, 3, 2), (3, 184, 7, 9, 5, 2), (2, 200, 15, 21, 5, 1),
          (2, 8, 1, 1, 5, 1), (1, 16, 2, 3, 5, 2), (2, 8, 4, 4, 5, 1), (1, 120, 4, 4, 5, 2), (4, 8, 9, 5, 3, 2),
          (1, 960, 1, 2, 3, 1)]


def _layer(C, k, s, seed=0):
    from monocular_depth_estimation_b200.model import DepthwiseConv2d
    g = torch.Generator().manual_seed(seed)
    m = DepthwiseConv2d(C, C, k, s, k // 2, groups=C, bias=False)
    with torch.no_grad():
        m.weight.copy_(torch.randn(C, 1, k, k, generator=g) / k)
    return m.to(DEV).to(memory_format=torch.channels_last)


def _input(B, C, H, W, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, C, H, W, generator=g).to(DEV, torch.bfloat16).contiguous(memory_format=torch.channels_last)


def _run(m, x, dy, autocast=True):
    xg = x.clone().requires_grad_(True)
    m.weight.grad = None
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        y = m(xg)
    y.backward(dy)
    return y.detach(), xg.grad, m.weight.grad


def _stock_run(m, x, dy):
    """The same layer as a stock nn.Conv2d holding the same weight: torch's bf16 cuDNN result."""
    ref = nn.Conv2d(m.in_channels, m.out_channels, m.kernel_size, m.stride, m.padding, groups=m.groups, bias=False)
    ref.weight = m.weight
    return _run(ref, x, dy)


def _exact(m, x, dy):
    """fp64 conv2d and its gradients on the bf16-rounded input and weight."""
    xd = x.double().requires_grad_(True)
    wd = m.weight.detach().to(torch.bfloat16).double().requires_grad_(True)
    y = F.conv2d(xd, wd, None, m.stride, m.padding, groups=m.groups)
    y.backward(dy.double())
    return y.detach(), xd.grad, wd.grad


def _within_ulp(a, b):
    """Fraction of elements of a within one bf16 ulp of b."""
    a, b = a.float(), b.float()
    return float(((a - b).abs() <= BF16_ULP * b.abs() + 1e-30).double().mean())


def _check(B, C, H, W, k, s, seed=0):
    m = _layer(C, k, s, seed)
    x = _input(B, C, H, W, seed + 1)
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    dy = _input(B, C, Ho, Wo, seed + 2)
    y, dx, dw = _run(m, x, dy)
    assert y.dtype == torch.bfloat16 and y.is_contiguous(memory_format=torch.channels_last)
    assert dx.dtype == torch.bfloat16 and dw.dtype == torch.float32 and dw.stride() == m.weight.stride()
    assert torch.equal(dw, dw.to(torch.bfloat16).float())          # rounded through bf16
    y_e, dx_e, dw_e = _exact(m, x, dy)
    errs = {"y": rel_l2(y, y_e), "dx": rel_l2(dx, dx_e), "dw": rel_l2(dw, dw_e)}
    assert all(e < 8e-3 for e in errs.values()), errs
    y_t, dx_t, dw_t = _stock_run(m, x, dy)
    ulp = {"y": _within_ulp(y, y_t), "dx": _within_ulp(dx, dx_t), "dw": _within_ulp(dw, dw_t)}
    assert ulp["y"] >= 0.99 and ulp["dx"] >= 0.99 and ulp["dw"] >= 0.9, (ulp, errs)
    return errs


@pytest.mark.parametrize("C,H,W,k,s", ENCODER_SHAPES, ids=[f"C{c}_{h}x{w}_k{k}_s{s}" for c, h, w, k, s in ENCODER_SHAPES])
def test_encoder_layer(C, H, W, k, s):
    _check(8, C, H, W, k, s)


def test_encoder_has_fifteen_depthwise_layers():
    assert len(ENCODER_SHAPES) == 15


@pytest.mark.parametrize("B,C,H,W,k,s", RAGGED)
def test_ragged(B, C, H, W, k, s):
    _check(B, C, H, W, k, s, seed=B + C + H)


@pytest.mark.parametrize("k,s", [(3, 1), (3, 2), (5, 1), (5, 2)])
def test_repeat_is_bit_identical(k, s):
    m = _layer(72, k, s)
    x = _input(4, 72, 45, 61)
    dy = _input(4, 72, (45 - 1) // s + 1, (61 - 1) // s + 1, 5)
    first = _run(m, x, dy)
    for _ in range(3):
        again = _run(m, x, dy)
        assert all(torch.equal(a, b) for a, b in zip(first, again))


def test_graph_replay_equals_eager_and_leaves_tickets_at_zero(monkeypatch):
    monkeypatch.setenv("CRF_DEBUG_GUARD", "0")         # the guard check synchronises, which a capture may not
    m = _layer(120, 5, 1)
    x = _input(8, 120, 60, 80)
    dy = _input(8, 120, 60, 80, 7)
    eager = [t.clone() for t in _run(m, x, dy)]     # the warm-up below accumulates into weight.grad in place
    xg = x.clone().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = m(xg)
            y.backward(dy)
    torch.cuda.current_stream().wait_stream(side)
    m.weight.grad, xg.grad = None, None
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = m(xg)
        y.backward(dy)
    for _ in range(3):
        m.weight.grad.zero_()
        xg.grad.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(y, eager[0]) and torch.equal(xg.grad, eager[1]) and torch.equal(m.weight.grad, eager[2])
        assert int(m._tickets.abs().sum()) == 0


def test_gradients_left_out():
    m = _layer(64, 3, 2)
    x = _input(2, 64, 31, 29)
    dy = _input(2, 64, 16, 15, 3)
    y, dx, dw = _run(m, x, dy)
    m.weight.requires_grad_(False)                     # input gradient only
    m.weight.grad = None
    with torch.autocast("cuda", dtype=torch.bfloat16):
        xg = x.clone().requires_grad_(True)
        y2 = m(xg)
    y2.backward(dy)
    assert torch.equal(xg.grad, dx) and m.weight.grad is None
    m.weight.requires_grad_(True)                      # weight gradient only
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y3 = m(x)
    y3.backward(dy)
    assert torch.equal(m.weight.grad, dw)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        assert torch.equal(m(x), y)


def _fallback_cases():
    base = dict(C=16, k=3, s=1, pad=None, dil=1, bias=False, mode="zeros", fmt=torch.channels_last,
                dtype=torch.bfloat16, autocast=torch.bfloat16)
    cases = {"no_autocast_fp32": dict(dtype=torch.float32, autocast=None),
             "fp16_autocast": dict(autocast=torch.float16),
             "nchw": dict(fmt=torch.contiguous_format),
             "fp32_input": dict(dtype=torch.float32),
             "c_not_multiple_of_8": dict(C=12),
             "k7": dict(k=7), "stride3": dict(s=3), "padding0": dict(pad=0), "dilation2": dict(dil=2, pad=2),
             "bias": dict(bias=True), "reflect": dict(mode="reflect")}
    return {n: {**base, **c} for n, c in cases.items()}


@pytest.mark.parametrize("name,case", list(_fallback_cases().items()))
def test_fallback_equals_stock_conv(name, case, monkeypatch):
    from monocular_depth_estimation_b200.model import DepthwiseConv2d
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)   # cuDNN's own weight gradients may use atomics
    C, k = case["C"], case["k"]
    pad = k // 2 if case["pad"] is None else case["pad"]
    args = (C, C, k, case["s"], pad, case["dil"], C, case["bias"], case["mode"])
    torch.manual_seed(0)
    ref = nn.Conv2d(*args).to(DEV)
    ours = DepthwiseConv2d.from_conv(copy_conv(ref))
    x = torch.randn(2, C, 13, 17, device=DEV).to(case["dtype"]).contiguous(memory_format=case["fmt"])
    outs = []
    for mod in (ref, ours):
        xg = x.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=case["autocast"] or torch.bfloat16, enabled=case["autocast"] is not None):
            y = mod(xg)
        y.float().square().sum().backward()
        outs.append((y, xg.grad, mod.weight.grad))
    assert ours._tickets is None                       # the library path was not taken
    for i, (a, b) in enumerate(zip(*outs)):
        if i == 1 and case["mode"] == "reflect":       # torch's reflection-pad backward adds with atomics
            torch.testing.assert_close(a, b, rtol=1e-2, atol=1e-2)
        else:
            assert torch.equal(a, b), (name, i)


def copy_conv(conv):
    c = nn.Conv2d(conv.in_channels, conv.out_channels, conv.kernel_size, conv.stride, conv.padding, conv.dilation,
                  conv.groups, conv.bias is not None, conv.padding_mode).to(conv.weight.device)
    c.load_state_dict(conv.state_dict())
    return c


def _unfuse(model):
    """The same model with stock nn.Conv2d depthwise modules (holding the same weights)."""
    from torchvision.ops.misc import Conv2dNormActivation
    from monocular_depth_estimation_b200.model import DepthwiseConv2d
    for mod in model.modules():
        if isinstance(mod, Conv2dNormActivation) and isinstance(mod[0], DepthwiseConv2d):
            d = mod[0]
            c = nn.Conv2d(d.in_channels, d.out_channels, d.kernel_size, d.stride, d.padding, d.dilation, d.groups,
                          False, device="meta")
            c._parameters.update(d._parameters)
            mod[0] = c.train(d.training)
    return model


def test_whole_model_step_matches_stock_depthwise():
    """One training step (bf16 autocast, channels-last): loss and per-group gradients of the library-depthwise model
    against the stock model stay within a small multiple of the stock model's own spread under a change of summation
    order -- the same step on the batch in reverse order."""
    from monocular_depth_estimation_b200.functional import depth_loss
    from monocular_depth_estimation_b200.model import DepthwiseConv2d, PTModel
    from monocular_depth_estimation_b200.training import depth_norm

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
            if p.grad is None:
                continue
            key = "encoder" if n.startswith("Unet.0") else n.split(".")[2]
            groups.setdefault(key, []).append(p.grad.detach().flatten().double())
        return float(loss), {k: torch.cat(v) for k, v in groups.items()}

    def build(fused):
        m = fill_by_name(PTModel()).to(DEV).train().to(memory_format=torch.channels_last)
        return m if fused else _unfuse(m)

    ours = build(True)
    assert sum(isinstance(m, DepthwiseConv2d) for m in ours.modules()) == 15
    l_o, g_o = step(ours)
    assert all(m._tickets is not None for m in ours.modules() if isinstance(m, DepthwiseConv2d))
    l_s, g_s = step(build(False))
    l_r, g_r = step(build(False), reverse=True)
    rec = {"loss_ours": abs(l_o - l_s) / abs(l_s), "loss_spread": abs(l_r - l_s) / abs(l_s)}
    for k in g_s:
        rec[k] = (rel_l2(g_o[k], g_s[k]), rel_l2(g_r[k], g_s[k]))
    assert rec["loss_ours"] <= 10 * max(rec["loss_spread"], 1e-6), rec
    for k in g_s:
        assert rec[k][0] <= 4 * max(rec[k][1], 1e-4), (k, rec)
