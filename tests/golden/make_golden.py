"""Generates the golden fixtures in this directory by EXECUTING THE UNMODIFIED REFERENCE
(/root/reference/src/newcrf_layers.py) on CPU in the build container.  /root/reference does not exist on the GPU box,
so the outputs are committed as small .npz files and this script documents how they were made.

    python tests/golden/make_golden.py            # rewrites tests/golden/*.npz
    python tests/golden/make_golden.py layer_8x13_c64_hd64 ...   # only the named fixtures

`timm` is not installed; the reference imports three trivial symbols from it that are only used at construction
time with rate 0 (newcrf_layers.py:6,107,184,187), so a stub module is injected (SURVEY.md Appendix A).
"""
import os
import sys
import types
import zlib

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
REF_SRC = "/root/reference/src"


def import_reference():
    tl = types.ModuleType("timm.models.layers")

    class DropPath(nn.Module):
        def __init__(self, p=0.):
            super().__init__()
            self.p = p

        def forward(self, x):
            return x

    tl.DropPath = DropPath
    tl.to_2tuple = lambda x: x if isinstance(x, tuple) else (x, x)
    tl.trunc_normal_ = nn.init.trunc_normal_
    sys.modules.update({"timm": types.ModuleType("timm"), "timm.models": types.ModuleType("timm.models"),
                        "timm.models.layers": tl})
    sys.path.insert(0, REF_SRC)
    import newcrf_layers as ref
    return ref


def randomize(module, gen):
    """Replace default-initialised parameters (zero biases, unit LN weights) by non-trivial values so that every
    parameter influences the output and receives a non-trivial gradient (tests.helpers.draw_layer_param, which the
    tests use to draw the same values again from the fixture's seed)."""
    from tests.helpers import draw_layer_param
    with torch.no_grad():
        for name, p in module.named_parameters():
            p.copy_(draw_layer_param(name, p.shape, gen))


# Gradients stored as a fixed half-sample of their elements, so that every fixture stays below 1 MB.
SAMPLED_GRADS = {"block_14x21_c128": ("blocks.0.mlp.fc1.weight", "blocks.0.mlp.fc2.weight")}


def write_layer_fixture(name, seed, meta, inputs, sd, outputs, grads):
    """A layer fixture holds the reference's outputs (y, dx, dv, `grad.<param>`) and what draws its inputs again
    (tests.helpers.layer_inputs_from_seed): the seed, the state_dict keys in order with their shapes, and the CRC32 of
    the inputs (x, v, dy, then the state_dict) the reference was run on."""
    crc = 0
    for t in [inputs["x"], inputs["v"], inputs["dy"]] + list(sd.values()):
        crc = zlib.crc32(np.ascontiguousarray(t).tobytes(), crc)
    blob = {"meta": meta, "seed": np.array([seed], dtype=np.int64), "sd_keys": np.array(list(sd)),
            "inputs_crc32": np.array([crc], dtype=np.int64)}
    blob.update({"shape." + k: np.array(t.shape, dtype=np.int64) for k, t in sd.items()})
    blob.update(outputs)
    blob.update({"grad." + k: g for k, g in grads.items()})
    rng = np.random.default_rng(seed)
    for k in SAMPLED_GRADS.get(name, ()):
        keep = rng.random(grads[k].size) < 0.5
        blob["mask.grad." + k] = np.packbits(keep)
        blob["grad." + k] = grads[k].reshape(-1)[keep]
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **blob)


def layer_case(ref, name, B, H, W, C, nH, depth, seed, strided):
    gen = torch.Generator().manual_seed(seed)
    layer = ref.BasicCRFLayer(dim=C, depth=depth, num_heads=nH, v_dim=C, window_size=7)
    randomize(layer, gen)
    if strided:   # the layouts NewCRF.forward hands over (newcrf_layers.py:426-427): strided views of NCHW
        x = torch.randn(B, C, H, W, generator=gen).flatten(2).transpose(1, 2)
        v = torch.randn(B, C, H, W, generator=gen).transpose(1, 2).transpose(2, 3)
    else:
        x = torch.randn(B, H * W, C, generator=gen)
        v = torch.randn(B, H, W, C, generator=gen)
    x = x.detach().requires_grad_(True)
    v = v.detach().requires_grad_(True)
    dy = torch.randn(B, H * W, C, generator=gen)
    out = layer(x, v, H, W)
    y = out[0]
    assert out[1] == H and out[2] == W and out[3] is y
    y.backward(dy)
    write_layer_fixture(name, seed, np.array([B, H, W, C, nH, depth, int(strided)], dtype=np.int64),
                        {"x": x.detach().contiguous().numpy(), "v": v.detach().contiguous().numpy(), "dy": dy.numpy()},
                        {k: t.numpy() for k, t in layer.state_dict().items()},
                        {"y": y.detach().numpy(), "dx": x.grad.contiguous().numpy(), "dv": v.grad.contiguous().numpy()},
                        {k: p.grad.numpy() for k, p in layer.named_parameters()})
    print(name, "y", tuple(y.shape), "abs-mean", float(y.abs().mean()))


def index_case(ref, name):
    """Integer-valued tensors through the reference's pad / roll / window_partition / window_reverse / crop and its
    attention mask: bit-exact index-map fixtures."""
    import torch.nn.functional as F
    blob = {}
    cases = [(15, 20, 0), (15, 20, 3), (9, 10, 3), (7, 7, 3), (14, 21, 0), (30, 40, 3), (8, 13, 3)]
    blob["cases"] = np.array(cases, dtype=np.int64)
    ws = 7
    for (H, W, s) in cases:
        x = torch.arange(1, 2 * H * W * 3 + 1, dtype=torch.float32).reshape(2, H, W, 3)
        pr, pb = (ws - W % ws) % ws, (ws - H % ws) % ws
        xp = F.pad(x, (0, 0, 0, pr, 0, pb))
        Hp, Wp = xp.shape[1], xp.shape[2]
        if s > 0:
            xp = torch.roll(xp, shifts=(-s, -s), dims=(1, 2))
        win = ref.window_partition(xp, ws).view(-1, ws * ws, 3)
        # reverse path on a different integer tensor
        wv = torch.arange(1, win.numel() + 1, dtype=torch.float32).reshape(win.shape)
        back = ref.window_reverse(wv.view(-1, ws, ws, 3), ws, Hp, Wp)
        if s > 0:
            back = torch.roll(back, shifts=(s, s), dims=(1, 2))
        back = back[:, :H, :W, :].contiguous()
        tag = f"{H}x{W}s{s}"
        blob["gather." + tag] = win.numpy()
        blob["scatter." + tag] = back.numpy()
        # the mask exactly as BasicCRFLayer.forward builds it (:332-350) with shift_size = ws // 2
        if s == ws // 2:
            img_mask = torch.zeros((1, Hp, Wp, 1))
            cnt = 0
            for hs in (slice(0, -ws), slice(-ws, -s), slice(-s, None)):
                for wsl in (slice(0, -ws), slice(-ws, -s), slice(-s, None)):
                    img_mask[:, hs, wsl, :] = cnt
                    cnt += 1
            mw = ref.window_partition(img_mask, ws).view(-1, ws * ws)
            am = mw.unsqueeze(1) - mw.unsqueeze(2)
            am = am.masked_fill(am != 0, float(-100.0)).masked_fill(am == 0, float(0.0))
            blob["mask." + tag] = am.numpy()
            blob["region." + tag] = mw.numpy().astype(np.int64)
    wa = ref.WindowAttention(64, (7, 7), 2, 64)
    blob["relative_position_index"] = wa.relative_position_index.numpy()
    blob["scale_hd32"] = np.array([wa.scale], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **blob)
    print(name, "ok")


def loss_case(name):
    """The training loss exactly as the reference computes it (src/train.py:94-100: l1_criterion = nn.L1Loss(),
    ssim = loss.SSIM(), loss = 1.0 * ssim + 0.1 * l1) on small maps, forward value and d loss / d prediction."""
    sys.path.insert(0, REF_SRC)
    import loss as ref_loss
    gen = torch.Generator().manual_seed(5)
    blob = {}
    for tag, shape in (("a", (2, 1, 11, 13)), ("b", (1, 1, 2, 2)), ("c", (3, 1, 3, 7))):
        pred = torch.rand(shape, generator=gen)
        tgt = (0.5 * pred + 0.5 * torch.rand(shape, generator=gen)).clamp(0, 1)
        tgt[..., : shape[-1] // 2] = pred[..., : shape[-1] // 2]   # SSIM = 1 there: the clamp's lower boundary
        pred = pred.detach().requires_grad_(True)
        val = 1.0 * ref_loss.SSIM()(pred, tgt) + 0.1 * nn.L1Loss()(pred, tgt)
        val.backward()
        blob[f"pred.{tag}"], blob[f"target.{tag}"] = pred.detach().numpy(), tgt.numpy()
        blob[f"loss.{tag}"] = np.array([float(val.detach())], dtype=np.float64)
        blob[f"dpred.{tag}"] = pred.grad.numpy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **blob)
    print(name, "ok")


def model_case(name):
    """The reference's whole model (src/model_mobileV3_large_newCRFs.py: torchvision MobileNetV3-large encoder + NeWCRFs
    decoder), unmodified, eval mode, on a small image: depth map, loss as in train.py:89-100, gradients of the image and
    of a dozen small parameters.  Weights come from tests.helpers.fill_by_name (seeded by parameter NAME), so the oracle
    and the product rebuild exactly the same model without a checkpoint.  Import shims (SURVEY.md Appendix A):
    matplotlib is absent (utils.py imports it for colour maps only) and `pretrained=True` needs the network."""
    from tests.helpers import MODEL_GRAD_KEYS, fill_by_name
    for m in ("matplotlib", "matplotlib.cm"):
        sys.modules.setdefault(m, types.ModuleType(m))
    import torchvision.models as tvm
    orig = tvm.mobilenet_v3_large
    tvm.mobilenet_v3_large = lambda *a, **k: orig(weights=None)
    try:
        import model_mobileV3_large_newCRFs as ref_model
        import loss as ref_loss
        from utils import DepthNorm
        model = ref_model.PTModel()
    finally:
        tvm.mobilenet_v3_large = orig
    fill_by_name(model).eval()
    gen = torch.Generator().manual_seed(11)
    image = torch.rand(2, 3, 64, 96, generator=gen).requires_grad_(True)
    depth = torch.rand(2, 1, 64, 96, generator=gen) * 9.0 + 1.0
    pred = model(image)
    val = 1.0 * ref_loss.SSIM()(pred, DepthNorm(depth)) + 0.1 * nn.L1Loss()(pred, DepthNorm(depth))
    val.backward()
    params = dict(model.named_parameters())
    blob = {"image": image.detach().numpy(), "depth": depth.numpy(), "pred": pred.detach().numpy(),
            "loss": np.array([float(val.detach())], dtype=np.float64), "dimage": image.grad.numpy(),
            "keys": np.array(sorted(model.state_dict().keys()))}
    for k in MODEL_GRAD_KEYS:
        blob["grad." + k] = params[k].grad.numpy().copy()
    # Yardstick for the bf16-I/O tolerance of deep gradients: the UNMODIFIED reference under torch's own bf16 autocast
    # against its fp32 run above, per quantity (rel-L2).  The product's bf16 path has to stay below the reference's own
    # bf16 deviation on every one of them (tests/test_gpu_block.py::test_full_model_matches_reference_model_golden).
    def rel(a, b):
        a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
        return float((a - b).norm() / b.norm())
    model.zero_grad(set_to_none=True)
    image2 = image.detach().clone().requires_grad_(True)
    with torch.autocast("cpu", dtype=torch.bfloat16):
        pred2 = model(image2)
    pred2 = pred2.float()
    val2 = 1.0 * ref_loss.SSIM()(pred2, DepthNorm(depth)) + 0.1 * nn.L1Loss()(pred2, DepthNorm(depth))
    val2.backward()
    blob["bf16ref.pred"] = np.array([rel(pred2.detach(), blob["pred"])])
    blob["bf16ref.dimage"] = np.array([rel(image2.grad, blob["dimage"])])
    for k in MODEL_GRAD_KEYS:
        blob["bf16ref." + k] = np.array([rel(params[k].grad, blob["grad." + k])])
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **blob)
    print(name, "pred", tuple(pred.shape), "mean", float(pred.mean()), "std", float(pred.std()), "loss", float(val))


def main():
    torch.manual_seed(0)
    torch.set_num_threads(4)
    ref = import_reference()
    only = set(sys.argv[1:])
    want = lambda name: not only or name in only
    if want("index_maps"):
        index_case(ref, "index_maps")
    if want("loss_ssim_l1"):
        loss_case("loss_ssim_l1")
    cases = [
        # (a) both blocks (shift 0 and 3), both dims padded, strided NCHW-view inputs like NewCRF.forward produces
        dict(name="layer_9x10_c64", B=2, H=9, W=10, C=64, nH=2, depth=2, seed=1, strided=True),
        # (b) decoder scale 1/32 geometry (15x20 -> 21x21) with contiguous inputs
        dict(name="layer_15x20_c64", B=1, H=15, W=20, C=64, nH=2, depth=2, seed=2, strided=False),
        # (c) no padding at all (14x21), C=128 / 4 heads (config-1 channel geometry), single unshifted block
        dict(name="block_14x21_c128", B=1, H=14, W=21, C=128, nH=4, depth=1, seed=3, strided=False),
        # (d), (e) BASELINE configs[2] head widths other than 32: one 64-wide head, four 16-wide heads
        dict(name="layer_8x13_c64_hd64", B=1, H=8, W=13, C=64, nH=1, depth=2, seed=4, strided=True),
        dict(name="layer_8x13_c64_hd16", B=1, H=8, W=13, C=64, nH=4, depth=2, seed=6, strided=True),
    ]
    for c in cases:
        if want(c["name"]):
            layer_case(ref, **c)
    if want("model_64x96"):
        model_case("model_64x96")


if __name__ == "__main__":
    main()
