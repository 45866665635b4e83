"""Shared test helpers: golden-fixture loading and error metrics."""
import os
import zlib

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LAYER_CASES = ["layer_9x10_c64", "layer_15x20_c64", "block_14x21_c128"]
HEAD_CASES = ["layer_8x13_c64_hd64", "layer_8x13_c64_hd16"]   # head widths other than 32 (BASELINE configs[2])


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    g = {k: z[k] for k in z.files}
    if "seed" in g:
        g.update(layer_inputs_from_seed(g))
    return g


def draw_layer_param(name, shape, gen):
    """One parameter of a layer fixture: non-trivial values (no zero biases or unit LN weights) so that every
    parameter influences the output and receives a non-trivial gradient."""
    if name.endswith("norm1.weight") or name.endswith("norm2.weight"):
        return 1.0 + 0.1 * torch.randn(shape, generator=gen)
    if name.endswith(".bias"):
        return 0.1 * torch.randn(shape, generator=gen)
    if name.endswith("relative_position_bias_table"):
        return 0.2 * torch.randn(shape, generator=gen)
    return torch.randn(shape, generator=gen) * shape[-1] ** -0.5


def layer_inputs_from_seed(g):
    """The inputs of a layer fixture (x, v, dy and the state_dict as `sd.<key>`), drawn from the fixture's seed in the
    order tests/golden/make_golden.py drew them for the reference: the parameters in state_dict order, then x, v, dy.
    A layer fixture stores only the seed, the reference's state_dict keys and shapes, and the reference's outputs;
    `inputs_crc32` pins the redrawn inputs to the ones the reference saw."""
    B, H, W, C, nH, depth, strided = [int(t) for t in g["meta"]]
    gen = torch.Generator().manual_seed(int(g["seed"][0]))
    out = {}
    for k in g["sd_keys"].tolist():
        shape = tuple(int(s) for s in g["shape." + k])
        if k.endswith("relative_position_index"):   # a buffer, not drawn: the reference's own index map
            idx = np.load(os.path.join(GOLDEN, "index_maps.npz"))["relative_position_index"]
            assert idx.shape == shape, (k, idx.shape, shape)
            out["sd." + k] = idx
        else:
            out["sd." + k] = draw_layer_param(k, shape, gen).numpy()
    if strided:   # drawn as NCHW maps, the layouts NewCRF.forward hands over (newcrf_layers.py:426-427)
        x = torch.randn(B, C, H, W, generator=gen).flatten(2).transpose(1, 2)
        v = torch.randn(B, C, H, W, generator=gen).transpose(1, 2).transpose(2, 3)
    else:
        x = torch.randn(B, H * W, C, generator=gen)
        v = torch.randn(B, H, W, C, generator=gen)
    out["x"], out["v"] = x.contiguous().numpy(), v.contiguous().numpy()
    out["dy"] = torch.randn(B, H * W, C, generator=gen).numpy()
    crc = 0
    for k in ["x", "v", "dy"] + ["sd." + k for k in g["sd_keys"].tolist()]:
        crc = zlib.crc32(np.ascontiguousarray(out[k]).tobytes(), crc)
    assert crc == int(g["inputs_crc32"][0]), "the redrawn inputs differ from the ones the reference was run on"
    return out


def golden_rel_l2(g, key, t):
    """rel_l2 of `t` against the fixture's `g[key]`.  Where the fixture stores a fixed sample of a large tensor
    (`mask.<key>`: np.packbits of a boolean mask over the flattened tensor), on the sampled elements."""
    if "mask." + key not in g:
        return rel_l2(t, g[key])
    t = torch.as_tensor(t).detach().reshape(-1).cpu()
    keep = np.unpackbits(g["mask." + key])[: t.numel()].astype(bool)
    return rel_l2(t[torch.from_numpy(keep)], g[key])


def rel_l2(a, b):
    """||a - b||_2 / ||b||_2 in float64 -- the 'rel' of BASELINE.json's tolerances."""
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def max_rel(a, b):
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def golden_layer_inputs(g, device="cpu"):
    """Rebuild the (possibly strided) inputs and the per-block parameter dicts of a layer fixture."""
    B, H, W, C, nH, depth, strided = [int(t) for t in g["meta"]]
    x = torch.from_numpy(g["x"]).to(device)
    v = torch.from_numpy(g["v"]).to(device)
    if strided:  # re-create the NCHW-view strides NewCRF.forward produces (newcrf_layers.py:426-427)
        x = x.transpose(1, 2).contiguous().transpose(1, 2)
        v = v.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)
    blocks = []
    for i in range(depth):
        pre = f"sd.blocks.{i}."
        blocks.append({k[len(pre):]: torch.from_numpy(t).to(device) for k, t in g.items()
                       if k.startswith(pre) and not k.endswith("relative_position_index")})
    return (B, H, W, C, nH, depth), x, v, blocks


def fill_by_name(module):
    """Deterministic, construction-order-independent values for every parameter and BatchNorm statistic of a model:
    each tensor is drawn from a generator seeded by the CRC32 of its state_dict name.  The reference model (in the build
    container, tests/golden/make_golden.py), the oracle model and the product model therefore get identical weights
    from their NAMES alone -- no 180 MB checkpoint has to travel to the GPU box."""
    with torch.no_grad():
        for name, t in list(module.named_parameters()) + list(module.named_buffers()):
            if name.endswith("relative_position_index") or name.endswith("num_batches_tracked"):
                continue
            g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            r = torch.randn(t.shape, generator=g)
            if name.endswith("running_var"):
                t.copy_(1.0 + 0.2 * r.abs())
            elif name.endswith("running_mean"):
                t.copy_(0.1 * r)
            elif name.endswith("relative_position_bias_table"):
                t.copy_(0.2 * r)
            elif t.dim() >= 2:                      # conv / linear weights: He scaling keeps activations O(1)
                t.copy_(r * (2.0 / t[0].numel()) ** 0.5)
            elif name.endswith("weight"):           # LayerNorm / BatchNorm scales
                t.copy_(1.0 + 0.1 * r)
            else:                                   # biases
                t.copy_(0.1 * r)
    return module


# parameters whose gradients the full-model fixture stores (small tensors spread over encoder, bridge, every stage, head)
MODEL_GRAD_KEYS = ["Unet.0.original_model.features.0.0.weight", "Unet.1.conv0.bias", "Unet.1.conv1.weight",
                   "Unet.1.crf3.norm_crf.weight", "Unet.1.crf3.crf_layer.blocks.1.attn.relative_position_bias_table",
                   "Unet.1.crf2.crf_layer.blocks.0.attn.qk.bias", "Unet.1.crf2.proj_v.bias",
                   "Unet.1.crf1.crf_layer.blocks.1.mlp.fc2.bias", "Unet.1.crf1.norm_crf.bias",
                   "Unet.1.crf0.crf_layer.blocks.0.norm1.weight", "Unet.1.crf0.crf_layer.blocks.1.attn.proj.bias",
                   "Unet.1.crf0.proj_x.bias"]
