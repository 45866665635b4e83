"""Parity of the fused CRF block / layer (CUDA path through the C ABI) with the reference: golden vectors produced by
the unmodified reference module, and the oracle on seeded inputs at BASELINE.json config-1 and config-2 shapes.

Tolerance: this is the bf16-I/O path (bf16 tensor-core operands and bf16 intermediates, fp32 accumulation, fp32
residual stream, fp32 softmax/LayerNorm): BASELINE.json states rel 2e-2 for it, rel = ||a-b||_2 / ||b||_2.
"""
import pytest
import torch

from oracle import crf_oracle as O
from tests.helpers import HEAD_CASES, LAYER_CASES, golden_layer_inputs, golden_rel_l2, load_golden, rel_l2

pytestmark = pytest.mark.gpu
TOL = 2e-2          # BASELINE.json's bound of the bf16-I/O tier; kept for parameter gradients (worst measured 1.1e-2)
TOL_Y = 6e-3        # forward output: worst measured 2.9e-3 (profiles/r02_parity_errs_*.jsonl)
TOL_DXDV = 1.5e-2   # input gradients: worst measured 6.4e-3
TOL_ROW = 2e-2      # per-token-row relative error of y / dx / dv: a defect confined to one window cannot hide in a
                    # whole-tensor norm (rows are ~3e-3 .. 8e-3 off)
DEV = "cuda"


def _tol(key, tier=None):
    """Bound for one compared quantity: ~3x the worst measured error of the bf16 tier, or the fp32 tier's bound."""
    if tier is not None:
        return tier
    return TOL_Y if key == "y" else TOL_DXDV if key in ("dx", "dv") else TOL


def _row_err(a, b):
    """max over token rows of ||a_t - b_t|| / ||b_t|| (rows with a negligible reference norm are skipped)."""
    a = torch.as_tensor(a).detach().double().cpu().reshape(-1, a.shape[-1])
    b = torch.as_tensor(b).detach().double().cpu().reshape(-1, b.shape[-1])
    nb = b.norm(dim=1)
    keep = nb > 1e-3 * nb.mean()
    return float(((a - b).norm(dim=1)[keep] / nb[keep]).max())


def _report(case, errs):
    """Append the measured relative errors to gpurun_out/parity_errs.jsonl (evidence for DESIGN.md)."""
    import json, os
    if os.path.isdir("gpurun_out"):
        with open("gpurun_out/parity_errs.jsonl", "a") as f:
            f.write(json.dumps({"case": case, "max": max(errs.values()), "errs": errs}) + "\n")


def _pkg():
    import monocular_depth_estimation_b200 as pkg
    return pkg


def _layer_from_golden(g, C, nH, depth):
    pkg = _pkg()
    layer = pkg.BasicCRFLayer(dim=C, depth=depth, num_heads=nH, v_dim=C, window_size=7)
    sd = {k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")}
    missing, unexpected = layer.load_state_dict(sd, strict=True)   # drop-in: reference checkpoint keys load as-is
    assert not missing and not unexpected
    return layer.to(DEV)


@pytest.mark.parametrize("name", HEAD_CASES)
def test_head_width_golden(name):
    """The reference's own outputs / gradients for one 64-wide head and for four 16-wide heads."""
    test_layer_matches_reference_golden(name)


@pytest.mark.parametrize("name", LAYER_CASES)
def test_layer_matches_reference_golden(name):
    g = load_golden(name)
    (B, H, W, C, nH, depth), x, v, _ = golden_layer_inputs(g, DEV)
    layer = _layer_from_golden(g, C, nH, depth)
    x = x.detach().requires_grad_(True)
    v = v.detach().requires_grad_(True)
    out = layer(x, v, H, W)
    assert out[1] == H and out[2] == W and out[3] is out[0] and out[4] == H and out[5] == W
    y = out[0]
    assert y.shape == (B, H * W, C) and y.is_contiguous()
    y.backward(torch.from_numpy(g["dy"]).to(DEV))
    torch.cuda.synchronize()
    errs = {"y": rel_l2(y.detach(), g["y"]), "dx": rel_l2(x.grad, g["dx"]), "dv": rel_l2(v.grad, g["dv"])}
    for k, p in layer.named_parameters():
        errs[k] = golden_rel_l2(g, "grad." + k, p.grad)
    _report("golden " + name, errs)
    bad = {k: e for k, e in errs.items() if not e < _tol(k)}
    assert not bad, f"rel_l2 above the bound: {bad}\nall: {errs}"


@pytest.mark.parametrize("out_bf16", [False, True])
@pytest.mark.parametrize("B,H,W,C,nH,depth", [(2, 9, 10, 64, 2, 2), (2, 15, 20, 128, 4, 2), (1, 30, 40, 256, 8, 1),
                                               (2, 9, 10, 192, 6, 2), (1, 15, 20, 640, 5, 1)])
def test_layer_with_pixel_shuffle_folded_in(B, H, W, C, nH, depth, out_bf16):
    """crf_layer_args.out_shuffle: the stage-closing LayerNorm writes nn.PixelShuffle(2) of the stage's NCHW output
    (model_mobileV3_large_newCRFs.py:116-120) -- bit-identical to the unshuffled layer call + F.pixel_shuffle, and the
    same gradients (the backward reads the shuffled gradient map)."""
    pkg = _pkg()
    torch.manual_seed(11 * depth + C)
    layer = pkg.BasicCRFLayer(dim=C, depth=depth, num_heads=nH, v_dim=C).to(DEV)
    norm = torch.nn.LayerNorm(C).to(DEV)
    with torch.no_grad():
        norm.weight.normal_(1.0, 0.2)
        norm.bias.normal_(0.0, 0.2)
    x0 = torch.randn(B, C, H, W, device=DEV).flatten(2).transpose(1, 2)
    v0 = torch.randn(B, C, H, W, device=DEV).permute(0, 2, 3, 1)
    odt = torch.bfloat16 if out_bf16 else torch.float32
    gy = torch.randn(B, C // 4, 2 * H, 2 * W, device=DEV).to(odt)

    def run(shuffle):
        for p_ in list(layer.parameters()) + list(norm.parameters()):
            p_.grad = None
        x, v = x0.detach().requires_grad_(True), v0.detach().requires_grad_(True)
        y = layer.run(x, v, H, W, norm=norm, out_dtype=odt, pixel_shuffle=shuffle)
        if not shuffle:
            y = torch.nn.functional.pixel_shuffle(y.view(B, H, W, C).permute(0, 3, 1, 2), 2)
        assert y.shape == (B, C // 4, 2 * H, 2 * W)
        y.backward(gy)
        grads = {k: p_.grad.clone() for k, p_ in layer.named_parameters()}
        grads.update({"norm." + k: p_.grad.clone() for k, p_ in norm.named_parameters()})
        return y.detach(), x.grad.clone(), v.grad.clone(), grads

    yf, dxf, dvf, gf = run(True)
    yr, dxr, dvr, gr = run(False)
    assert yf.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(yf, yr), "forward differs"
    assert rel_l2(dxf, dxr) < 1e-6 and rel_l2(dvf, dvr) < 1e-6, (rel_l2(dxf, dxr), rel_l2(dvf, dvr))
    bad = {k: rel_l2(gf[k], gr[k]) for k in gr if not rel_l2(gf[k], gr[k]) < 1e-5}
    assert not bad, bad


@pytest.mark.parametrize("with_norm,out_bf16", [(False, False), (True, False), (True, True)])
@pytest.mark.parametrize("B,H,W,C,nH,depth", [(2, 9, 10, 64, 2, 2), (2, 15, 20, 128, 4, 3), (1, 30, 40, 256, 8, 1),
                                               (2, 9, 10, 192, 6, 2), (1, 15, 20, 640, 5, 1)])
def test_layer_call_equals_block_by_block(B, H, W, C, nH, depth, with_norm, out_bf16):
    """crf_layer_fwd / crf_layer_bwd (one call per BasicCRFLayer incl. the closing norm_crf) against the same layer run
    block by block through crf_block_fwd / crf_block_bwd + the stand-alone LayerNorm: same kernels, same order of
    fp32 operations -> outputs, dx, dv and every parameter gradient must agree to fp32 round-off (the bf16 twins the
    layer call hands between blocks are bit-identical to the casts the block path makes)."""
    pkg = _pkg()
    from monocular_depth_estimation_b200 import functional as CF
    torch.manual_seed(7 * depth + C)
    layer = pkg.BasicCRFLayer(dim=C, depth=depth, num_heads=nH, v_dim=C).to(DEV)
    norm = torch.nn.LayerNorm(C).to(DEV) if with_norm else None
    if norm is not None:
        with torch.no_grad():
            norm.weight.normal_(1.0, 0.2)
            norm.bias.normal_(0.0, 0.2)
    x0 = torch.randn(B, C, H, W, device=DEV).flatten(2).transpose(1, 2)
    v0 = torch.randn(B, C, H, W, device=DEV).permute(0, 2, 3, 1)
    gy = torch.randn(B, H * W, C, device=DEV)
    odt = torch.bfloat16 if out_bf16 else torch.float32

    def run(fused):
        for p_ in list(layer.parameters()) + (list(norm.parameters()) if norm is not None else []):
            p_.grad = None
        x = x0.detach().clone().requires_grad_(True) if False else x0.detach().requires_grad_(True)
        v = v0.detach().requires_grad_(True)
        if fused:
            y = layer.run(x, v, H, W, norm=norm, out_dtype=odt)
        else:
            vb = CF.convert_v(v)
            y = x
            for blk in layer.blocks:
                blk.H, blk.W = H, W
                y = blk(y, v, None, v_bf16=vb)
            if norm is not None:
                y = CF.layer_norm(y, norm.weight, norm.bias, norm.eps, out_dtype=odt)
        y.backward(gy.to(y.dtype))
        grads = {k: p_.grad.clone() for k, p_ in layer.named_parameters()}
        if norm is not None:
            grads.update({"norm." + k: p_.grad.clone() for k, p_ in norm.named_parameters()})
        return y.detach().float(), x.grad.clone(), v.grad.clone(), grads

    yf, dxf, dvf, gf = run(True)
    yb, dxb, dvb, gb = run(False)
    assert yf.dtype == yb.dtype and torch.equal(yf, yb), "forward differs"
    assert rel_l2(dxf, dxb) < 1e-6 and rel_l2(dvf, dvb) < 1e-6, (rel_l2(dxf, dxb), rel_l2(dvf, dvb))
    bad = {k: rel_l2(gf[k], gb[k]) for k in gb if not rel_l2(gf[k], gb[k]) < 1e-5}
    assert not bad, bad


def test_layer_call_bf16_inputs_gradient_dtype():
    """bf16 x / v (the autocast pipeline): the layer call returns dx in bf16 straight from the LayerNorm backward; it must
    equal the block-by-block path, whose fp32 dx autograd rounds to bf16 afterwards."""
    pkg = _pkg()
    from monocular_depth_estimation_b200 import functional as CF
    torch.manual_seed(11)
    B, H, W, C, nH = 2, 15, 20, 128, 4
    layer = pkg.BasicCRFLayer(dim=C, depth=2, num_heads=nH, v_dim=C).to(DEV)
    xs = torch.randn(B, H, W, C, device=DEV).to(torch.bfloat16)      # channels-last conv output: token-major rows
    vs = torch.randn(B, H, W, C, device=DEV).to(torch.bfloat16)
    gy = torch.randn(B, H * W, C, device=DEV)
    outs = []
    for fused in (True, False):
        x = xs.view(B, H * W, C).detach().requires_grad_(True)
        v = vs.detach().requires_grad_(True)
        if fused:
            y = layer.run(x, v, H, W)
        else:
            vb = CF.convert_v(v)
            y = x
            for blk in layer.blocks:
                blk.H, blk.W = H, W
                y = blk(y, v, None, v_bf16=vb)
        y.backward(gy)
        assert x.grad.dtype == torch.bfloat16 and v.grad.dtype == torch.bfloat16
        outs.append((y.detach(), x.grad.clone(), v.grad.clone()))
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][1], outs[1][1]), rel_l2(outs[0][1].float(), outs[1][1].float())
    # dv: the block path sums two bf16-rounded gradients in bf16 (autograd), the layer call rounds the fp32 sum once
    assert rel_l2(outs[0][2].float(), outs[1][2].float()) < 1e-2


def _run_block_vs_oracle(B, H, W, C, nH, shift, seed, strided, oracle_device, precision=None, tol=TOL, mask=None):
    from monocular_depth_estimation_b200 import functional as CF
    gen = torch.Generator().manual_seed(seed)
    p = O.init_block_params(C, nH, gen)
    if strided:
        x = torch.randn(B, C, H, W, generator=gen).flatten(2).transpose(1, 2)
        v = torch.randn(B, C, H, W, generator=gen).permute(0, 2, 3, 1)
    else:
        x = torch.randn(B, H * W, C, generator=gen)
        v = torch.randn(B, H, W, C, generator=gen)
    dy = torch.randn(B, H * W, C, generator=gen)
    # oracle (fp32)
    po = {k: t.detach().clone().to(oracle_device).requires_grad_(True) for k, t in p.items()}
    xo = x.to(oracle_device).detach().requires_grad_(True)
    vo = v.to(oracle_device).detach().requires_grad_(True)
    yo = O.crf_block(xo, vo, H, W, po, nH, 7, shift, mask_matrix=mask)
    yo.backward(dy.to(oracle_device))
    # CUDA path
    pc = {k: t.detach().clone().to(DEV).requires_grad_(True) for k, t in p.items()}
    xc = x.to(DEV)
    vc = v.to(DEV)
    if strided and H * W > 1:  # .to() keeps the permuted strides
        assert not xc.is_contiguous()
    xc = xc.detach().requires_grad_(True)
    vc = vc.detach().requires_grad_(True)
    yc = CF.crf_block(xc, vc, H, W, [pc[k] for k in CF.PARAM_KEYS], nH, window=7, shift=shift, precision=precision,
                      mask=None if mask is None else mask.to(DEV))
    yc.backward(dy.to(DEV))
    torch.cuda.synchronize()
    errs = {"y": rel_l2(yc.detach(), yo.detach()), "dx": rel_l2(xc.grad, xo.grad), "dv": rel_l2(vc.grad, vo.grad)}
    for k in CF.PARAM_KEYS:
        errs[k] = rel_l2(pc[k].grad, po[k].grad)
    _report(f"block B{B} {H}x{W} C{C} nH{nH} shift{shift} strided{int(strided)} oracle@{oracle_device}"
            + (f" precision={precision}" if precision else "") + (" custom-mask" if mask is not None else ""), errs)
    fp32 = precision == "fp32"
    bad = {k: e for k, e in errs.items() if not e < (tol if (fp32 or tol != TOL) else _tol(k))}
    assert not bad, f"rel_l2 above the bound: {bad}\nall: {errs}"
    rows = {"y": _row_err(yc, yo), "dx": _row_err(xc.grad, xo.grad), "dv": _row_err(vc.grad, vo.grad)}
    row_tol = 1e-3 if fp32 else TOL_ROW   # fp32 tier: the spec bound per row
    assert all(e < row_tol for e in rows.values()), f"per-token-row error above {row_tol}: {rows}"
    return errs


# ---------------------------------------------------------------------------------------------------------------------
# The fp32 precision mode: BASELINE.json's "rel 1e-3 for the fp32-accumulate path" (split-operand tensor-core GEMMs,
# fp32 intermediates, fp32 attention; csrc/crf_precise.cu).  Same cases as the bf16 tier, tolerance 1e-3 on the output,
# dx, dv and every one of the 13 parameter gradients.
# ---------------------------------------------------------------------------------------------------------------------
TOL_FP32 = 1.5e-4   # BASELINE.json asks for rel 1e-3; measured worst 3.6e-5 (C = 1024), typical 1.2e-5: bound at ~4x


@pytest.mark.parametrize("shift", [0, 3])
@pytest.mark.parametrize("strided", [False, True])
def test_fp32_mode_config1_block_vs_oracle_cpu(shift, strided):
    """BASELINE.json configs[0] in the fp32 mode against the fp32 CPU oracle."""
    _run_block_vs_oracle(2, 60, 80, 128, 4, shift, seed=10 + shift, strided=strided, oracle_device="cpu",
                         precision="fp32", tol=TOL_FP32)


@pytest.mark.parametrize("H,W,C,nH,B", [(120, 160, 128, 4, 8), (60, 80, 256, 8, 2), (30, 40, 512, 16, 2), (15, 20, 1024, 32, 8),
                                        (9, 10, 64, 4, 2), (9, 10, 64, 1, 2), (16, 23, 256, 2, 1), (1, 1, 64, 2, 1)])
def test_fp32_mode_shapes_vs_oracle(H, W, C, nH, B):
    """Decoder-scale shapes of configs[1], head widths 16 / 32 / 64 / 128, ragged maps; shifted windows."""
    _run_block_vs_oracle(B, H, W, C, nH, 3, seed=500 + C + H, strided=True, oracle_device=DEV, precision="fp32", tol=TOL_FP32)


@pytest.mark.parametrize("name", LAYER_CASES + HEAD_CASES)
def test_fp32_mode_layer_matches_reference_golden(name):
    """The reference's own golden vectors (whole BasicCRFLayer: both blocks, strided NCHW-view inputs) at rel 1e-3."""
    g = load_golden(name)
    (B, H, W, C, nH, depth), x, v, _ = golden_layer_inputs(g, DEV)
    layer = _layer_from_golden(g, C, nH, depth)
    layer.precision = "fp32"
    x = x.detach().requires_grad_(True)
    v = v.detach().requires_grad_(True)
    y = layer(x, v, H, W)[0]
    y.backward(torch.from_numpy(g["dy"]).to(DEV))
    torch.cuda.synchronize()
    errs = {"y": rel_l2(y.detach(), g["y"]), "dx": rel_l2(x.grad, g["dx"]), "dv": rel_l2(v.grad, g["dv"])}
    for k, p in layer.named_parameters():
        errs[k] = golden_rel_l2(g, "grad." + k, p.grad)
    _report("golden fp32-mode " + name, errs)
    bad = {k: e for k, e in errs.items() if not e < TOL_FP32}
    assert not bad, f"rel_l2 above {TOL_FP32}: {bad}\nall: {errs}"


# ---------------------------------------------------------------------------------------------------------------------
# CRFBlock.forward(x, v, mask_matrix): a mask other than the standard one is honoured (newcrf_layers.py:195,225-236)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("H,W,C,nH", [(15, 20, 128, 4), (9, 10, 64, 1)])
def test_block_honours_custom_mask_matrix(H, W, C, nH, precision):
    gen = torch.Generator().manual_seed(77)
    nW = (-(-H // 7)) * (-(-W // 7))
    mask = torch.where(torch.rand(nW, 49, 49, generator=gen) < 0.3, -100.0, 0.0) + 0.5 * torch.randn(nW, 49, 49, generator=gen)
    _run_block_vs_oracle(2, H, W, C, nH, 3, seed=700 + C, strided=True, oracle_device=DEV, precision=precision,
                         tol=TOL if precision == "bf16" else TOL_FP32, mask=mask)


def test_block_module_recognises_the_standard_mask():
    """Handing CRFBlock.forward the mask BasicCRFLayer builds gives bit-identical results to passing None (closed form);
    a different mask changes the result; an unshifted block ignores the argument, as the reference does."""
    pkg = _pkg()
    torch.manual_seed(3)
    H, W, C, nH = 15, 20, 64, 2
    x = torch.randn(2, H * W, C, device=DEV)
    v = torch.randn(2, H, W, C, device=DEV)
    std = torch.from_numpy(O.shift_mask(H, W, 7, 3)).to(DEV)
    blk = pkg.CRFBlock(C, nH, C, shift_size=3).to(DEV)
    blk.H, blk.W = H, W
    with torch.no_grad():
        y_none, y_std = blk(x, v, None), blk(x, v, std)
        y_other = blk(x, v, torch.zeros_like(std))
    assert torch.equal(y_none, y_std)
    assert not torch.equal(y_none, y_other)
    blk0 = pkg.CRFBlock(C, nH, C, shift_size=0).to(DEV)
    blk0.H, blk0.W = H, W
    with torch.no_grad():
        assert torch.equal(blk0(x, v, None), blk0(x, v, torch.full_like(std, -3.0)))


@pytest.mark.parametrize("shift", [0, 3])
@pytest.mark.parametrize("strided", [False, True])
def test_config1_block_vs_oracle_cpu(shift, strided):
    """BASELINE.json configs[0]: one CRFBlock fwd+bwd, window 7, C=128, 4 heads, 60x80 (1/4 of 240x320), batch 2."""
    _run_block_vs_oracle(2, 60, 80, 128, 4, shift, seed=10 + shift, strided=strided, oracle_device="cpu")


@pytest.mark.parametrize("H,W,C,nH", [(120, 160, 128, 4), (60, 80, 256, 8), (30, 40, 512, 16), (15, 20, 1024, 32)])
@pytest.mark.parametrize("shift", [0, 3])
def test_config2_stage_shapes_vs_oracle(H, W, C, nH, shift):
    """The four decoder scales of configs[1] (480x640, batch 8).  The oracle is evaluated with torch on the GPU here
    only because the fp32 CPU run of the 1/4 scale takes minutes; it is the same oracle code."""
    _run_block_vs_oracle(8, H, W, C, nH, shift, seed=100 + C + shift, strided=True, oracle_device=DEV)


@pytest.mark.parametrize("H,W,C,nH,shift", [(9, 10, 64, 4, 3), (30, 40, 128, 8, 0), (15, 20, 256, 16, 3), (30, 40, 512, 32, 3)])
def test_head_dim_16_block_vs_oracle(H, W, C, nH, shift):
    """BASELINE.json configs[2] sweeps heads 4-32 at embed 64-512: the head_dim = 16 points (the attention tiles stay
    32 wide, the upper half zero-filled)."""
    _run_block_vs_oracle(2, H, W, C, nH, shift, seed=300 + C + shift, strided=True, oracle_device=DEV)


@pytest.mark.parametrize("H,W,C,nH,shift", [(9, 10, 64, 1, 3), (30, 40, 128, 2, 0), (15, 20, 256, 4, 3), (15, 20, 256, 2, 0),
                                            (30, 40, 512, 8, 3), (16, 23, 512, 4, 3)])
def test_wide_head_block_vs_oracle(H, W, C, nH, shift):
    """BASELINE.json configs[2], the head_dim = 64 and 128 points (crf_attn_wide.cu: 32-wide slices of a head)."""
    _run_block_vs_oracle(2, H, W, C, nH, shift, seed=400 + C + shift, strided=True, oracle_device=DEV)


# Every width the library accepts that is not a power of two.  The width picks the GEMM kernel of each projection (the
# CTA-pair kernel needs N % 256 == 0, the persistent one N % 128 == 0, else gemm_kernel<64> with C / 64 column tiles),
# the LayerNorm row-kernel instance (C / 64 channel groups) and, with the head width, the head count.
_ODD_WIDTHS = [192, 320, 384, 448, 576, 640, 704, 768, 832, 896, 960]
_WIDTH_CASES = ([(C, 32, p, 2, 15, 20, 3) for C in _ODD_WIDTHS for p in ("bf16", "fp32")]
                # head widths other than 32 at these widths: odd head counts of 3 ... 15
                + [(C, hd, p, 2, 15, 20, 3) for C, hd in [(192, 64), (320, 64), (960, 64), (384, 128), (640, 128),
                                                          (896, 128), (448, 16)] for p in ("bf16", "fp32")]
                # T = 9600: the CTA-pair GEMMs run several tiles per pair
                + [(C, 32, "bf16", 8, 30, 40, 0) for C in (576, 768, 960)])


@pytest.mark.parametrize("C,hd,precision,B,H,W,shift", _WIDTH_CASES)
def test_channel_widths_vs_oracle(C, hd, precision, B, H, W, shift):
    """One block, forward and backward, at a channel width that is not a power of two, against the fp32 oracle: y, dx,
    dv, all 13 parameter gradients and the per-token-row error, in both precision modes."""
    _run_block_vs_oracle(B, H, W, C, C // hd, shift, seed=800 + C + hd, strided=True, oracle_device=DEV,
                         precision=precision, tol=TOL_FP32 if precision == "fp32" else TOL)


def test_inference_path_matches_training_path():
    pkg = _pkg()
    torch.manual_seed(0)
    layer = pkg.BasicCRFLayer(dim=128, depth=2, num_heads=4, v_dim=128).to(DEV)
    x = torch.randn(2, 128, 30, 40, device=DEV).flatten(2).transpose(1, 2)
    v = torch.randn(2, 128, 30, 40, device=DEV).permute(0, 2, 3, 1)
    with torch.no_grad():
        y0 = layer(x, v, 30, 40)[0]
    y1 = layer(x.clone().requires_grad_(True), v, 30, 40)[0]
    torch.cuda.synchronize()
    assert torch.equal(y0, y1.detach())


def test_bf16_inputs_and_autocast_like_usage():
    """Under bf16 autocast the conv projections hand over bf16 NCHW views; output stays fp32 (residual stream)."""
    pkg = _pkg()
    torch.manual_seed(1)
    layer = pkg.BasicCRFLayer(dim=64, depth=2, num_heads=2, v_dim=64).to(DEV)
    xb = torch.randn(2, 64, 15, 20, device=DEV).to(torch.bfloat16)
    vb = torch.randn(2, 64, 15, 20, device=DEV).to(torch.bfloat16)
    x = xb.flatten(2).transpose(1, 2).requires_grad_(True)
    v = vb.permute(0, 2, 3, 1).requires_grad_(True)
    y = layer(x, v, 15, 20)[0]
    assert y.dtype == torch.float32
    y.square().mean().backward()
    blocks = [{k: p.detach().float().cpu() for k, p in blk.state_dict().items()
               if not k.endswith("relative_position_index")} for blk in layer.blocks]
    yo = O.basic_crf_layer(xb.float().cpu().flatten(2).transpose(1, 2), vb.float().cpu().permute(0, 2, 3, 1), 15, 20,
                           blocks, 2)
    assert rel_l2(y.detach(), yo) < TOL
    assert x.grad.dtype == torch.bfloat16 and torch.isfinite(x.grad.float()).all()


def test_reference_error_behaviour():
    pkg = _pkg()
    blk = pkg.CRFBlock(64, 2, 64).to(DEV)
    blk.H, blk.W = 5, 5
    with pytest.raises(AssertionError, match="input feature has wrong size"):
        blk(torch.randn(1, 24, 64, device=DEV), torch.randn(1, 5, 5, 64, device=DEV), None)
    with pytest.raises(AssertionError, match="self.dim != v.shape"):
        blk(torch.randn(1, 25, 64, device=DEV), torch.randn(1, 5, 5, 32, device=DEV), None)
    with pytest.raises(AssertionError, match="shift_size must in 0-window_size"):
        pkg.CRFBlock(64, 2, 64, window_size=7, shift_size=7)


def test_full_model_dropin_matches_oracle_model():
    """SURVEY.md section 4 item 4: one state_dict, the oracle's full model on CPU (fp32) vs the product model on the GPU
    (fp32 everywhere except the CRF blocks' bf16 tensor-core operands)."""
    from monocular_depth_estimation_b200.model import PTModel
    from oracle.model_oracle import OraclePTModel
    torch.manual_seed(3)
    ref = OraclePTModel().eval()
    ours = PTModel().eval()
    ours.load_state_dict(ref.state_dict(), strict=True)
    ours = ours.to(DEV)
    img = torch.rand(1, 3, 224, 288)
    with torch.no_grad():
        yo = ref(img)
        yc = ours(img.to(DEV))
    torch.cuda.synchronize()
    assert yc.shape == yo.shape == (1, 1, 224, 288)
    err = rel_l2(yc, yo)
    _report("full model 224x288", {"depth": err})
    assert err < TOL, err


def test_full_model_matches_reference_model_golden():
    """The product model against the UNMODIFIED reference model's own numbers (tests/golden/model_64x96.npz: name-seeded
    weights, eval mode): depth map, loss, image gradient, parameter gradients across encoder, bridge, stages and head."""
    from monocular_depth_estimation_b200 import training as TR
    from monocular_depth_estimation_b200.model import PTModel
    from tests.helpers import MODEL_GRAD_KEYS, fill_by_name
    g = load_golden("model_64x96")
    model = fill_by_name(PTModel()).eval().to(DEV)
    image = torch.from_numpy(g["image"]).to(DEV).requires_grad_(True)
    pred = model(image)
    loss = TR.depth_loss(pred, TR.depth_norm(torch.from_numpy(g["depth"]).to(DEV)))
    loss.backward()
    torch.cuda.synchronize()
    params = dict(model.named_parameters())
    errs = {"pred": rel_l2(pred.detach(), g["pred"]), "dimage": rel_l2(image.grad, g["dimage"]),
            "loss": abs(float(loss.detach()) - float(g["loss"][0])) / float(g["loss"][0])}
    for k in MODEL_GRAD_KEYS:
        errs[k] = rel_l2(params[k].grad, g["grad." + k])
    _report("full model vs reference golden 64x96", errs)
    # depth / loss: the block tolerance (2e-2).  Gradients cross all eight bf16 blocks in both directions and, for the
    # image and the first convolution, the whole encoder backward, which amplifies them (measured on a B200, round 2:
    # dimage 5.7e-2, features.0.0.weight 4.5e-2, everything inside the decoder <= 1.3e-2).  The bound per quantity is
    # the reference's OWN bf16 deviation: the unmodified reference model under torch's bf16 autocast against its fp32
    # run (`bf16ref.*` in the fixture, written by tests/golden/make_golden.py; dimage 0.19, features.0.0.weight 0.12,
    # decoder parameters 3e-3 ... 3.5e-2) -- the product's bf16-I/O path has to be at least as close to the fp32
    # reference as the reference's own bf16 arithmetic is, on every stored quantity.
    def bound(k):
        return TOL if k in ("pred", "loss") else float(g["bf16ref." + k][0])
    bad = {k: (e, bound(k)) for k, e in errs.items() if not e < bound(k)}
    assert not bad, f"{bad}\nall: {errs}"


def test_config5_highres_inference_vs_oracle():
    """BASELINE.json configs[4]: 960x1280 inference, batch 16 -> scale 1/4 is 240x320 (245x322 padded, 25 760
    windows per block).  Forward only, no saved tensors; oracle evaluated with torch on the GPU (same oracle code)."""
    pkg = _pkg()
    torch.manual_seed(5)
    B, H, W, C, nH = 16, 240, 320, 128, 4
    layer = pkg.BasicCRFLayer(dim=C, depth=2, num_heads=nH, v_dim=C).to(DEV)
    x = torch.randn(B, C, H, W, device=DEV).flatten(2).transpose(1, 2)
    v = torch.randn(B, C, H, W, device=DEV).permute(0, 2, 3, 1)
    with torch.no_grad():
        y = layer(x, v, H, W)[0]
        blocks = [{k: p.detach() for k, p in blk.named_parameters()} for blk in layer.blocks]
        yo = torch.cat([O.basic_crf_layer(x[i:i + 4], v[i:i + 4], H, W, blocks, nH) for i in range(0, B, 4)])
    torch.cuda.synchronize()
    err, row = rel_l2(y, yo), _row_err(y, yo)
    _report("config5 B16 240x320 C128 inference", {"y": err, "y_row_max": row})
    assert err < TOL_Y and row < TOL_ROW, (err, row)


@pytest.mark.parametrize("H,W,C,nH", [(120, 160, 256, 8), (60, 80, 512, 16), (30, 40, 1024, 32)])
def test_config5_other_scales_inference_vs_oracle(H, W, C, nH):
    """configs[4] at the other three decoder scales (960x1280, batch 16: 6 624 / 1 728 / 480 windows per block)."""
    pkg = _pkg()
    torch.manual_seed(50 + C)
    B = 16
    layer = pkg.BasicCRFLayer(dim=C, depth=2, num_heads=nH, v_dim=C).to(DEV)
    x = torch.randn(B, C, H, W, device=DEV).flatten(2).transpose(1, 2)
    v = torch.randn(B, C, H, W, device=DEV).permute(0, 2, 3, 1)
    with torch.no_grad():
        y = layer(x, v, H, W)[0]
        blocks = [{k: p.detach() for k, p in blk.named_parameters()} for blk in layer.blocks]
        yo = torch.cat([O.basic_crf_layer(x[i:i + 4], v[i:i + 4], H, W, blocks, nH) for i in range(0, B, 4)])
    torch.cuda.synchronize()
    err, row = rel_l2(y, yo), _row_err(y, yo)
    _report(f"config5 B16 {H}x{W} C{C} inference", {"y": err, "y_row_max": row})
    assert err < TOL_Y and row < TOL_ROW, (err, row)


def test_config5_whole_model_960x1280_vs_oracle_model():
    """configs[4] through the WHOLE model (MobileNetV3-large encoder + all four decoder stages + head) at 960x1280:
    the product model (eval, fp32 encoder / convs, CRF blocks on the library) against the oracle's restatement of the
    reference model with the same state_dict, both on the GPU in fp32 (batch 2: the oracle materialises the 49 x 49
    attention tensors)."""
    from monocular_depth_estimation_b200.model import PTModel
    from oracle.model_oracle import OraclePTModel
    from tests.helpers import fill_by_name
    conv_tf32, mm_tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False   # fp32 oracle, fp32 encoder
    try:
        ref = fill_by_name(OraclePTModel()).eval().to(DEV)
        ours = fill_by_name(PTModel()).eval().to(DEV)
        gen = torch.Generator().manual_seed(9)
        img = torch.rand(2, 3, 960, 1280, generator=gen).to(DEV)
        with torch.no_grad():
            yo = ref(img)
            yc = ours(img)
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = conv_tf32, mm_tf32
    assert yc.shape == yo.shape == (2, 1, 960, 1280)
    err = rel_l2(yc, yo)
    _report("config5 whole model 960x1280 B2", {"depth": err})
    assert err < TOL, err


def test_batch_permutation_equivariance_is_bit_exact():
    """Size-independent property at the full config-2 shape: windows never cross images, so permuting the images of
    the batch must permute outputs and input gradients bit-exactly (different CTAs / tiles, same arithmetic)."""
    pkg = _pkg()
    torch.manual_seed(6)
    B, H, W, C, nH = 8, 120, 160, 128, 4
    layer = pkg.BasicCRFLayer(dim=C, depth=2, num_heads=nH, v_dim=C).to(DEV)
    x = torch.randn(B, C, H, W, device=DEV)
    v = torch.randn(B, C, H, W, device=DEV)
    perm = torch.tensor([3, 0, 7, 1, 6, 2, 5, 4], device=DEV)

    def run(xi, vi):
        xt = xi.flatten(2).transpose(1, 2).detach().requires_grad_(True)
        vt = vi.permute(0, 2, 3, 1).detach().requires_grad_(True)
        y = layer(xt, vt, H, W)[0]
        y.square().sum().backward()
        return y.detach(), xt.grad, vt.grad

    y0, dx0, dv0 = run(x, v)
    y1, dx1, dv1 = run(x[perm].contiguous(), v[perm].contiguous())
    torch.cuda.synchronize()
    assert torch.equal(y0[perm], y1)
    assert torch.equal(dx0[perm], dx1)
    assert torch.equal(dv0[perm], dv1)


@pytest.mark.parametrize("with_mask", [False, True])
def test_window_attention_standalone_matches_oracle(with_mask):
    """WindowAttention.forward(x, v, mask) on pre-partitioned windows (newcrf_layers.py:110-149), incl. an arbitrary
    additive mask indexed by window-within-image."""
    pkg = _pkg()
    torch.manual_seed(11)
    C, nH, nW, B = 128, 4, 6, 3
    wa = pkg.WindowAttention(C, (7, 7), nH, C).to(DEV)
    with torch.no_grad():
        wa.relative_position_bias_table.normal_(0, 0.3)
        wa.qk.bias.normal_(0, 0.2)
    x = torch.randn(B * nW, 49, C, device=DEV, requires_grad=True)
    v = torch.randn(B * nW, 49, C, device=DEV, requires_grad=True)
    mask = None
    if with_mask:
        mask = torch.where(torch.rand(nW, 49, 49, device=DEV) < 0.3, -100.0, 0.0)
        mask[:, torch.arange(49), torch.arange(49)] = 0.0
    dy = torch.randn(B * nW, 49, C, device=DEV)
    y = wa(x, v, mask)
    y.backward(dy)
    p = {"attn." + k: t.detach().clone().requires_grad_(True) for k, t in wa.named_parameters()}
    xo, vo = x.detach().clone().requires_grad_(True), v.detach().clone().requires_grad_(True)
    yo = O.window_attention(xo, vo, p, nH, mask)
    yo.backward(dy)
    torch.cuda.synchronize()
    errs = {"y": rel_l2(y.detach(), yo.detach()), "dx": rel_l2(x.grad, xo.grad), "dv": rel_l2(v.grad, vo.grad)}
    for k, t in wa.named_parameters():
        errs[k] = rel_l2(t.grad, p["attn." + k].grad)
    _report(f"window_attention standalone mask={with_mask}", errs)
    bad = {k: e for k, e in errs.items() if not e < TOL}
    assert not bad, f"{bad}\nall: {errs}"


@pytest.mark.parametrize("C,nH", [(64, 2), (128, 4), (256, 8)])
@pytest.mark.parametrize("B,H,W", [(1, 1, 1), (1, 3, 5), (1, 7, 7), (3, 8, 13), (2, 6, 50), (5, 14, 7), (1, 20, 29)])
def test_ragged_geometries_vs_oracle(B, H, W, C, nH):
    """Edge geometries: maps smaller than one window (all-pad windows but one), exact multiples of 7 (no padding),
    odd numbers of windows (the last window pair is half empty), token counts that are not multiples of the 128-row
    GEMM tile (nor of the 8-row granularity of the balanced tiles).  Two blocks (shift 0 and 3), fwd + bwd, vs the fp32
    oracle.  C = 64 runs the unfused kernels, C = 128 / 256 the fused MLP forward and the fused d.LN' kernels."""
    pkg = _pkg()
    torch.manual_seed(B * 1000 + H * 31 + W)
    layer = pkg.BasicCRFLayer(dim=C, depth=2, num_heads=nH, v_dim=C).to(DEV)
    with torch.no_grad():
        for p in layer.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    x = torch.randn(B, C, H, W, device=DEV).flatten(2).transpose(1, 2).requires_grad_(True)
    v = torch.randn(B, C, H, W, device=DEV).permute(0, 2, 3, 1).requires_grad_(True)
    dy = torch.randn(B, H * W, C, device=DEV)
    y = layer(x, v, H, W)[0]
    y.backward(dy)
    blocks = [{k: p.detach().clone().requires_grad_(True) for k, p in blk.named_parameters()} for blk in layer.blocks]
    xo, vo = x.detach().clone().requires_grad_(True), v.detach().clone().requires_grad_(True)
    yo = O.basic_crf_layer(xo, vo, H, W, blocks, nH)
    yo.backward(dy)
    torch.cuda.synchronize()
    errs = {"y": rel_l2(y.detach(), yo.detach()), "dx": rel_l2(x.grad, xo.grad), "dv": rel_l2(v.grad, vo.grad)}
    for i, blk in enumerate(layer.blocks):
        for k, p in blk.named_parameters():
            errs[f"{i}.{k}"] = rel_l2(p.grad, blocks[i][k].grad)
    _report(f"ragged B{B} {H}x{W} C{C}", errs)
    bad = {k: e for k, e in errs.items() if not e < TOL}
    assert not bad, f"{bad}\nall: {errs}"


def test_c_api_rejects_bad_arguments():
    """Error behaviour of the C ABI itself: non-zero return + message, no crash, no kernel launch."""
    import ctypes as C
    from monocular_depth_estimation_b200 import _lib, ops
    lib = _lib.lib()
    d = ops.make_desc(1, 7, 7, 64, 2, 0, device=0)
    assert lib.crf_block_fwd(C.byref(d), None, None, None, None, None, None, 0, None) != 0
    assert b"null pointer" in lib.crf_last_error()
    d.num_heads = 8  # head_dim 8: not a supported head width
    s = C.c_size_t()
    assert lib.crf_block_sizes(C.byref(d), C.byref(s), None, None) != 0
    assert b"head_dim must be 16, 32, 64 or 128" in lib.crf_last_error()
    a = _lib.GemmArgs()
    x = torch.zeros(128, 64, dtype=torch.bfloat16, device=DEV)
    a.A, a.B, a.out0 = x.data_ptr(), x.data_ptr(), x.data_ptr()
    a.M, a.N, a.K, a.ld_out = 128, 96, 64, 96   # N not a multiple of 64
    assert lib.crf_gemm(C.byref(a), None) != 0
    assert b"multiple of 64" in lib.crf_last_error()
