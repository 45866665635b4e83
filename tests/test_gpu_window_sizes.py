"""Window sizes 2..8 on the GPU: the CRF block, the layer call, the stand-alone WindowAttention and the whole model at
every window the kernels implement, against the fp32 oracle, in both precision tiers.

Tolerances are those of tests/test_gpu_block.py: bf16 tier y 6e-3, dx / dv 1.5e-2, parameter gradients 2e-2 and 2e-2
per token row; fp32 tier 1.5e-4 (1e-3 per row).  Window 7 runs as the control.  A bf16-tier parameter gradient above
its bound is held instead to the reference's own bf16 deviation on the same inputs (as the whole-model golden test
does); y, dx, dv and the per-row bounds are never relaxed.
"""
import pytest
import torch

from oracle import crf_oracle as O
from tests.helpers import rel_l2
from tests.test_gpu_block import TOL, TOL_FP32, TOL_ROW, _report, _row_err, _tol

pytestmark = pytest.mark.gpu
DEV = "cuda"
WINDOWS = [2, 3, 4, 5, 6, 7, 8]


def _block_case(ws, shift, B, H, W, C, nH, precision, seed, mask=None):
    """One CRFBlock forward + backward (functional.crf_block: the C ABI block call) against the oracle on the GPU."""
    from monocular_depth_estimation_b200 import functional as CF
    gen = torch.Generator().manual_seed(seed)
    p = O.init_block_params(C, nH, gen, ws=ws)
    x = torch.randn(B, C, H, W, generator=gen).flatten(2).transpose(1, 2)   # NCHW views, as the decoder hands them
    v = torch.randn(B, C, H, W, generator=gen).permute(0, 2, 3, 1)
    dy = torch.randn(B, H * W, C, generator=gen)
    po = {k: t.detach().clone().to(DEV).requires_grad_(True) for k, t in p.items()}
    xo = x.to(DEV).detach().requires_grad_(True)
    vo = v.to(DEV).detach().requires_grad_(True)
    yo = O.crf_block(xo, vo, H, W, po, nH, ws, shift, mask_matrix=mask)
    yo.backward(dy.to(DEV))
    pc = {k: t.detach().clone().to(DEV).requires_grad_(True) for k, t in p.items()}
    xc = x.to(DEV).detach().requires_grad_(True)
    vc = v.to(DEV).detach().requires_grad_(True)
    yc = CF.crf_block(xc, vc, H, W, [pc[k] for k in CF.PARAM_KEYS], nH, window=ws, shift=shift, precision=precision,
                      mask=None if mask is None else mask.to(DEV))
    yc.backward(dy.to(DEV))
    torch.cuda.synchronize()
    errs = {"y": rel_l2(yc.detach(), yo.detach()), "dx": rel_l2(xc.grad, xo.grad), "dv": rel_l2(vc.grad, vo.grad)}
    for k in CF.PARAM_KEYS:
        errs[k] = rel_l2(pc[k].grad, po[k].grad)
    _report(f"ws{ws} block B{B} {H}x{W} C{C} nH{nH} shift{shift} {precision}" + (" custom-mask" if mask is not None else ""),
            errs)
    fp32 = precision == "fp32"
    bad = {k: e for k, e in errs.items() if not e < (TOL_FP32 if fp32 else _tol(k))}
    if bad and not fp32 and set(bad) <= set(CF.PARAM_KEYS):
        # A parameter gradient above the bf16-tier bound is held to the reference's OWN bf16 deviation on the same
        # inputs instead (the oracle under bf16 autocast against its fp32 run), as the whole-model golden test does.
        # This happens on maps of one real token per image: its attention gradient is a handful of entries, mostly
        # cancelling in dS = P (dP - sum P dP), and bf16 operands move them by several percent in any implementation.
        own = _oracle_bf16_deviation(p, x, v, dy, H, W, nH, ws, shift, mask)
        errs_bound = {k: max(_tol(k), own[k]) for k in bad}
        _report(f"ws{ws} block B{B} {H}x{W} C{C} nH{nH} shift{shift} bf16: reference bf16 deviation", own)
        bad = {k: (e, errs_bound[k]) for k, e in bad.items() if not e < errs_bound[k]}
    assert not bad, f"rel_l2 above the bound: {bad}\nall: {errs}"
    rows = {"y": _row_err(yc, yo), "dx": _row_err(xc.grad, xo.grad), "dv": _row_err(vc.grad, vo.grad)}
    row_tol = 1e-3 if fp32 else TOL_ROW
    assert all(e < row_tol for e in rows.values()), f"per-token-row error above {row_tol}: {rows}"


def _oracle_bf16_deviation(p, x, v, dy, H, W, nH, ws, shift, mask):
    """rel_l2 of every parameter gradient of the oracle evaluated under CPU bf16 autocast against its fp32 run."""
    grads = []
    for bf16 in (False, True):
        po = {k: t.detach().clone().requires_grad_(True) for k, t in p.items()}
        with torch.autocast("cpu", dtype=torch.bfloat16, enabled=bf16):
            yo = O.crf_block(x.detach(), v.detach(), H, W, po, nH, ws, shift, mask_matrix=mask)
        yo.float().backward(dy)
        grads.append({k: t.grad for k, t in po.items()})
    return {k: rel_l2(grads[1][k], grads[0][k]) for k in p}


def _geometries(ws):
    """(B, H, W): an exact multiple of the window, a 1 x 1 map, a map smaller than one window, a ragged map, and an odd
    number of windows in the batch (the last window pair has a dead half)."""
    return [(2, 2 * ws, 3 * ws), (2, 1, 1), (2, max(ws - 1, 1), max(ws - 1, 1)), (2, 2 * ws + 1, 3 * ws - 2),
            (1, ws, 3 * ws)]


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("hd", [32, 16])
@pytest.mark.parametrize("shifted", [False, True])
@pytest.mark.parametrize("ws", WINDOWS)
def test_block_vs_oracle_small_maps(ws, shifted, hd, precision):
    C = 64
    for i, (B, H, W) in enumerate(_geometries(ws)):
        _block_case(ws, ws // 2 if shifted else 0, B, H, W, C, C // hd, precision, seed=1000 * ws + 10 * i + hd)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("hd", [32, 16])
@pytest.mark.parametrize("shifted", [False, True])
@pytest.mark.parametrize("ws", WINDOWS)
def test_block_vs_oracle_60x80_c128(ws, shifted, hd, precision):
    """The 1/4 scale of BASELINE.json configs[0] (240 x 320 input) at every window."""
    _block_case(ws, ws // 2 if shifted else 0, 2, 60, 80, 128, 128 // hd, precision, seed=2000 * ws + hd)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("ws", [2, 4, 5, 8])
def test_block_vs_oracle_head_dim_64(ws, precision):
    """head_dim 64 (crf_attn_wide.cu) on a ragged map, both shifts."""
    for shift in (0, ws // 2):
        _block_case(ws, shift, 2, 2 * ws + 1, 3 * ws - 2, 128, 2, precision, seed=3000 * ws + shift)


@pytest.mark.parametrize("ws", [5, 8])
def test_layer_call_with_norm_and_pixel_shuffle_equals_block_by_block(ws):
    """crf_layer_fwd / _bwd (both blocks, the closing LayerNorm, PixelShuffle(2) folded into its store) against the
    same layer run block by block + the stand-alone LayerNorm + F.pixel_shuffle: same kernels, same fp32 order."""
    import monocular_depth_estimation_b200 as pkg
    from monocular_depth_estimation_b200 import functional as CF
    torch.manual_seed(40 + ws)
    B, H, W, C, nH = 2, 2 * ws + 3, 3 * ws + 1, 128, 4
    layer = pkg.BasicCRFLayer(dim=C, depth=2, num_heads=nH, v_dim=C, window_size=ws).to(DEV)
    norm = torch.nn.LayerNorm(C).to(DEV)
    with torch.no_grad():
        for blk in layer.blocks:
            blk.attn.relative_position_bias_table.normal_(0, 0.3)
        norm.weight.normal_(1.0, 0.2)
        norm.bias.normal_(0.0, 0.2)
    x0 = torch.randn(B, C, H, W, device=DEV).flatten(2).transpose(1, 2)
    v0 = torch.randn(B, C, H, W, device=DEV).permute(0, 2, 3, 1)
    gy = torch.randn(B, C // 4, 2 * H, 2 * W, device=DEV)

    def run(fused):
        for p_ in list(layer.parameters()) + list(norm.parameters()):
            p_.grad = None
        x, v = x0.detach().requires_grad_(True), v0.detach().requires_grad_(True)
        if fused:
            y = layer.run(x, v, H, W, norm=norm, pixel_shuffle=True)
        else:
            vb = CF.convert_v(v)
            y = x
            for blk in layer.blocks:
                blk.H, blk.W = H, W
                y = blk(y, v, None, v_bf16=vb)
            y = CF.layer_norm(y, norm.weight, norm.bias, norm.eps)
            y = torch.nn.functional.pixel_shuffle(y.view(B, H, W, C).permute(0, 3, 1, 2), 2)
        assert y.shape == (B, C // 4, 2 * H, 2 * W)
        y.backward(gy)
        grads = {k: p_.grad.clone() for k, p_ in layer.named_parameters()}
        grads.update({"norm." + k: p_.grad.clone() for k, p_ in norm.named_parameters()})
        return y.detach(), x.grad.clone(), v.grad.clone(), grads

    yf, dxf, dvf, gf = run(True)
    yb, dxb, dvb, gb = run(False)
    assert torch.equal(yf, yb), "forward differs"
    assert rel_l2(dxf, dxb) < 1e-6 and rel_l2(dvf, dvb) < 1e-6, (rel_l2(dxf, dxb), rel_l2(dvf, dvb))
    bad = {k: rel_l2(gf[k], gb[k]) for k in gb if not rel_l2(gf[k], gb[k]) < 1e-5}
    assert not bad, bad
    # and the layer against the oracle (closing norm, then the shuffle)
    blocks = [{k: p_.detach() for k, p_ in blk.named_parameters()} for blk in layer.blocks]
    yo = O.basic_crf_layer(x0, v0, H, W, blocks, nH, ws)
    yo = torch.nn.functional.layer_norm(yo, (C,), norm.weight.detach(), norm.bias.detach(), norm.eps)
    yo = torch.nn.functional.pixel_shuffle(yo.view(B, H, W, C).permute(0, 3, 1, 2), 2)
    assert rel_l2(yf, yo) < TOL, rel_l2(yf, yo)


@pytest.mark.parametrize("with_mask", [False, True])
@pytest.mark.parametrize("ws", [4, 8])
def test_window_attention_standalone(ws, with_mask):
    """WindowAttention.forward(x, v, mask) on pre-partitioned (nW*B, ws*ws, C) windows, with an arbitrary additive mask."""
    import monocular_depth_estimation_b200 as pkg
    torch.manual_seed(11 + ws)
    C, nH, nW, B, N = 128, 4, 6, 3, ws * ws
    wa = pkg.WindowAttention(C, (ws, ws), nH, C).to(DEV)
    with torch.no_grad():
        wa.relative_position_bias_table.normal_(0, 0.3)
        wa.qk.bias.normal_(0, 0.2)
    x = torch.randn(B * nW, N, C, device=DEV, requires_grad=True)
    v = torch.randn(B * nW, N, C, device=DEV, requires_grad=True)
    mask = None
    if with_mask:
        mask = torch.where(torch.rand(nW, N, N, device=DEV) < 0.3, -100.0, 0.0) + 0.5 * torch.randn(nW, N, N, device=DEV)
        mask[:, torch.arange(N), torch.arange(N)] = 0.0
    dy = torch.randn(B * nW, N, C, device=DEV)
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
    _report(f"ws{ws} window_attention standalone mask={with_mask}", errs)
    bad = {k: e for k, e in errs.items() if not e < TOL}
    assert not bad, f"{bad}\nall: {errs}"


def test_window_attention_rejects_unsupported_windows():
    import monocular_depth_estimation_b200 as pkg
    wa = pkg.WindowAttention(64, (3, 3), 2, 64).to(DEV)
    for N in (1, 50, 81):
        x = torch.randn(2, N, 64, device=DEV)
        with pytest.raises(AssertionError, match="ws in 2..8"):
            wa(x, x)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_custom_mask_matrix_at_window_8(precision):
    """A non-standard mask_matrix (nW, 64, 64) is honoured at window 8, in both tiers."""
    ws, H, W = 8, 17, 20
    gen = torch.Generator().manual_seed(88)
    nW = (-(-H // ws)) * (-(-W // ws))
    mask = torch.where(torch.rand(nW, 64, 64, generator=gen) < 0.3, -100.0, 0.0) + 0.5 * torch.randn(nW, 64, 64, generator=gen)
    _block_case(ws, 4, 2, H, W, 128, 4, precision, seed=808, mask=mask)


def test_block_module_recognises_the_standard_mask_at_window_8():
    """CRFBlock.forward given the mask BasicCRFLayer builds == None (closed form), bit for bit; another mask differs."""
    import monocular_depth_estimation_b200 as pkg
    torch.manual_seed(3)
    H, W, C, nH = 17, 20, 64, 2
    x = torch.randn(2, H * W, C, device=DEV)
    v = torch.randn(2, H, W, C, device=DEV)
    std = torch.from_numpy(O.shift_mask(H, W, 8, 4)).to(DEV)
    blk = pkg.CRFBlock(C, nH, C, window_size=8, shift_size=4).to(DEV)
    blk.H, blk.W = H, W
    with torch.no_grad():
        y_none, y_std = blk(x, v, None), blk(x, v, std)
        y_other = blk(x, v, torch.zeros_like(std))
    assert torch.equal(y_none, y_std)
    assert not torch.equal(y_none, y_other)


def _oracle_model_with_window(ws):
    """oracle.model_oracle.OraclePTModel with every decoder stage rebuilt for window `ws` (the oracle's stages take the
    window as an argument; its decoder builds them at the reference's default 7)."""
    from oracle import model_oracle as MO
    ref = MO.OraclePTModel()
    dec = ref.Unet[1]
    for s in range(4):
        crf = getattr(dec, f"crf{s}")
        crf.window_size = ws
        crf.crf_layer.blocks = torch.nn.ModuleList([MO._block_holder(crf.embed_dim, crf.num_heads, ws) for _ in range(2)])
    return ref


@pytest.mark.parametrize("ws", [5, 8])
def test_whole_model_with_decoder_window(ws):
    """PTModel with Decoder(window_size=ws) against the oracle's model on a 64 x 96 image with one state_dict (fp32
    everywhere except the CRF blocks' bf16 tensor-core operands): depth map within the whole-model bound (2e-2)."""
    from monocular_depth_estimation_b200.model import Decoder, PTModel
    from tests.helpers import fill_by_name
    torch.manual_seed(20 + ws)
    ref = fill_by_name(_oracle_model_with_window(ws)).eval()
    ours = PTModel()
    ours.Unet[1] = Decoder(window_size=ws)
    ours.eval()
    ours.load_state_dict(ref.state_dict(), strict=True)
    conv_tf32, mm_tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref, ours = ref.to(DEV), ours.to(DEV)
        img = torch.rand(2, 3, 64, 96, generator=torch.Generator().manual_seed(ws)).to(DEV)
        with torch.no_grad():
            yo = ref(img)
            yc = ours(img)
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = conv_tf32, mm_tf32
    assert yc.shape == yo.shape == (2, 1, 64, 96)
    err = rel_l2(yc, yo)
    _report(f"ws{ws} whole model 64x96", {"depth": err})
    assert err < TOL, err


def test_window_8_attention_is_deterministic():
    """Two runs of the window-8 attention core on the same inputs give bit-identical outputs and gradients (run once)."""
    from monocular_depth_estimation_b200 import ops
    torch.manual_seed(8)
    B, H, W, C, nH, ws = 2, 30, 40, 128, 4, 8
    T = B * H * W
    qk = (torch.randn(T, 2 * C, device=DEV) * 0.5).to(torch.bfloat16)
    vb = torch.randn(T, C, device=DEV).to(torch.bfloat16)
    qkb = 0.1 * torch.randn(2 * C, device=DEV)
    tab = 0.3 * torch.randn((2 * ws - 1) ** 2, nH, device=DEV)
    dout = torch.randn(T, C, device=DEV).to(torch.bfloat16)
    outs = []
    for _ in range(2):
        desc = ops.make_desc(B, H, W, C, nH, ws // 2, window=ws, device=0)
        o, lse = ops.attn_fwd(desc, qk, vb, qkb, 0.17, tab, want_lse=True)
        dqk, dv, dtab, dqkb = ops.attn_bwd(desc, qk, vb, qkb, 0.17, tab, lse, dout)
        torch.cuda.synchronize()
        outs.append((o, lse, dqk, dv))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
