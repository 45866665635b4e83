"""torch.autograd bridge to the C ABI: one C call per CRFBlock forward, one per backward.

`crf_block(x, v, ...)` is the functional form of the reference's CRFBlock.forward
(/root/reference/src/newcrf_layers.py:195-257).  PyTorch is used for device memory (every buffer the library
touches is a torch tensor allocated here), the current CUDA stream and autograd bookkeeping -- nothing else.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from .ops import _precision_code, make_desc

# order of the parameter tensors in every call (matches _lib.PARAM_NAMES / crf_block_params)
PARAM_KEYS = ("norm1.weight", "norm1.bias", "attn.qk.weight", "attn.qk.bias", "attn.relative_position_bias_table",
              "attn.proj.weight", "attn.proj.bias", "norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias",
              "mlp.fc2.weight", "mlp.fc2.bias")


_GUARD = 4096


def _guard_on():
    """CRF_DEBUG_GUARD=1 (tests): every caller-allocated byte buffer gets a patterned tail that must survive the call --
    the library's sub-allocations inside `saved` / workspace are checked for overruns this way."""
    import os
    return os.environ.get("CRF_DEBUG_GUARD", "0") == "1"


def _alloc_bytes(nbytes, device):
    if not _guard_on():
        return torch.empty(nbytes, dtype=torch.uint8, device=device)
    buf = torch.empty(nbytes + _GUARD, dtype=torch.uint8, device=device)
    buf[nbytes:].fill_(0xA5)
    return buf


def _check_guard(buf, nbytes, what):
    if _guard_on() and buf.numel() == nbytes + _GUARD:
        torch.cuda.synchronize(buf.device)
        if not bool((buf[nbytes:] == 0xA5).all()):
            raise RuntimeError(f"{what}: the library wrote past the end of a {nbytes}-byte buffer")


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _param_struct(params, qk_scale, eps, mask=None):
    ps = L.BlockParams()
    for name, t in zip(L.PARAM_NAMES, params):
        setattr(ps, name, t.data_ptr())
    ps.qk_scale = float(qk_scale)
    ps.ln_eps = float(eps)
    if mask is not None:     # a non-standard mask_matrix: replaces the closed-form shift mask inside the kernels
        ps.ext_mask, ps.ext_mask_windows = mask.data_ptr(), mask.shape[0]
    return ps


def _sizes(desc):
    s, f, b = C.c_size_t(), C.c_size_t(), C.c_size_t()
    L.check(L.lib().crf_block_sizes(C.byref(desc), C.byref(s), C.byref(f), C.byref(b)), "crf_block_sizes")
    return s.value, f.value, b.value


def convert_v(v: torch.Tensor) -> torch.Tensor:
    """(B, H, W, C) fp32/bf16 with NCHW-view or contiguous strides -> bf16 (B*H*W, C).  No autograd."""
    from .ops import convert_v as _cv
    return _cv(v.detach())


class _CRFBlockFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, v, vb, mask, precision, H, W, num_heads, window, shift, qk_scale, eps, *params):
        B, Ltok, Cd = x.shape
        dev = x.device
        params = tuple(p.detach().contiguous() for p in params)
        training = any(ctx.needs_input_grad)  # all False under torch.no_grad()
        xd = x.detach()
        if vb is not None and precision == L.PREC_BF16:
            v_arg, desc = vb, make_desc(B, H, W, Cd, num_heads, shift, window=window, training=training,
                                        device=dev.index, x=xd, v_preconverted=1, precision=precision)
        else:
            v_arg = v.detach()
            if v_arg.stride(1) != W * v_arg.stride(2):
                v_arg = v_arg.contiguous()
            desc = make_desc(B, H, W, Cd, num_heads, shift, window=window, training=training, device=dev.index,
                             x=xd, v=v_arg, precision=precision)
        mask = None if mask is None else mask.detach().float().contiguous()
        saved_bytes, _, ws_bwd = _sizes(desc)
        saved = _alloc_bytes(saved_bytes, dev)
        y = torch.empty(B, Ltok, Cd, dtype=torch.float32, device=dev)
        ps = _param_struct(params, qk_scale, eps, mask)
        L.check(L.lib().crf_block_fwd(C.byref(desc), C.byref(ps), xd.data_ptr(), v_arg.data_ptr(), y.data_ptr(),
                                      saved.data_ptr(), None, 0, _stream_ptr(dev)), "crf_block_fwd")
        _check_guard(saved, saved_bytes, "crf_block_fwd saved")
        if training:
            ctx.save_for_backward(xd, v_arg, saved, *params)
            ctx.mask = mask
            ctx.desc = desc
            ctx.scalars = (qk_scale, eps, ws_bwd, H, W)
        return y

    @staticmethod
    def backward(ctx, dy):
        xd, v_arg, saved, *params = ctx.saved_tensors
        qk_scale, eps, ws_bwd, H, W = ctx.scalars
        desc = ctx.desc
        dev = xd.device
        B, Ltok, Cd = xd.shape
        dy = dy.contiguous().float()
        ws = _alloc_bytes(ws_bwd, dev)
        dx = torch.empty(B, Ltok, Cd, dtype=torch.float32, device=dev)
        dv = torch.empty(B, H, W, Cd, dtype=torch.float32, device=dev)
        # one zero-filled buffer, 13 views (256-byte aligned: the kernels store with 16-byte vectors and TMA)
        offs, o = [], 0
        for p in params:
            offs.append(o)
            o += (p.numel() + 63) // 64 * 64
        flat = torch.zeros(o, dtype=torch.float32, device=dev)
        grads = [flat[a:a + p.numel()].view(p.shape) for a, p in zip(offs, params)]
        gs = L.BlockGrads()
        for name, t in zip(L.PARAM_NAMES, grads):
            setattr(gs, name, t.data_ptr())
        ps = _param_struct(params, qk_scale, eps, ctx.mask)
        L.check(L.lib().crf_block_bwd(C.byref(desc), C.byref(ps), xd.data_ptr(), v_arg.data_ptr(), dy.data_ptr(),
                                      saved.data_ptr(), dx.data_ptr(), dv.data_ptr(), 0, C.byref(gs), ws.data_ptr(),
                                      ws_bwd, _stream_ptr(dev)), "crf_block_bwd")
        _check_guard(ws, ws_bwd, "crf_block_bwd workspace")
        return (dx, dv, None, None, None, None, None, None, None, None, None, None, *grads)


def crf_block(x, v, H, W, params, num_heads, *, window=7, shift=0, qk_scale=None, eps=1e-5, v_bf16=None, mask=None,
              precision=None):
    """One CRF block: LN1 -> (shifted-)window attention with q,k from x and v used raw -> +x -> LN2 -> MLP -> +.

    x: (B, H*W, C) fp32/bf16, any strides (the reference hands over a view of NCHW); v: (B, H, W, C);
    params: 13 fp32 tensors in PARAM_KEYS order; v_bf16: optional result of convert_v(v) shared between blocks;
    window: 2..8; mask: None = the shifted-window mask of BasicCRFLayer.forward in closed form, else an additive
    (nW, N, N) mask (N = window^2) that replaces it; precision: "bf16" | "fp32" | None (process default, ops.set_precision).
    Returns (B, H*W, C) fp32.  Mirrors the reference's error behaviour (newcrf_layers.py:205,143,180).
    """
    assert x.dim() == 3 and v.dim() == 4
    B, Ltok, Cd = x.shape
    assert Ltok == H * W, "input feature has wrong size"
    assert Cd == v.shape[-1], "self.dim != v.shape[-1]"
    assert 0 <= shift < window, "shift_size must in 0-window_size"
    if not x.is_cuda:
        raise RuntimeError("monocular_depth_estimation_b200 runs on CUDA (sm_100a) only; there is no CPU path")
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    if v.dtype not in (torch.float32, torch.bfloat16):
        v = v.float()
    if qk_scale is None:
        qk_scale = (Cd // num_heads) ** -0.5
    return _CRFBlockFn.apply(x, v, v_bf16, mask, _precision_code(precision), H, W, num_heads, window, shift,
                             float(qk_scale), float(eps), *params)


class _CRFLayerFn(torch.autograd.Function):
    """BasicCRFLayer.forward (/root/reference/src/newcrf_layers.py:323-363) -- `depth` blocks, shift alternating 0 and
    window // 2, the same v for all -- optionally closed by NewCRF.norm_crf (:430-431): one C call each way
    (crf_layer_fwd / crf_layer_bwd)."""

    @staticmethod
    def forward(ctx, x, v, precision, H, W, num_heads, window, qk_scale, eps, out_bf16, shuffle, depth, norm_w, norm_b,
                *params):
        B, Ltok, Cd = x.shape
        dev = x.device
        params = tuple(p.detach().contiguous() for p in params)
        assert len(params) == 13 * depth
        with_norm = norm_w is not None
        training = any(ctx.needs_input_grad)
        xd, v_arg = x.detach(), v.detach()
        if v_arg.stride(1) != W * v_arg.stride(2):
            v_arg = v_arg.contiguous()
        desc = make_desc(B, H, W, Cd, num_heads, 0, window=window, training=training, device=dev.index, x=xd, v=v_arg,
                         precision=precision)
        sb, wb = C.c_size_t(), C.c_size_t()
        L.check(L.lib().crf_layer_sizes(C.byref(desc), depth, int(with_norm), C.byref(sb), C.byref(wb)),
                "crf_layer_sizes")
        saved = _alloc_bytes(sb.value, dev)
        odt = torch.bfloat16 if out_bf16 else torch.float32
        # shuffle: the closing LayerNorm stores with the decoder's PixelShuffle(2) folded in -> (B, C/4, 2H, 2W), NHWC memory
        y = (torch.empty(B, 2 * H, 2 * W, Cd // 4, dtype=odt, device=dev) if shuffle
             else torch.empty(B, Ltok, Cd, dtype=odt, device=dev))
        pa = (L.BlockParams * depth)()
        for i in range(depth):
            for name, t in zip(L.PARAM_NAMES, params[13 * i:13 * i + 13]):
                setattr(pa[i], name, t.data_ptr())
            pa[i].qk_scale, pa[i].ln_eps = float(qk_scale), float(eps)
        nw = norm_w.detach().contiguous() if with_norm else None
        nb = norm_b.detach().contiguous() if with_norm else None
        la = L.LayerArgs(depth, L.CRF_DT_BF16 if out_bf16 else L.CRF_DT_F32, pa,
                         nw.data_ptr() if with_norm else None, nb.data_ptr() if with_norm else None, int(bool(shuffle)))
        L.check(L.lib().crf_layer_fwd(C.byref(desc), C.byref(la), xd.data_ptr(), v_arg.data_ptr(), y.data_ptr(),
                                      saved.data_ptr(), _stream_ptr(dev)), "crf_layer_fwd")
        _check_guard(saved, sb.value, "crf_layer_fwd saved")
        if training:
            ctx.save_for_backward(xd, v_arg, saved, *((nw, nb) if with_norm else ()), *params)
            ctx.desc = desc
            ctx.meta = (H, W, qk_scale, eps, out_bf16, depth, with_norm, wb.value, bool(shuffle))
        return y.permute(0, 3, 1, 2) if shuffle else y

    @staticmethod
    def backward(ctx, dy):
        H, W, qk_scale, eps, out_bf16, depth, with_norm, ws_bytes, shuffle = ctx.meta
        xd, v_arg, saved, *rest = ctx.saved_tensors
        nw, nb = (rest[0], rest[1]) if with_norm else (None, None)
        params = rest[2:] if with_norm else rest
        desc, dev = ctx.desc, xd.device
        B, Ltok, Cd = xd.shape
        if shuffle:   # (B, C/4, 2H, 2W) gradient -> NHWC memory, the layout the fused LayerNorm backward reads
            dy = dy.to(torch.bfloat16 if out_bf16 else torch.float32).contiguous(memory_format=torch.channels_last)
        else:
            dy = dy.contiguous().to(torch.bfloat16 if out_bf16 else torch.float32)
        ws = _alloc_bytes(ws_bytes, dev)
        dx = torch.empty(B, Ltok, Cd, dtype=xd.dtype, device=dev)   # in x's dtype: no autograd cast afterwards
        dv = torch.empty(B, H, W, Cd, dtype=torch.float32, device=dev)
        # one zero-filled buffer for every parameter gradient (256-byte aligned views)
        shapes = [p.shape for p in params] + ([nw.shape, nb.shape] if with_norm else [])
        offs, o = [], 0
        for shp in shapes:
            offs.append(o)
            o += (shp.numel() + 63) // 64 * 64
        flat = torch.zeros(o, dtype=torch.float32, device=dev)
        views = [flat[a:a + shp.numel()].view(shp) for a, shp in zip(offs, shapes)]
        pa, ga = (L.BlockParams * depth)(), (L.BlockGrads * depth)()
        for i in range(depth):
            for k, name in enumerate(L.PARAM_NAMES):
                setattr(pa[i], name, params[13 * i + k].data_ptr())
                setattr(ga[i], name, views[13 * i + k].data_ptr())
            pa[i].qk_scale, pa[i].ln_eps = float(qk_scale), float(eps)
        la = L.LayerArgs(depth, L.CRF_DT_BF16 if out_bf16 else L.CRF_DT_F32, pa,
                         nw.data_ptr() if with_norm else None, nb.data_ptr() if with_norm else None, int(shuffle))
        dnw = views[13 * depth].data_ptr() if with_norm else None
        dnb = views[13 * depth + 1].data_ptr() if with_norm else None
        L.check(L.lib().crf_layer_bwd(C.byref(desc), C.byref(la), xd.data_ptr(), v_arg.data_ptr(), dy.data_ptr(),
                                      saved.data_ptr(), dx.data_ptr(), dv.data_ptr(), ga, dnw, dnb, ws.data_ptr(),
                                      ws_bytes, _stream_ptr(dev)), "crf_layer_bwd")
        _check_guard(ws, ws_bytes, "crf_layer_bwd workspace")
        gn = (views[13 * depth], views[13 * depth + 1]) if with_norm else (None, None)
        return (dx, dv, None, None, None, None, None, None, None, None, None, None, gn[0], gn[1], *views[:13 * depth])


def crf_layer(x, v, H, W, block_params, num_heads, *, window=7, qk_scale=None, eps=1e-5, norm=None, out_dtype=None,
              precision=None, pixel_shuffle=False):
    """BasicCRFLayer.forward as one call: block_params = [13 tensors in PARAM_KEYS order] per block (shift 0,
    window // 2, 0, ...); norm = (weight, bias) of a closing LayerNorm or None; out_dtype torch.bfloat16 only with
    norm.  Returns (B, H*W, C) -- or, with pixel_shuffle=True (needs norm), F.pixel_shuffle(y as NCHW, 2): a
    (B, C/4, 2H, 2W) channels-last tensor written directly by the closing LayerNorm
    (model_mobileV3_large_newCRFs.py:116-120).  Mirrors the reference's error behaviour (newcrf_layers.py:205,143)."""
    assert x.dim() == 3 and v.dim() == 4
    B, Ltok, Cd = x.shape
    assert Ltok == H * W, "input feature has wrong size"
    assert Cd == v.shape[-1], "self.dim != v.shape[-1]"
    if not x.is_cuda:
        raise RuntimeError("monocular_depth_estimation_b200 runs on CUDA (sm_100a) only; there is no CPU path")
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    if v.dtype not in (torch.float32, torch.bfloat16):
        v = v.float()
    if qk_scale is None:
        qk_scale = (Cd // num_heads) ** -0.5
    flat = [t for blk in block_params for t in blk]
    nw, nb = norm if norm is not None else (None, None)
    out_bf16 = out_dtype == torch.bfloat16
    assert not out_bf16 or norm is not None, "bf16 output needs the closing LayerNorm"
    assert not pixel_shuffle or (norm is not None and Cd % 4 == 0), "pixel_shuffle needs the closing LayerNorm"
    return _CRFLayerFn.apply(x, v, _precision_code(precision), H, W, num_heads, window, float(qk_scale), float(eps),
                             out_bf16, bool(pixel_shuffle), len(block_params), nw, nb, *flat)


class _LayerNormFn(torch.autograd.Function):
    """LayerNorm over the last dim of contiguous fp32 token rows (the stage-closing `norm_crf`,
    /root/reference/src/newcrf_layers.py:430-431) on the library's row kernels; output fp32, or bf16 when asked."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps, out_bf16):
        Cd = x.shape[-1]
        xd = x.detach().contiguous()
        T, dev = xd.numel() // Cd, xd.device
        w, b = weight.detach().contiguous(), bias.detach().contiguous()
        y = torch.empty(x.shape, dtype=torch.bfloat16 if out_bf16 else torch.float32, device=dev)
        stats = torch.empty(T, 2, dtype=torch.float32, device=dev)
        L.check(L.lib().crf_layernorm_fwd(xd.data_ptr(), w.data_ptr(), b.data_ptr(), float(eps), y.data_ptr(),
                                          L.CRF_DT_BF16 if out_bf16 else L.CRF_DT_F32, stats.data_ptr(), T, Cd,
                                          dev.index, _stream_ptr(dev)), "crf_layernorm_fwd")
        ctx.save_for_backward(xd, stats, w)
        return y

    @staticmethod
    def backward(ctx, g):
        xd, stats, w = ctx.saved_tensors
        Cd = xd.shape[-1]
        T, dev = xd.numel() // Cd, xd.device
        if g.dtype not in (torch.float32, torch.bfloat16):
            g = g.float()
        g = g.contiguous()
        dx = torch.empty_like(xd)
        dwb = torch.zeros(2, Cd, dtype=torch.float32, device=dev)
        L.check(L.lib().crf_layernorm_bwd(g.data_ptr(), L.CRF_DT_BF16 if g.dtype == torch.bfloat16 else L.CRF_DT_F32,
                                          xd.data_ptr(), stats.data_ptr(), w.data_ptr(), dx.data_ptr(),
                                          dwb[0].data_ptr(), dwb[1].data_ptr(), T, Cd, dev.index, _stream_ptr(dev)),
                "crf_layernorm_bwd")
        return dx, dwb[0], dwb[1], None, None


def layer_norm(x, weight, bias, eps=1e-5, out_dtype=None):
    """nn.LayerNorm(C)(x) for fp32 CUDA x (..., C), C a multiple of 64 up to 1024.  out_dtype: torch.float32 (default)
    or torch.bfloat16 (what a following autocast convolution would cast to anyway)."""
    if not x.is_cuda:
        raise RuntimeError("monocular_depth_estimation_b200 runs on CUDA (sm_100a) only; there is no CPU path")
    return _LayerNormFn.apply(x.float(), weight, bias, float(eps), out_dtype == torch.bfloat16)


class _DepthLossFn(torch.autograd.Function):
    """loss = SSIM(pred, target) + 0.1 * L1(pred, target) of the reference loop (src/train.py:94-100, src/loss.py:57-88)
    in one forward and one backward kernel; pred fp32 or bf16 (B, C, H, W), target fp32, no gradient for target."""

    @staticmethod
    def forward(ctx, pred, target):
        p = pred.detach().contiguous()
        t = target.detach().float().contiguous()
        H, W = p.shape[-2:]
        n_img, dev = p.numel() // (H * W), p.device
        need = ctx.needs_input_grad[0]
        sums = torch.zeros(2, dtype=torch.float32, device=dev)
        G = torch.empty(3, n_img, H, W, dtype=torch.float32, device=dev) if need else None
        dt = L.CRF_DT_BF16 if p.dtype == torch.bfloat16 else L.CRF_DT_F32
        L.check(L.lib().crf_depth_loss_fwd(p.data_ptr(), dt, t.data_ptr(), n_img, H, W, sums.data_ptr(),
                                           None if G is None else G.data_ptr(), dev.index, _stream_ptr(dev)),
                "crf_depth_loss_fwd")
        if need:
            ctx.save_for_backward(p, t, G)
        return (sums[0] + 0.1 * sums[1]) / float(p.numel())

    @staticmethod
    def backward(ctx, g):
        p, t, G = ctx.saved_tensors
        H, W = p.shape[-2:]
        n_img, dev = p.numel() // (H * W), p.device
        g = g.detach().float().contiguous()
        dp = torch.empty_like(p)
        dt = L.CRF_DT_BF16 if p.dtype == torch.bfloat16 else L.CRF_DT_F32
        L.check(L.lib().crf_depth_loss_bwd(p.data_ptr(), dt, t.data_ptr(), G.data_ptr(), g.data_ptr(), n_img, H, W,
                                           dp.data_ptr(), dev.index, _stream_ptr(dev)), "crf_depth_loss_bwd")
        return dp, None


def depth_loss(pred, target):
    """1.0 * SSIM + 0.1 * L1 (src/train.py:94-100) for CUDA tensors (B, C, H, W), H, W >= 2."""
    if not pred.is_cuda:
        raise RuntimeError("monocular_depth_estimation_b200 runs on CUDA (sm_100a) only; there is no CPU path")
    assert pred.shape == target.shape and pred.dim() == 4, "depth_loss expects pred and target of one (B, C, H, W) shape"
    if pred.dtype not in (torch.float32, torch.bfloat16):
        pred = pred.float()
    return _DepthLossFn.apply(pred, target)


class _PixelShuffleFn(torch.autograd.Function):
    """nn.PixelShuffle(2) for channels-last CUDA tensors (model_mobileV3_large_newCRFs.py:116-120): one permutation
    pass in NHWC memory each way instead of torch's NCHW shuffle plus a layout copy for the following convolution."""

    @staticmethod
    def _run(src, inverse):
        if inverse:   # src logical (B, C/4, 2H, 2W) -> (B, C, H, W)
            B, Cq, H2, W2 = src.shape
            Cd, H, W = Cq * 4, H2 // 2, W2 // 2
            out_shape = (B, Cd, H, W)
        else:         # src logical (B, C, H, W) -> (B, C/4, 2H, 2W)
            B, Cd, H, W = src.shape
            out_shape = (B, Cd // 4, 2 * H, 2 * W)
        dst = torch.empty(out_shape, dtype=src.dtype, device=src.device, memory_format=torch.channels_last)
        dt = L.CRF_DT_BF16 if src.dtype == torch.bfloat16 else L.CRF_DT_F32
        L.check(L.lib().crf_pixel_shuffle_nhwc(src.data_ptr(), dst.data_ptr(), dt, B, H, W, Cd, int(inverse),
                                               src.device.index, _stream_ptr(src.device)), "crf_pixel_shuffle_nhwc")
        return dst

    @staticmethod
    def forward(ctx, x):
        return _PixelShuffleFn._run(x.detach(), False)

    @staticmethod
    def backward(ctx, g):
        return _PixelShuffleFn._run(g.contiguous(memory_format=torch.channels_last), True)


def pixel_shuffle2(x):
    """F.pixel_shuffle(x, 2); channels-last fp32 / bf16 CUDA tensors take the library's NHWC permutation kernel."""
    if (x.is_cuda and x.dim() == 4 and x.shape[1] % 4 == 0 and x.dtype in (torch.float32, torch.bfloat16)
            and x.is_contiguous(memory_format=torch.channels_last)):
        return _PixelShuffleFn.apply(x)
    return torch.nn.functional.pixel_shuffle(x, 2)


class _WindowAttentionFn(torch.autograd.Function):
    """Stand-alone WindowAttention.forward (newcrf_layers.py:110-149) on already-partitioned windows, built from the
    stage-level entry points: qk GEMM -> attention core (each window = a ws x ws image, no pad, no shift) -> proj GEMM."""

    @staticmethod
    def forward(ctx, x, v, mask, num_heads, scale, qk_w, qk_b, table, proj_w, proj_b):
        from . import ops
        B_, N, Cd = x.shape
        T = B_ * N
        dev = x.device
        xb = x.detach().reshape(T, Cd).to(torch.bfloat16).contiguous()
        vb = v.detach().reshape(T, Cd).to(torch.bfloat16).contiguous()
        wqk, wp = ops.cast_bf16(qk_w.detach().contiguous()), ops.cast_bf16(proj_w.detach().contiguous())
        qkb, pb = qk_b.detach().contiguous(), proj_b.detach().contiguous()
        tab = table.detach().contiguous()
        m = None if mask is None else mask.detach().float().contiguous()
        ws = _window_of(N)
        desc = make_desc(B_, ws, ws, Cd, num_heads, 0, window=ws, device=dev.index)
        qk = torch.empty(T, 2 * Cd, dtype=torch.bfloat16, device=dev)
        ops.gemm(xb, wqk, T, 2 * Cd, Cd, epilogue=L.EPI_STORE_BF16, out0=qk, bias=qkb, scale=scale, scale_cols=Cd)
        o, lse = ops.attn_fwd(desc, qk, vb, qkb, scale, tab, want_lse=True, mask=m)
        out = torch.empty(T, Cd, dtype=torch.float32, device=dev)
        ops.gemm(o, wp, T, Cd, Cd, epilogue=L.EPI_STORE_F32, out0=out, bias=pb)
        ctx.save_for_backward(xb, vb, wqk, wp, qkb, tab, qk, o, lse, m if m is not None else torch.empty(0, device=dev))
        ctx.meta = (B_, N, Cd, num_heads, scale, m is not None)
        return out.view(B_, N, Cd)

    @staticmethod
    def backward(ctx, dout):
        from . import ops
        xb, vb, wqk, wp, qkb, tab, qk, o, lse, m = ctx.saved_tensors
        B_, N, Cd, num_heads, scale, has_mask = ctx.meta
        T, dev = B_ * N, xb.device
        ws = _window_of(N)
        desc = make_desc(B_, ws, ws, Cd, num_heads, 0, window=ws, device=dev.index)
        dob = ops.cast_bf16(dout.contiguous().float().reshape(T, Cd))
        d_o = torch.empty(T, Cd, dtype=torch.bfloat16, device=dev)
        ops.gemm(dob, wp, T, Cd, Cd, b_major=1, epilogue=L.EPI_STORE_BF16, out0=d_o)
        d_wp, d_pb = torch.zeros(Cd, Cd, device=dev), torch.zeros(Cd, device=dev)
        ops.gemm(dob, o, Cd, Cd, T, a_major=1, b_major=1, epilogue=L.EPI_SPLITK_F32, out0=d_wp, colsum=d_pb)
        dqk, dv, d_tab, d_qkb = ops.attn_bwd(desc, qk, vb, qkb, scale, tab, lse, d_o, mask=m if has_mask else None)
        dx = torch.empty(T, Cd, dtype=torch.float32, device=dev)
        ops.gemm(dqk, wqk, T, Cd, 2 * Cd, b_major=1, epilogue=L.EPI_STORE_F32, out0=dx)
        d_wqk = torch.zeros(2 * Cd, Cd, device=dev)
        ops.gemm(dqk, xb, 2 * Cd, Cd, T, a_major=1, b_major=1, epilogue=L.EPI_SPLITK_F32, out0=d_wqk, colsum=d_qkb)
        return (dx.view(B_, N, Cd), dv.view(B_, N, Cd), None, None, None, d_wqk, d_qkb, d_tab, d_wp, d_pb)


MIN_WINDOW, MAX_WINDOW = 2, 8   # window sizes the attention kernels implement (N = ws^2 <= 64 tokens per window)


def _window_of(N):
    """The window size ws of an N = ws * ws token window, or None."""
    ws = int(round(N ** 0.5))
    return ws if ws * ws == N and MIN_WINDOW <= ws <= MAX_WINDOW else None


def window_attention(x, v, qk_w, qk_b, table, proj_w, proj_b, num_heads, scale, mask=None):
    """WindowAttention.forward(x, v, mask): x, v (num_windows*B, N, C) windows of ws x ws tokens (N = ws^2, ws in 2..8);
    mask (nW, N, N) or None -> (B_, N, C) fp32."""
    assert x.dim() == 3 and _window_of(x.shape[1]) is not None, \
        f"window attention expects (num_windows*B, ws*ws, C) windows with ws in {MIN_WINDOW}..{MAX_WINDOW}"
    assert x.shape[-1] == v.shape[-1], "self.dim != v.shape[-1]"
    if not x.is_cuda:
        raise RuntimeError("monocular_depth_estimation_b200 runs on CUDA (sm_100a) only; there is no CPU path")
    return _WindowAttentionFn.apply(x, v, mask, num_heads, float(scale), qk_w, qk_b, table, proj_w, proj_b)


_ACT_CODES = {None: L.ACT_NONE, "relu": L.ACT_RELU, "hardswish": L.ACT_HARDSWISH}


class _BatchNormActFn(torch.autograd.Function):
    """Training-mode BatchNorm2d + activation over a channels-last bf16 map on the library (crf_bn_fwd / crf_bn_bwd):
    two kernels each way.  Saves x and the batch statistics only; the BN output the activation's backward needs is
    recomputed from them."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, num_batches_tracked, tickets, eps, momentum, act):
        B, Cd, H, W = x.shape
        T, dev = B * H * W, x.device
        xd = x.detach()
        w, b = weight.detach(), bias.detach()
        y = torch.empty_like(xd)                        # channels-last, like x
        stats = torch.empty(2, Cd, dtype=torch.float32, device=dev)   # save_mean, save_invstd
        ws_bytes = L.lib().crf_bn_workspace_bytes(T, Cd, dev.index)
        ws = _alloc_bytes(ws_bytes, dev)
        L.check(L.lib().crf_bn_fwd(xd.data_ptr(), y.data_ptr(), w.data_ptr(), b.data_ptr(), running_mean.data_ptr(),
                                   running_var.data_ptr(), num_batches_tracked.data_ptr(), stats[0].data_ptr(),
                                   stats[1].data_ptr(), T, Cd, float(eps), float(momentum), act, ws.data_ptr(),
                                   ws_bytes, tickets.data_ptr(), dev.index, _stream_ptr(dev)), "crf_bn_fwd")
        _check_guard(ws, ws_bytes, "crf_bn_fwd workspace")
        ctx.save_for_backward(xd, w, b, stats)
        ctx.tickets, ctx.act = tickets, act
        return y

    @staticmethod
    def backward(ctx, dy):
        xd, w, b, stats = ctx.saved_tensors
        B, Cd, H, W = xd.shape
        T, dev = B * H * W, xd.device
        dy = dy.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        dx = torch.empty_like(xd)
        dwb = torch.empty(2, Cd, dtype=torch.float32, device=dev)
        ws_bytes = L.lib().crf_bn_workspace_bytes(T, Cd, dev.index)
        ws = _alloc_bytes(ws_bytes, dev)
        L.check(L.lib().crf_bn_bwd(xd.data_ptr(), dy.data_ptr(), w.data_ptr(), b.data_ptr(), stats[0].data_ptr(),
                                   stats[1].data_ptr(), dx.data_ptr(), dwb[0].data_ptr(), dwb[1].data_ptr(), T, Cd,
                                   ctx.act, ws.data_ptr(), ws_bytes, ctx.tickets.data_ptr(), dev.index,
                                   _stream_ptr(dev)), "crf_bn_bwd")
        _check_guard(ws, ws_bytes, "crf_bn_bwd workspace")
        return dx, dwb[0], dwb[1], None, None, None, None, None, None, None


def batch_norm_act(x, weight, bias, running_mean, running_var, num_batches_tracked, tickets, eps, momentum, act=None):
    """act(F.batch_norm(x, running_mean, running_var, weight, bias, training=True, momentum, eps)) for a CUDA bf16
    channels-last (B, C, H, W) map, C % 8 == 0, B H W >= 2, fp32 parameters and running statistics; act is None, "relu"
    or "hardswish".  Updates the running statistics and adds 1 to num_batches_tracked on the device.  tickets: int32,
    at least C / 8 zeros, owned by the caller and used by one call at a time."""
    return _BatchNormActFn.apply(x, weight, bias, running_mean, running_var, num_batches_tracked, tickets, eps,
                                 momentum, _ACT_CODES[act])
