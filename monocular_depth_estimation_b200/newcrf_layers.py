"""Drop-in modules for the reference's NeWCRFs CRF layers, backed by the sm_100a C-ABI library.

Same class names, constructor signatures, parameter / buffer names (hence state_dict keys) and forward signatures
as /root/reference/src/newcrf_layers.py, so `NewCRF` / `Decoder` / `PTModel` and a training loop written against the
reference keep working:

    reference class (file:line)                 here
    Mlp                  newcrf_layers.py:9      Mlp              (parameter holder; math runs inside the fused block)
    WindowAttention      newcrf_layers.py:62     WindowAttention.forward(x, v, mask) on pre-partitioned windows (stage-level kernels)
    CRFBlock             newcrf_layers.py:152    CRFBlock.forward(x, v, mask_matrix) with .H/.W set by the caller
    BasicCRFLayer        newcrf_layers.py:260    BasicCRFLayer.forward(x, v, H, W) -> (x, H, W, x, H, W)
    NewCRF               newcrf_layers.py:367    NewCRF.forward(x_nchw, v_nchw) -> nchw

The forward bodies do not build pad / roll / partition tensors or an attention mask: the kernels evaluate those index
maps in closed form (csrc/crf_window.cuh).  Dropout / DropPath rates other than 0 are rejected -- the reference
hard-wires them to 0 (newcrf_layers.py:407-409).
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as CF


def _pair(v):
    return v if isinstance(v, tuple) else (v, v)


def _require_window(window_size):
    if not CF.MIN_WINDOW <= window_size <= CF.MAX_WINDOW:
        raise NotImplementedError(f"window_size={window_size}: the sm_100a attention kernels implement window sizes "
                                  f"{CF.MIN_WINDOW} to {CF.MAX_WINDOW} (a window's ws*ws tokens fill at most 64 tile rows)")


def _require_zero(name, rate):
    if rate != 0.0:
        raise NotImplementedError(f"{name}={rate}: the fused sm_100a CRF block implements the reference's "
                                  "configuration (all dropout / drop-path rates 0)")


class Mlp(nn.Module):
    """fc1 -> GELU(erf) -> fc2. Holds the parameters; CRFBlock runs the math in the fused kernels."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.):
        super().__init__()
        _require_zero("drop", drop)
        if act_layer is not nn.GELU:
            raise NotImplementedError("only nn.GELU (exact erf) is implemented")
        hidden_features = hidden_features or in_features
        out_features = out_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)

    def forward(self, x):
        # Stand-alone use is outside the hot path; the block never calls this.
        return self.fc2(self.act(self.fc1(x)))


class WindowAttention(nn.Module):
    """Parameters of the window attention: qk projection (q and k from x), relative-position-bias table and index
    buffer, output projection.  v is used raw (no V projection), so v_dim must equal dim."""

    def __init__(self, dim, window_size, num_heads, v_dim, qkv_bias=True, qk_scale=None, attn_drop=0., proj_drop=0.):
        super().__init__()
        _require_zero("attn_drop", attn_drop)
        _require_zero("proj_drop", proj_drop)
        if not qkv_bias:
            raise NotImplementedError("qkv_bias=False is not implemented (the reference always uses a bias)")
        self.dim = dim
        self.window_size = _pair(window_size)
        self.num_heads = num_heads
        self.scale = qk_scale or (dim // num_heads) ** -0.5
        wh, ww = self.window_size
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * wh - 1) * (2 * ww - 1), num_heads))
        # idx[i, j] = (yi - yj + wh-1) * (2ww-1) + (xi - xj + ww-1); persistent buffer -> part of the state_dict
        ys, xs = torch.arange(wh * ww) // ww, torch.arange(wh * ww) % ww
        index = (ys[:, None] - ys[None, :] + wh - 1) * (2 * ww - 1) + (xs[:, None] - xs[None, :] + ww - 1)
        self.register_buffer("relative_position_index", index.to(torch.int64))
        self.qk = nn.Linear(dim, dim * 2, bias=True)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(v_dim, v_dim)
        self.proj_drop = nn.Dropout(proj_drop)
        nn.init.trunc_normal_(self.relative_position_bias_table, std=.02)
        self.softmax = nn.Softmax(dim=-1)

    def forward(self, x, v, mask=None):
        """x, v: (num_windows*B, N, C) pre-partitioned windows, N = ws*ws; mask: (nW, N, N) additive or None.
        The fused CRFBlock never materialises windows and does not call this; it exists for drop-in use of the class
        on its own (qk GEMM -> attention core -> proj GEMM through the stage-level entry points)."""
        return CF.window_attention(x, v, self.qk.weight, self.qk.bias, self.relative_position_bias_table,
                                   self.proj.weight, self.proj.bias, self.num_heads, self.scale, mask)


class CRFBlock(nn.Module):
    def __init__(self, dim, num_heads, v_dim, window_size=7, shift_size=0, mlp_ratio=4., qkv_bias=True, qk_scale=None,
                 drop=0., attn_drop=0., drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm):
        super().__init__()
        _require_zero("drop_path", drop_path)
        _require_window(window_size)
        if norm_layer is not nn.LayerNorm:
            raise NotImplementedError("only nn.LayerNorm is implemented")
        assert 0 <= shift_size < window_size, "shift_size must in 0-window_size"
        self.dim, self.num_heads, self.v_dim = dim, num_heads, v_dim
        self.window_size, self.shift_size, self.mlp_ratio = window_size, shift_size, mlp_ratio
        self.norm1 = norm_layer(dim)
        self.attn = WindowAttention(dim, window_size=_pair(window_size), num_heads=num_heads, v_dim=v_dim,
                                    qkv_bias=qkv_bias, qk_scale=qk_scale, attn_drop=attn_drop, proj_drop=drop)
        self.drop_path = nn.Identity()
        self.norm2 = norm_layer(v_dim)
        self.mlp = Mlp(in_features=v_dim, hidden_features=int(v_dim * mlp_ratio), act_layer=act_layer, drop=drop)
        self.H = None
        self.W = None
        self.precision = None      # None: process default (ops.set_precision); "bf16" | "fp32"
        self._mask_checked = None  # (id, version, device) of the last mask_matrix found equal to the closed form

    def fused_params(self):
        """The 13 parameter tensors in the order the C ABI expects (functional.PARAM_KEYS)."""
        return (self.norm1.weight, self.norm1.bias, self.attn.qk.weight, self.attn.qk.bias,
                self.attn.relative_position_bias_table, self.attn.proj.weight, self.attn.proj.bias,
                self.norm2.weight, self.norm2.bias, self.mlp.fc1.weight, self.mlp.fc1.bias,
                self.mlp.fc2.weight, self.mlp.fc2.bias)

    def _custom_mask(self, mask_matrix, H, W):
        """None when `mask_matrix` is the mask BasicCRFLayer.forward builds for this (H, W) (newcrf_layers.py:332-350:
        the kernels evaluate that one in closed form), else the mask itself (handed to the kernels, where it replaces
        the closed form).  As in the reference (:225-236) an unshifted block ignores the argument."""
        if mask_matrix is None or self.shift_size == 0:
            return None
        ws = self.window_size
        hp, wp, n = -(-H // ws) * ws, -(-W // ws) * ws, ws * ws
        assert tuple(mask_matrix.shape) == ((hp // ws) * (wp // ws), n, n), \
            "mask_matrix does not belong to this (H, W, window_size)"
        if not mask_matrix.is_cuda or torch.cuda.is_current_stream_capturing():
            return mask_matrix.to(self.norm1.weight.device)   # no host comparison inside a graph capture
        key = (id(mask_matrix), mask_matrix._version, H, W)
        if self._mask_checked == key:
            return None
        from . import ops
        if torch.equal(mask_matrix.float(), ops.shift_mask(H, W, ws, self.shift_size, mask_matrix.device)):
            self._mask_checked = key
            return None
        return mask_matrix

    def forward(self, x, v, mask_matrix=None, v_bf16=None):
        """x: (B, H*W, C); v: (B, H, W, C); self.H / self.W set by the caller (as BasicCRFLayer does).
        mask_matrix: the (nW, N, N) additive mask of a shifted block (N = window_size^2).  The standard one (what BasicCRFLayer.forward
        builds) is recognised and evaluated in closed form inside the kernels; any other mask is honoured as given."""
        H, W = self.H, self.W
        B, Ltok, _ = x.shape
        assert Ltok == H * W, "input feature has wrong size"
        mask = self._custom_mask(mask_matrix, H, W)
        return CF.crf_block(x, v, H, W, self.fused_params(), self.num_heads, window=self.window_size,
                            shift=self.shift_size, qk_scale=self.attn.scale, eps=self.norm1.eps, v_bf16=v_bf16,
                            mask=mask, precision=self.precision)


class BasicCRFLayer(nn.Module):
    def __init__(self, dim, depth, num_heads, v_dim, window_size=7, mlp_ratio=4., qkv_bias=True, qk_scale=None,
                 drop=0., attn_drop=0., drop_path=0., norm_layer=nn.LayerNorm, downsample=None, use_checkpoint=False):
        super().__init__()
        if downsample is not None:
            raise NotImplementedError("downsample is always None in the reference (newcrf_layers.py:411)")
        _require_window(window_size)
        self.window_size = window_size
        self.shift_size = window_size // 2
        self.depth = depth
        self.use_checkpoint = use_checkpoint  # the fused backward recomputes S/P itself; flag kept for the signature
        self.precision = None                 # None: process default (ops.set_precision); "bf16" | "fp32"
        self.blocks = nn.ModuleList([
            CRFBlock(dim=dim, num_heads=num_heads, v_dim=v_dim, window_size=window_size,
                     shift_size=0 if i % 2 == 0 else window_size // 2, mlp_ratio=mlp_ratio, qkv_bias=qkv_bias,
                     qk_scale=qk_scale, drop=drop, attn_drop=attn_drop,
                     drop_path=drop_path[i] if isinstance(drop_path, list) else drop_path, norm_layer=norm_layer)
            for i in range(depth)])
        self.downsample = None

    def _fusable(self, x):
        """One crf_layer_fwd / crf_layer_bwd call covers the whole layer when the blocks are the stock alternation."""
        blk0 = self.blocks[0]
        return (x.is_cuda and 1 <= self.depth <= 8
                and all(b.shift_size == (0 if i % 2 == 0 else self.window_size // 2) and b.num_heads == blk0.num_heads
                        and b.window_size == self.window_size and b.norm1.eps == blk0.norm1.eps
                        and b.attn.scale == blk0.attn.scale for i, b in enumerate(self.blocks)))

    def run(self, x, v, H, W, norm=None, out_dtype=None, pixel_shuffle=False):
        """The layer, optionally closed by `norm` (an nn.LayerNorm: NewCRF.norm_crf) -> (B, H*W, C); with
        pixel_shuffle=True (fused path only, needs norm) -> F.pixel_shuffle of the NCHW result, (B, C/4, 2H, 2W)."""
        for blk in self.blocks:
            blk.H, blk.W = H, W
        if self._fusable(x) and (norm is None or (type(norm) is nn.LayerNorm and norm.elementwise_affine
                                                  and norm.eps == self.blocks[0].norm1.eps)):
            blk0 = self.blocks[0]
            assert x.shape[1] == H * W, "input feature has wrong size"
            return CF.crf_layer(x, v, H, W, [b.fused_params() for b in self.blocks], blk0.num_heads,
                                window=self.window_size, qk_scale=blk0.attn.scale, eps=blk0.norm1.eps,
                                norm=None if norm is None else (norm.weight, norm.bias), out_dtype=out_dtype,
                                precision=self.precision, pixel_shuffle=pixel_shuffle)
        v_bf16 = CF.convert_v(v) if (v.is_cuda and self.depth > 1) else None  # both blocks read the same v
        for blk in self.blocks:
            if blk.precision is None:
                blk.precision = self.precision
            x = blk(x, v, None, v_bf16=v_bf16)
        if norm is not None:
            x = norm(x)
        if pixel_shuffle:
            B, _, Cd = x.shape
            x = F.pixel_shuffle(x.view(B, H, W, Cd).permute(0, 3, 1, 2), 2)
        return x

    def forward(self, x, v, H, W):
        """x: (B, H*W, C); v: (B, H, W, C), the same for every block.  Returns (x, H, W, x, H, W)."""
        x = self.run(x, v, H, W)
        return x, H, W, x, H, W


class _ConvBiasFn(torch.autograd.Function):
    """y + bias for the output of a bias-free convolution.  Exists for its backward: stock PyTorch computes a conv
    bias gradient with a generic reduction that takes ~170 us on a channels-last bf16 (8, 128, 120, 160) gradient
    (0.7 ms per training step over the decoder's projections); here it is the library's column-sum kernel over the
    same memory viewed as (B*H*W, C) rows (~20 us).  The gradient of y passes through untouched."""

    @staticmethod
    def forward(ctx, y, bias):
        ctx.bias_dtype = bias.dtype
        return y + bias.to(y.dtype).view(1, -1, 1, 1)

    @staticmethod
    def backward(ctx, g):
        Cd = g.shape[1]
        if (g.is_cuda and g.dtype == torch.bfloat16 and g.is_contiguous(memory_format=torch.channels_last)
                and Cd % 8 == 0):
            from . import ops
            db = ops.colsum_bf16(g.permute(0, 2, 3, 1).reshape(-1, Cd))
        else:
            db = g.float().sum((0, 2, 3))
        return g, db.to(ctx.bias_dtype)


def _project(conv, x):
    """conv(x) as in the reference (newcrf_layers.py:420-423), with the bias added outside cuDNN on CUDA (see above)."""
    if conv.bias is None or not x.is_cuda:
        return conv(x)
    y = F.conv2d(x, conv.weight, None, conv.stride, conv.padding, conv.dilation, conv.groups)
    return _ConvBiasFn.apply(y, conv.bias)


class NewCRF(nn.Module):
    """One decoder stage: 3x3 conv projections of the image feature (x) and the depth feature (v), the CRF layer on
    token views of the NCHW tensors, a final LayerNorm, back to NCHW (newcrf_layers.py:367-434)."""

    def __init__(self, input_dim=96, embed_dim=96, v_dim=64, window_size=7, num_heads=4, depth=2, patch_size=4,
                 in_chans=3, norm_layer=nn.LayerNorm, patch_norm=True):
        super().__init__()
        self.embed_dim = embed_dim
        self.patch_norm = patch_norm
        self.proj_x = nn.Conv2d(input_dim, embed_dim, 3, padding=1) if input_dim != embed_dim else None
        self.proj_v = nn.Conv2d(v_dim, embed_dim, 3, padding=1) if v_dim != embed_dim else None
        self.crf_layer = BasicCRFLayer(dim=embed_dim, depth=depth, num_heads=num_heads, v_dim=embed_dim,
                                       window_size=window_size, mlp_ratio=4., qkv_bias=True, qk_scale=None, drop=0.,
                                       attn_drop=0., drop_path=0., norm_layer=norm_layer, downsample=None,
                                       use_checkpoint=False)
        self.norm_crf = norm_layer(embed_dim)

    def forward(self, x, v, pixel_shuffle=False):
        """pixel_shuffle=True returns nn.PixelShuffle(2) of the stage's output (the decoder applies it to three of the
        four stages, model_mobileV3_large_newCRFs.py:116-120): the closing LayerNorm then writes the shuffled map itself."""
        if self.proj_x is not None:
            x = _project(self.proj_x, x)
        if self.proj_v is not None:
            v = _project(self.proj_v, v)
        B, Cd, Wh, Ww = x.shape
        tokens = x.flatten(2).transpose(1, 2)      # (B, H*W, C) view of NCHW -- the kernel reads it strided
        v_hwc = v.permute(0, 2, 3, 1)              # (B, H, W, C) view of NCHW
        # the layer and the closing norm in one library call; under bf16 autocast the result is emitted in bf16 (the
        # next consumer is a convolution that would cast the fp32 result anyway -- same values, one pass less)
        bf16 = x.is_cuda and torch.is_autocast_enabled() and torch.get_autocast_gpu_dtype() == torch.bfloat16
        y = self.crf_layer.run(tokens, v_hwc, Wh, Ww, norm=self.norm_crf,
                               out_dtype=torch.bfloat16 if bf16 else torch.float32, pixel_shuffle=pixel_shuffle)
        if pixel_shuffle:
            return y   # (B, C/4, 2H, 2W), channels-last memory
        out = y.view(B, Wh, Ww, self.embed_dim).permute(0, 3, 1, 2)
        if x.is_contiguous(memory_format=torch.channels_last) and not x.is_contiguous():
            return out  # channels-last pipeline: the token-major result already IS NHWC memory, no copy needed
        return out.contiguous()
