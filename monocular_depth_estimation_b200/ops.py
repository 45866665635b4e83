"""Thin torch-tensor wrappers over the stage-level C-ABI entry points (include/crf_sm100.h).

These exist for unit tests and profiling of the individual kernels; the training path goes through
`functional.crf_block` which makes ONE C call per block forward / backward.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(t):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _dev(t):
    return t.device.index if t.device.index is not None else torch.cuda.current_device()


_DEFAULT_PRECISION = [L.PREC_BF16]


def set_precision(mode):
    """Process-wide default arithmetic of the CRF blocks: "bf16" (bf16 tensor-core operands and intermediates, the rel 2e-2
    tier of BASELINE.json) or "fp32" (split-operand tensor-core GEMMs with fp32 intermediates and fp32 attention: the
    rel 1e-3 tier).  Returns the previous mode.  Modules / functional calls can override it per call (precision=...)."""
    prev = "fp32" if _DEFAULT_PRECISION[0] == L.PREC_FP32 else "bf16"
    _DEFAULT_PRECISION[0] = _precision_code(mode)
    return prev


def _precision_code(mode):
    if mode is None:
        return _DEFAULT_PRECISION[0]
    if mode in (L.PREC_BF16, "bf16", "bfloat16"):
        return L.PREC_BF16
    if mode in (L.PREC_FP32, "fp32", "float32"):
        return L.PREC_FP32
    raise ValueError(f"precision must be 'bf16' or 'fp32' (got {mode!r})")


def make_desc(B, H, W, Cdim, num_heads, shift, *, window=7, training=1, device=0, x=None, v=None,
              v_preconverted=0, precision=None):
    d = L.BlockDesc()
    d.precision = _precision_code(precision)
    d.B, d.H, d.W, d.C = B, H, W, Cdim
    d.num_heads, d.window, d.shift = num_heads, window, shift
    d.training, d.device = int(training), int(device)
    d.v_preconverted = int(v_preconverted)
    if x is not None:
        assert x.dim() == 3
        d.x_dtype = L.CRF_DT_BF16 if x.dtype == torch.bfloat16 else L.CRF_DT_F32
        d.x_stride_b, d.x_stride_t, d.x_stride_c = x.stride()
    else:
        d.x_dtype = L.CRF_DT_F32
        d.x_stride_b, d.x_stride_t, d.x_stride_c = H * W * Cdim, Cdim, 1
    if v is not None and not v_preconverted:
        assert v.dim() == 4
        d.v_dtype = L.CRF_DT_BF16 if v.dtype == torch.bfloat16 else L.CRF_DT_F32
        d.v_stride_b, d.v_stride_h, d.v_stride_w, d.v_stride_c = v.stride()
    else:
        d.v_dtype = L.CRF_DT_BF16
        d.v_stride_b, d.v_stride_h, d.v_stride_w, d.v_stride_c = H * W * Cdim, W * Cdim, Cdim, 1
    return d


def gemm(A, B, M, N, K, *, a_major=0, b_major=0, epilogue=L.EPI_STORE_F32, out0, out1=None, bias=None, aux1=None,
         ld_out=None, scale=1.0, scale_cols=0, split_k=0, colsum=None):
    a = L.GemmArgs()
    a.A, a.B = A.data_ptr(), B.data_ptr()
    a.a_major, a.b_major = a_major, b_major
    a.M, a.N, a.K = M, N, K
    a.epilogue, a.split_k = epilogue, split_k
    a.out0 = out0.data_ptr()
    a.out1 = out1.data_ptr() if out1 is not None else None
    a.bias = bias.data_ptr() if bias is not None else None
    a.aux1 = aux1.data_ptr() if aux1 is not None else None
    a.ld_out = N if ld_out is None else ld_out
    a.scale, a.scale_cols = scale, scale_cols
    a.device = _dev(A)
    a.colsum = colsum.data_ptr() if colsum is not None else None
    ws = None
    if epilogue == L.EPI_SPLITK_F32:
        need = L.lib().crf_gemm_workspace_bytes(M, N, K, a.device)
        if need:
            ws = torch.empty(need, dtype=torch.uint8, device=A.device)
            a.workspace, a.workspace_bytes = ws.data_ptr(), need
    L.check(L.lib().crf_gemm(C.byref(a), _stream(A)), "crf_gemm")
    return out0


def mlp_fwd(x1, norm_w, norm_b, w1_bf16, b1, w2_bf16, b2, eps=1e-5, training=True):
    """Fused LayerNorm -> fc1 -> GELU -> fc2 -> + x1 (crf_mlp_fwd; C = 128 / 256).  x1: fp32 (T, C) contiguous.
    Returns (y, xn2, stats, pre, act); the last four are None with training=False."""
    T, Cd = x1.shape
    dev = x1.device
    y = torch.empty(T, Cd, dtype=torch.float32, device=dev)
    xn2 = stats = pre = act = None
    if training:
        xn2 = torch.empty(T, Cd, dtype=torch.bfloat16, device=dev)
        stats = torch.empty(T, 2, dtype=torch.float32, device=dev)
        pre = torch.empty(T, 4 * Cd, dtype=torch.bfloat16, device=dev)
        act = torch.empty(T, 4 * Cd, dtype=torch.bfloat16, device=dev)
    a = L.MlpArgs()
    a.x1, a.y = x1.data_ptr(), y.data_ptr()
    a.w1_bf16, a.w2_bf16 = w1_bf16.data_ptr(), w2_bf16.data_ptr()
    a.b1, a.b2, a.norm_w, a.norm_b = b1.data_ptr(), b2.data_ptr(), norm_w.data_ptr(), norm_b.data_ptr()
    if training:
        a.xn2, a.stats, a.pre, a.act = xn2.data_ptr(), stats.data_ptr(), pre.data_ptr(), act.data_ptr()
    a.eps, a.T, a.C, a.training, a.device = eps, T, Cd, int(training), _dev(x1)
    L.check(L.lib().crf_mlp_fwd(C.byref(a), _stream(x1)), "crf_mlp_fwd")
    return y, xn2, stats, pre, act


def ln_fwd(x, gamma, beta, eps=1e-5, want_copy=False):
    """x: logical (B, T_img, C) any strides -> (xn bf16 (B*T_img, C), stats (B*T_img, 2), copy or None)"""
    Bn, T_img, Cd = x.shape
    xn = torch.empty(Bn * T_img, Cd, dtype=torch.bfloat16, device=x.device)
    stats = torch.empty(Bn * T_img, 2, dtype=torch.float32, device=x.device)
    cp = torch.empty(Bn * T_img, Cd, dtype=torch.float32, device=x.device) if want_copy else None
    dt = L.CRF_DT_BF16 if x.dtype == torch.bfloat16 else L.CRF_DT_F32
    sb, st, sc = x.stride()
    L.check(L.lib().crf_ln_fwd(_ptr(x), dt, sb, st, sc, Bn, T_img, Cd, _ptr(gamma), _ptr(beta), eps, _ptr(xn),
                               _ptr(stats), _ptr(cp), _dev(x), _stream(x)), "crf_ln_fwd")
    return xn, stats, cp


def ln_bwd(g, x, stats, gamma, dres=None, want_bf16=False):
    T, Cd = g.shape
    dx = torch.empty_like(g)
    dxb = torch.empty(T, Cd, dtype=torch.bfloat16, device=g.device) if want_bf16 else None
    dgamma = torch.zeros(Cd, dtype=torch.float32, device=g.device)
    dbeta = torch.zeros(Cd, dtype=torch.float32, device=g.device)
    L.check(L.lib().crf_ln_bwd(_ptr(g), _ptr(x), _ptr(stats), _ptr(gamma), _ptr(dres), _ptr(dx), _ptr(dxb),
                               _ptr(dgamma), _ptr(dbeta), T, Cd, _dev(g), _stream(g)), "crf_ln_bwd")
    return dx, dxb, dgamma, dbeta


def dgrad_ln_bwd(dy_bf16, w_bf16, x, stats, gamma, dres=None, want_f32=True, want_bf16=True):
    """dx = LN'(dy @ W; x, stats, gamma) + dres in one kernel (crf_dgrad_ln_bwd; C = 128 / 256).
    dy_bf16 (T, K), w_bf16 (K, C) -> (dx f32 or None, dx bf16 or None, dgamma, dbeta)."""
    T, K = dy_bf16.shape
    Cd = w_bf16.shape[1]
    dev = x.device
    dx = torch.empty(T, Cd, dtype=torch.float32, device=dev) if want_f32 else None
    dxb = torch.empty(T, Cd, dtype=torch.bfloat16, device=dev) if want_bf16 else None
    dgamma = torch.zeros(Cd, dtype=torch.float32, device=dev)
    dbeta = torch.zeros(Cd, dtype=torch.float32, device=dev)
    L.check(L.lib().crf_dgrad_ln_bwd(_ptr(dy_bf16), _ptr(w_bf16), K, _ptr(x), _ptr(stats), _ptr(gamma), _ptr(dres),
                                     _ptr(dx), _ptr(dxb), _ptr(dgamma), _ptr(dbeta), T, Cd, _dev(x), _stream(x)),
            "crf_dgrad_ln_bwd")
    return dx, dxb, dgamma, dbeta


def colsum_bf16(g):
    T, N = g.shape
    out = torch.zeros(N, dtype=torch.float32, device=g.device)
    L.check(L.lib().crf_colsum_bf16(_ptr(g), _ptr(out), T, N, _dev(g), _stream(g)), "crf_colsum_bf16")
    return out


def cast_bf16(src):
    dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    L.check(L.lib().crf_cast_bf16(_ptr(src), _ptr(dst), src.numel(), _dev(src), _stream(src)), "crf_cast_bf16")
    return dst


def convert_v(v):
    """v: logical (B, H, W, C), any (H,W)-collapsible strides, fp32/bf16 -> bf16 (B*H*W, C)"""
    Bn, H, W, Cd = v.shape
    d = make_desc(Bn, H, W, Cd, Cd // 32, 0, device=_dev(v), v=v)
    out = torch.empty(Bn * H * W, Cd, dtype=torch.bfloat16, device=v.device)
    L.check(L.lib().crf_convert_v(C.byref(d), _ptr(v), _ptr(out), _stream(v)), "crf_convert_v")
    return out


def window_gather(x, window, shift):
    Bn, H, W, Cd = x.shape
    Hp, Wp = -(-H // window) * window, -(-W // window) * window
    nW = (Hp // window) * (Wp // window)
    out = torch.empty(Bn * nW, window * window, Cd, dtype=torch.float32, device=x.device)
    L.check(L.lib().crf_window_gather(_ptr(x), _ptr(out), Bn, H, W, Cd, window, shift, _stream(x)),
            "crf_window_gather")
    return out


def window_scatter(windows, Bn, H, W, window, shift):
    Cd = windows.shape[-1]
    out = torch.zeros(Bn, H, W, Cd, dtype=torch.float32, device=windows.device)
    L.check(L.lib().crf_window_scatter(_ptr(windows), _ptr(out), Bn, H, W, Cd, window, shift, _stream(windows)),
            "crf_window_scatter")
    return out


def shift_mask(H, W, window, shift, device):
    Hp, Wp = -(-H // window) * window, -(-W // window) * window
    nW = (Hp // window) * (Wp // window)
    N = window * window
    out = torch.empty(nW, N, N, dtype=torch.float32, device=device)
    L.check(L.lib().crf_shift_mask(_ptr(out), H, W, window, shift, _stream(out)), "crf_shift_mask")
    return out


def attn_fwd(desc, qk, vb, qk_bias, scale, table, want_lse=True, mask=None):
    T, Cd = vb.shape
    ws = desc.window
    Hp, Wp = -(-desc.H // ws) * ws, -(-desc.W // ws) * ws
    nW = (Hp // ws) * (Wp // ws)
    o = torch.zeros(T, Cd, dtype=torch.bfloat16, device=vb.device)
    lse = torch.zeros(desc.B * nW, desc.num_heads, 64, dtype=torch.float32, device=vb.device) if want_lse else None
    L.check(L.lib().crf_attn_fwd(C.byref(desc), _ptr(qk), _ptr(vb), _ptr(qk_bias), scale, _ptr(table), _ptr(mask),
                                 0 if mask is None else mask.shape[0], _ptr(o), _ptr(lse), _stream(vb)),
            "crf_attn_fwd")
    return o, lse


def attn_bwd(desc, qk, vb, qk_bias, scale, table, lse, dout, mask=None):
    T, Cd = vb.shape
    dqk = torch.zeros(T, 2 * Cd, dtype=torch.bfloat16, device=vb.device)
    dv = torch.zeros(T, Cd, dtype=torch.float32, device=vb.device)
    d_table = torch.zeros_like(table)
    d_bias = torch.zeros_like(qk_bias)
    L.check(L.lib().crf_attn_bwd(C.byref(desc), _ptr(qk), _ptr(vb), _ptr(qk_bias), scale, _ptr(table), _ptr(mask),
                                 0 if mask is None else mask.shape[0], _ptr(lse), _ptr(dout), _ptr(dqk), _ptr(dv), 0,
                                 _ptr(d_table), _ptr(d_bias), _stream(vb)), "crf_attn_bwd")
    return dqk, dv, d_table, d_bias
