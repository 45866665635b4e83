"""Stage-level parity tests of the individual sm_100a kernels, called through the C ABI (ctypes) and compared with
plain PyTorch fp32 references of the same op evaluated on the same (bf16-rounded) inputs."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import crf_oracle as O
from tests.helpers import load_golden, rel_l2

pytestmark = pytest.mark.gpu


def _ops():
    from monocular_depth_estimation_b200 import ops
    return ops


def _L():
    from monocular_depth_estimation_b200 import _lib
    return _lib


def _block_err_map(got, ref, bm=32, bn=32):
    """Coarse map of max |err| per (bm x bn) block -- tells which tile / k-slice of a GEMM went wrong."""
    e = (got.double() - ref.double()).abs()
    M, N = e.shape
    Mp, Np = -(-M // bm) * bm, -(-N // bn) * bn
    pad = torch.zeros(Mp, Np, dtype=e.dtype, device=e.device)
    pad[:M, :N] = e
    m = pad.reshape(Mp // bm, bm, Np // bn, bn).amax(dim=(1, 3))
    return np.array2string(m.cpu().numpy()[:12, :12], precision=2, max_line_width=200)


def _check(got, ref, tol, what):
    err = rel_l2(got, ref)
    assert err < tol and torch.isfinite(got.float()).all(), (
        f"{what}: rel_l2={err:.3e} (tol {tol:g})\nblock max-abs-error map (first 12x12 blocks of 32x32):\n"
        + (_block_err_map(got.reshape(-1, got.shape[-1]), ref.reshape(-1, ref.shape[-1])) if got.dim() >= 2 else ""))


DEV = "cuda"


def _rand_bf16(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(torch.bfloat16).to(DEV)


# ---------------------------------------------------------------------------------------------------------
# GEMM: the three operand orientations
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (90, 128, 128), (300, 128, 128), (1000, 256, 512), (257, 64, 192),
                                   (4800, 512, 128), (640, 1024, 256), (384, 128, 2048), (200, 256, 4096),
                                   # 152 / 300 tiles on 148 SMs: the K-split work units with the TMA reduce-add
                                   (2400, 1024, 4096), (2400, 1024, 1024), (9600, 512, 2048),
                                   # a block's N = C projections at C = 64 (mod 128): gemm_kernel<64>, 3 / 15 column tiles
                                   (600, 192, 192), (600, 192, 768), (600, 960, 960), (600, 960, 3840)])
def test_gemm_fprop(M, N, K):
    ops, L = _ops(), _L()
    A, W = _rand_bf16(M, K, seed=1), _rand_bf16(N, K, seed=2, scale=K ** -0.5)
    out = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm(A, W, M, N, K, a_major=0, b_major=0, epilogue=L.EPI_STORE_F32, out0=out)
    torch.cuda.synchronize()
    _check(out, A.float() @ W.float().t(), 1e-5, f"fprop {M}x{N}x{K}")


@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (300, 128, 128), (1000, 512, 128), (257, 128, 512),
                                   (640, 256, 1024), (500, 2048, 512), (2400, 1024, 4096), (2400, 1024, 2048),
                                   (9600, 512, 2048),
                                   # d fc1 / d qk of a block at C = 320 and 576: gemm_kernel<64>, 5 / 9 column tiles
                                   (600, 320, 1280), (600, 320, 640), (600, 576, 2304), (600, 576, 1152)])
def test_gemm_dgrad(M, N, K):
    """dX = dY (M,K) @ W (K,N): B operand read MN-major from the (out,in) weight."""
    ops, L = _ops(), _L()
    A, W = _rand_bf16(M, K, seed=3), _rand_bf16(K, N, seed=4, scale=K ** -0.5)
    out = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm(A, W, M, N, K, a_major=0, b_major=1, epilogue=L.EPI_STORE_F32, out0=out)
    torch.cuda.synchronize()
    _check(out, A.float() @ W.float(), 1e-5, f"dgrad {M}x{N}x{K}")


@pytest.mark.parametrize("M,N,K,split", [(128, 64, 64, 1), (128, 128, 1000, 1), (512, 128, 1000, 4),
                                         (64, 256, 333, 3), (256, 512, 4800, 16), (1024, 256, 2400, 0),
                                         (128, 512, 153600, 0), (4096, 1024, 2400, 0), (2048, 512, 9600, 0),
                                         # the four weight gradients of a block at C = 192 (BN 64 and 256)
                                         (192, 192, 600, 0), (384, 192, 600, 0), (768, 192, 600, 4), (192, 768, 600, 0)])
def test_gemm_wgrad(M, N, K, split):
    """dW (M,N) += dY (K,M)^T @ X (K,N): both operands MN-major, split-K over tokens (partials + reduce)."""
    ops, L = _ops(), _L()
    A, B = _rand_bf16(K, M, seed=5), _rand_bf16(K, N, seed=6, scale=K ** -0.5)
    out = torch.ones(M, N, device=DEV)        # accumulate semantics: starts non-zero
    db = torch.ones(M, device=DEV)            # fused bias gradient: db[m] += sum_k A[k, m]
    ops.gemm(A, B, M, N, K, a_major=1, b_major=1, epilogue=L.EPI_SPLITK_F32, out0=out, split_k=split, colsum=db)
    torch.cuda.synchronize()
    _check(out - 1.0, A.float().t() @ B.float(), 2e-5, f"wgrad {M}x{N}x{K} split {split}")
    _check(db - 1.0, A.float().sum(0), 2e-5, f"wgrad colsum {M}x{N}x{K} split {split}")


@pytest.mark.parametrize("M,N,K,kind", [(300, 128, 128, "fprop"), (1000, 256, 512, "fprop"), (257, 64, 192, "fprop"),
                                        (300, 128, 128, "dgrad"), (1000, 512, 128, "dgrad"), (90, 64, 1024, "dgrad"),
                                        (128, 128, 1000, "wgrad"), (512, 128, 5000, "wgrad"), (64, 256, 333, "wgrad"),
                                        (600, 192, 192, "fprop"), (600, 320, 1280, "dgrad"), (192, 192, 600, "wgrad")])
def test_gemm_split3_fp32_emulation(M, N, K, kind):
    """crf_gemm_args.split3 (the fp32 precision mode, csrc/crf_precise.cu): operands stored as [hi | lo] bf16 pairs, the
    product accumulates hi*hi + hi*lo + lo*hi in fp32.  Against a float64 product of the ORIGINAL fp32 matrices: rel
    2e-5 (bf16 x bf16 alone gives 3e-3), for all three operand orientations, with bias / column sums."""
    ops, L = _ops(), _L()
    g = torch.Generator(device="cpu").manual_seed(M + N + K)

    def split(t):   # (rows, cols) fp32 -> (rows, 2 cols) bf16 [hi | lo]
        hi = t.to(torch.bfloat16)
        lo = (t - hi.float()).to(torch.bfloat16)
        return torch.cat([hi, lo], dim=1).contiguous()

    if kind == "fprop":      # D = A W^T + b : A (M, K), W (N, K), both K-major
        A, B_ = torch.randn(M, K, generator=g).to(DEV), (torch.randn(N, K, generator=g) * K ** -0.5).to(DEV)
        bias = torch.randn(N, generator=g).to(DEV)
        out = torch.full((M, N), float("nan"), device=DEV)
        a = L.GemmArgs()
        As, Bs = split(A), split(B_)
        ref = A.double() @ B_.double().t() + bias.double()
        am, bm = 0, 0
    elif kind == "dgrad":    # D = A W : A (M, K) K-major, W (K, N) MN-major
        A, B_ = torch.randn(M, K, generator=g).to(DEV), (torch.randn(K, N, generator=g) * K ** -0.5).to(DEV)
        bias = None
        out = torch.full((M, N), float("nan"), device=DEV)
        As, Bs = split(A), split(B_)
        ref = A.double() @ B_.double()
        am, bm = 0, 1
    else:                    # D += A^T B : A (K, M), B (K, N), both MN-major, K = tokens (split-K), colsum = sum_k A
        A, B_ = (torch.randn(K, M, generator=g) * K ** -0.5).to(DEV), torch.randn(K, N, generator=g).to(DEV)
        bias = None
        out = torch.zeros(M, N, device=DEV)
        As, Bs = split(A), split(B_)
        ref = A.double().t() @ B_.double()
        am, bm = 1, 1
    a = L.GemmArgs()
    a.A, a.B, a.a_major, a.b_major = As.data_ptr(), Bs.data_ptr(), am, bm
    a.M, a.N, a.K = M, N, K
    a.epilogue = L.EPI_SPLITK_F32 if kind == "wgrad" else L.EPI_STORE_F32
    a.out0, a.ld_out, a.scale, a.device, a.split3 = out.data_ptr(), N, 1.0, 0, 1
    if bias is not None:
        a.bias = bias.data_ptr()
    colsum = None
    if kind == "wgrad":
        colsum = torch.zeros(M, device=DEV)
        a.colsum = colsum.data_ptr()
        need = L.lib().crf_gemm_workspace_bytes(M, N, 3 * K, 0)
        ws = torch.empty(max(need, 256), dtype=torch.uint8, device=DEV)
        a.workspace, a.workspace_bytes = ws.data_ptr(), need
    import ctypes as C
    L.check(L.lib().crf_gemm(C.byref(a), C.c_void_p(torch.cuda.current_stream().cuda_stream)), "crf_gemm split3")
    torch.cuda.synchronize()
    _check(out, ref, 2e-5, f"gemm split3 {kind}")
    if colsum is not None:
        _check(colsum, A.double().sum(0), 2e-5, "gemm split3 colsum")


@pytest.mark.parametrize("M,N,K", [(2400, 1024, 4096), (2400, 1024, 1024), (9600, 512, 2048)])
def test_gemm_bias_residual_with_k_splits(M, N, K):
    """fc2 / proj of the 1/32 and 1/16 decoder scales: out = A W^T + bias + residual with the output tile summed over
    K-split work units by TMA reduce-adds (only the first unit adds bias and residual)."""
    ops, L = _ops(), _L()
    A, W = _rand_bf16(M, K, seed=11), _rand_bf16(N, K, seed=12, scale=K ** -0.5)
    bias = torch.randn(N, device=DEV)
    res = torch.randn(M, N, device=DEV)
    out = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm(A, W, M, N, K, epilogue=L.EPI_BIAS_RES_F32, out0=out, bias=bias, aux1=res)
    torch.cuda.synchronize()
    _check(out, A.float() @ W.float().t() + bias + res, 1e-5, f"bias+res {M}x{N}x{K}")


@pytest.mark.parametrize("M,N,K", [(2400, 4096, 1024), (2400, 1024, 4096), (2400, 1024, 1024), (2400, 2048, 1024),
                                   (9600, 512, 512), (9600, 2048, 512), (9600, 512, 2048), (9600, 1024, 512),
                                   (1000, 512, 1024), (300, 1024, 2048),
                                   # odd numbers of 256-wide column tiles (3 ... 15), the q-scale boundary inside a tile
                                   # at 5 and 7 tiles, and several rounds of the 74 pairs at T = 9600
                                   (2400, 768, 768), (2400, 1280, 640), (2400, 1792, 896), (9600, 2304, 576),
                                   (2400, 3840, 960)])
@pytest.mark.parametrize("kind", ["fprop", "dgrad"])
def test_gemm_pair_epilogues(M, N, K, kind):
    """The CTA-pair GEMM (csrc/crf_gemm_pair.cu, 256 x 256 tiles on the two SMs of a TPC) with every epilogue the
    C >= 512 projections use, against fp32 PyTorch."""
    ops, L = _ops(), _L()
    bm = 0 if kind == "fprop" else 1
    A = _rand_bf16(M, K, seed=21)
    W = _rand_bf16(N, K, seed=22, scale=K ** -0.5) if bm == 0 else _rand_bf16(K, N, seed=22, scale=K ** -0.5)
    acc = A.float() @ (W.float().t() if bm == 0 else W.float())
    bias = torch.randn(N, device=DEV)
    res = torch.randn(M, N, device=DEV)
    o32 = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm(A, W, M, N, K, b_major=bm, epilogue=L.EPI_STORE_F32, out0=o32)
    _check(o32, acc, 1e-5, "store_f32")
    o16 = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
    ops.gemm(A, W, M, N, K, b_major=bm, epilogue=L.EPI_STORE_BF16, out0=o16, bias=bias, scale=0.25, scale_cols=N // 2)
    ref = acc + bias
    ref[:, :N // 2] *= 0.25
    _check(o16.float(), ref, 4e-3, "store_bf16")
    ores = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm(A, W, M, N, K, b_major=bm, epilogue=L.EPI_BIAS_RES_F32, out0=ores, bias=bias, aux1=res)
    _check(ores, acc + bias + res, 1e-5, "bias_res")
    pre = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
    act = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
    ops.gemm(A, W, M, N, K, b_major=bm, epilogue=L.EPI_BIAS_GELU, out0=pre, out1=act, bias=bias)
    _check(pre.float(), acc + bias, 4e-3, "gelu.pre")
    _check(act.float(), F.gelu(acc + bias), 4e-3, "gelu.act")
    dg = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
    ops.gemm(A, W, M, N, K, b_major=bm, epilogue=L.EPI_MUL_DGELU, out0=dg, aux1=pre)
    p = pre.float().requires_grad_(True)
    F.gelu(p).sum().backward()
    _check(dg.float(), acc * p.grad, 4e-3, "mul_dgelu")
    # repeatable: two runs of the same call give the same bits
    o2 = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm(A, W, M, N, K, b_major=bm, epilogue=L.EPI_STORE_F32, out0=o2)
    torch.cuda.synchronize()
    assert torch.equal(o2, o32)


def test_gemm_epilogues():
    _check_epilogues(333, 256, 128)


@pytest.mark.parametrize("M,N,K", [(333, 384, 192), (333, 640, 320),   # persistent kernel, q-scale boundary inside a tile
                                   (333, 192, 192), (333, 320, 320)])  # gemm_kernel<64> with several column tiles
def test_gemm_epilogues_inside_tiles(M, N, K):
    _check_epilogues(M, N, K)


def _check_epilogues(M, N, K):
    """Every fprop epilogue against fp32 PyTorch, with the q scale on the first N / 2 columns."""
    ops, L = _ops(), _L()
    A, W = _rand_bf16(M, K, seed=7), _rand_bf16(N, K, seed=8, scale=K ** -0.5)
    bias = torch.randn(N, device=DEV)
    acc = A.float() @ W.float().t()
    # bf16 store with bias and a scale on the first N / 2 columns (the q half of the qk projection)
    out = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
    ops.gemm(A, W, M, N, K, epilogue=L.EPI_STORE_BF16, out0=out, bias=bias, scale=0.25, scale_cols=N // 2)
    ref = acc + bias
    ref[:, :N // 2] *= 0.25
    _check(out.float(), ref, 4e-3, "store_bf16")
    # bias + residual, fp32
    res = torch.randn(M, N, device=DEV)
    out = torch.zeros(M, N, device=DEV)
    ops.gemm(A, W, M, N, K, epilogue=L.EPI_BIAS_RES_F32, out0=out, bias=bias, aux1=res)
    _check(out, acc + bias + res, 1e-5, "bias_res_f32")
    # bias + exact GELU, both pre- and post-activation
    pre = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
    act = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
    ops.gemm(A, W, M, N, K, epilogue=L.EPI_BIAS_GELU, out0=pre, out1=act, bias=bias)
    _check(pre.float(), acc + bias, 4e-3, "gelu.pre")
    _check(act.float(), F.gelu(acc + bias), 4e-3, "gelu.act")
    # multiply by gelu'(pre)
    out = torch.zeros(M, N, dtype=torch.bfloat16, device=DEV)
    ops.gemm(A, W, M, N, K, epilogue=L.EPI_MUL_DGELU, out0=out, aux1=pre)
    p = pre.float().requires_grad_(True)
    F.gelu(p).sum().backward()
    _check(out.float(), acc * p.grad, 4e-3, "mul_dgelu")
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------
# LayerNorm / conversions / reductions
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,C,K", [(128, 128, 256), (300, 128, 512), (1000, 128, 256), (19200, 128, 512),
                                   (153600, 128, 512), (153600, 128, 256), (77, 256, 512), (1000, 256, 1024),
                                   (38400, 256, 1024), (38400, 256, 512)])
@pytest.mark.parametrize("with_res", [True, False])
def test_dgrad_ln_bwd_fused(T, C, K, with_res):
    """d fc1 / d qk GEMM with the LayerNorm backward in its epilogue (csrc/crf_dgrad_lnbwd.cu) against fp32 autograd
    through F.layer_norm on the same bf16-rounded operands, and against the two-kernel path (GEMM, then crf_ln_bwd)."""
    ops, L = _ops(), _L()
    g = torch.Generator(device="cpu").manual_seed(T + C + K)
    x = (torch.randn(T, C, generator=g) * 1.5 + 0.3).to(DEV)
    gam = (1.0 + 0.1 * torch.randn(C, generator=g)).to(DEV)
    bet = torch.zeros(C, device=DEV)
    dy = _rand_bf16(T, K, seed=31)
    W = _rand_bf16(K, C, seed=32, scale=K ** -0.5)
    dres = torch.randn(T, C, generator=g).to(DEV) if with_res else None
    mean = x.mean(1)
    rstd = (x.var(1, unbiased=False) + 1e-5).rsqrt()
    stats = torch.stack([mean, rstd], 1).contiguous()
    dx, dxb, dga, dbe = ops.dgrad_ln_bwd(dy, W, x, stats, gam, dres)
    torch.cuda.synchronize()
    # reference: autograd through layer_norm with upstream gradient g = dy @ W
    gxn = dy.float() @ W.float()
    xr = x.clone().requires_grad_(True)
    gr, br = gam.clone().requires_grad_(True), bet.clone().requires_grad_(True)
    F.layer_norm(xr, (C,), gr, br, 1e-5).backward(gxn)
    ref = xr.grad + (dres if with_res else 0)
    _check(dx, ref, 2e-5, "dgrad_ln_bwd.dx")
    _check(dxb.float(), ref, 4e-3, "dgrad_ln_bwd.dx_bf16")
    _check(dga, gr.grad, 1e-4, "dgrad_ln_bwd.dgamma")
    _check(dbe, br.grad, 1e-4, "dgrad_ln_bwd.dbeta")
    # two-kernel path on the same operands
    gx = torch.empty(T, C, device=DEV)
    ops.gemm(dy, W, T, C, K, a_major=0, b_major=1, epilogue=L.EPI_STORE_F32, out0=gx)
    dx2, dxb2, dga2, dbe2 = ops.ln_bwd(gx, x, stats, gam, dres, want_bf16=True)
    torch.cuda.synchronize()
    _check(dx, dx2, 1e-5, "fused vs two kernels dx")
    _check(dga, dga2, 1e-4, "fused vs two kernels dgamma")
    # only one of the two outputs
    dx3, none16, _, _ = ops.dgrad_ln_bwd(dy, W, x, stats, gam, dres, want_bf16=False)
    none32, dxb3, _, _ = ops.dgrad_ln_bwd(dy, W, x, stats, gam, dres, want_f32=False)
    torch.cuda.synchronize()
    assert none16 is None and none32 is None
    assert torch.equal(dx3, dx) and torch.equal(dxb3, dxb)


@pytest.mark.parametrize("T,C,K", [(38400, 256, 1024), (38400, 256, 512), (153600, 128, 512)])
def test_dgrad_ln_bwd_fused_repeatable(T, C, K):
    """Bit-identical dx over repeated launches: guards the slab-ring hand-over of the fused kernel (a slab released
    before its reads had completed showed up as 4-column glitches in a few rows, in ~1 of 3 launches)."""
    ops = _ops()
    g = torch.Generator(device="cpu").manual_seed(T + C + K)
    x = (torch.randn(T, C, generator=g) * 1.5 + 0.3).to(DEV)
    gam = (1.0 + 0.1 * torch.randn(C, generator=g)).to(DEV)
    dy, W = _rand_bf16(T, K, seed=31), _rand_bf16(K, C, seed=32, scale=K ** -0.5)
    dres = torch.randn(T, C, generator=g).to(DEV)
    stats = torch.stack([x.mean(1), (x.var(1, unbiased=False) + 1e-5).rsqrt()], 1).contiguous()
    dx0, dxb0, _, _ = ops.dgrad_ln_bwd(dy, W, x, stats, gam, dres)
    for i in range(10):
        f32, b16 = (i % 3) != 2, (i % 3) != 1
        dx, dxb, _, _ = ops.dgrad_ln_bwd(dy, W, x, stats, gam, dres, want_f32=f32, want_bf16=b16)
        torch.cuda.synchronize()
        assert dx is None or torch.equal(dx, dx0), f"run {i}: dx differs"
        assert dxb is None or torch.equal(dxb, dxb0), f"run {i}: dx_bf16 differs"


# ---------------------------------------------------------------------------------------------------------
# fused MLP half: LayerNorm-2 -> fc1 -> GELU -> fc2 -> + residual in one kernel (csrc/crf_mlp_fused.cu)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,C", [(128, 128), (300, 128), (1000, 128), (19200, 128), (153600, 128),
                                 (77, 256), (1000, 256), (38400, 256)])
@pytest.mark.parametrize("training", [True, False])
def test_mlp_fused_fwd(T, C, training):
    """y = x1 + fc2(gelu(fc1(LN(x1)))) (newcrf_layers.py:255, :21-27) against fp32 PyTorch on the same bf16-rounded
    weights; the saved tensors (xn2, stats, pre, act) against the same reference and against the stand-alone
    LayerNorm kernel; pre / act / y against the unfused GEMM kernels on the same operands."""
    ops, L = _ops(), _L()
    g = torch.Generator(device="cpu").manual_seed(T + C)
    x1 = (torch.randn(T, C, generator=g) * 1.5 + 0.3).to(DEV)
    gam = (1.0 + 0.1 * torch.randn(C, generator=g)).to(DEV)
    bet = (0.1 * torch.randn(C, generator=g)).to(DEV)
    w1, w2 = _rand_bf16(4 * C, C, seed=3, scale=C ** -0.5), _rand_bf16(C, 4 * C, seed=4, scale=(4 * C) ** -0.5)
    b1 = (0.1 * torch.randn(4 * C, generator=g)).to(DEV)
    b2 = (0.1 * torch.randn(C, generator=g)).to(DEV)
    y, xn2, stats, pre, act = ops.mlp_fwd(x1, gam, bet, w1, b1, w2, b2, eps=1e-5, training=training)
    torch.cuda.synchronize()
    # reference with the kernel's rounding points (xn2 and act are bf16 tensor-core operands)
    xn_ref = F.layer_norm(x1, (C,), gam, bet, 1e-5)
    pre_ref = xn_ref.to(torch.bfloat16).float() @ w1.float().t() + b1
    act_ref = F.gelu(pre_ref)
    y_ref = x1 + act_ref.to(torch.bfloat16).float() @ w2.float().t() + b2
    _check(y, y_ref, 2e-3, "mlp_fused.y")
    assert float((y - y_ref).abs().max()) < 2e-2 * float(y_ref.abs().max()), "mlp_fused.y max-abs"
    # fp32 reference without any bf16 rounding: the bf16-I/O tolerance of the path
    y_f32 = x1 + F.gelu(xn_ref @ w1.float().t() + b1) @ w2.float().t() + b2
    _check(y, y_f32, 6e-3, "mlp_fused.y vs fp32")
    if training:
        _check(xn2.float(), xn_ref, 4e-3, "mlp_fused.xn2")
        _check(pre.float(), pre_ref, 4e-3, "mlp_fused.pre")
        _check(act.float(), act_ref, 5e-3, "mlp_fused.act")
        xn_k, stats_k, _ = ops.ln_fwd(x1.view(1, T, C), gam, bet, 1e-5)
        # the fused prologue sums a row in a different order (8 lanes per row) than the stand-alone kernel (32 lanes):
        # statistics agree to fp32 round-off, the bf16 outputs to one rounding step in a few elements
        _check(stats, stats_k, 1e-6, "mlp_fused.stats vs stand-alone LayerNorm")
        _check(xn2.float(), xn_k.float(), 1e-3, "mlp_fused.xn2 vs stand-alone LayerNorm")
        assert float((xn2 != xn_k).float().mean()) < 0.02, "too many bf16 outputs differ from the stand-alone LayerNorm"
        # the unfused path on the same operands: fc1 (+GELU) and fc2 (+residual) through crf_gemm
        pre_k = torch.empty(T, 4 * C, dtype=torch.bfloat16, device=DEV)
        act_k = torch.empty(T, 4 * C, dtype=torch.bfloat16, device=DEV)
        ops.gemm(xn2, w1, T, 4 * C, C, epilogue=L.EPI_BIAS_GELU, out0=pre_k, out1=act_k, bias=b1)
        y_k = torch.empty(T, C, device=DEV)
        ops.gemm(act_k, w2, T, C, 4 * C, epilogue=L.EPI_BIAS_RES_F32, out0=y_k, bias=b2, aux1=x1)
        torch.cuda.synchronize()
        _check(pre.float(), pre_k.float(), 1e-4, "mlp_fused.pre vs GEMM epilogue")   # same MMA sequence: expected bit-equal
        _check(act.float(), act_k.float(), 1e-4, "mlp_fused.act vs GEMM epilogue")
        _check(y, y_k, 1e-5, "mlp_fused.y vs unfused kernels")   # same products, different K-chunk summation order


LN_WIDTHS = list(range(64, 1025, 64))   # every width the library accepts: one row-kernel instance each


@pytest.mark.parametrize("C", LN_WIDTHS)
@pytest.mark.parametrize("layout", ["nchw_view", "contig", "bf16_nchw"])
def test_ln_fwd(C, layout):
    ops = _ops()
    B, H, W = 2, 9, 10
    g = torch.Generator().manual_seed(C)
    base = torch.randn(B, C, H, W, generator=g).to(DEV) * 2 + 0.5
    if layout == "contig":
        x = base.flatten(2).transpose(1, 2).contiguous()
    elif layout == "bf16_nchw":
        x = base.to(torch.bfloat16).flatten(2).transpose(1, 2)
    else:
        x = base.flatten(2).transpose(1, 2)
    gamma, beta = torch.randn(C, device=DEV), torch.randn(C, device=DEV)
    xn, stats, cp = ops.ln_fwd(x, gamma, beta, 1e-5, want_copy=True)
    torch.cuda.synchronize()
    xf = x.float().reshape(-1, C)
    assert torch.equal(cp, xf.contiguous()), "fp32 copy must be bit-exact"
    ref = F.layer_norm(xf, (C,), gamma, beta, 1e-5)
    _check(xn.float(), ref, 4e-3, "ln_fwd.xn")
    _check(stats[:, 0], xf.mean(-1), 1e-5, "ln_fwd.mean")
    _check(stats[:, 1], (xf.var(-1, unbiased=False) + 1e-5).rsqrt(), 1e-5, "ln_fwd.rstd")


@pytest.mark.parametrize("C", LN_WIDTHS)
def test_ln_bwd(C):
    ops = _ops()
    T = 777
    g = torch.Generator().manual_seed(C + 1)
    x = (torch.randn(T, C, generator=g) * 2 + 0.3).to(DEV).requires_grad_(True)
    gamma = torch.randn(C, generator=g).to(DEV).requires_grad_(True)
    beta = torch.randn(C, generator=g).to(DEV).requires_grad_(True)
    go = torch.randn(T, C, generator=g).to(DEV)
    dres = torch.randn(T, C, generator=g).to(DEV)
    y = F.layer_norm(x, (C,), gamma, beta, 1e-5)
    y.backward(go)
    xd = x.detach()
    stats = torch.stack([xd.mean(-1), (xd.var(-1, unbiased=False) + 1e-5).rsqrt()], dim=1).contiguous()
    dx, dxb, dgamma, dbeta = ops.ln_bwd(go, xd, stats, gamma.detach(), dres, want_bf16=True)
    torch.cuda.synchronize()
    _check(dx, x.grad + dres, 1e-5, "ln_bwd.dx")
    _check(dxb.float(), x.grad + dres, 4e-3, "ln_bwd.dx_bf16")
    _check(dgamma, gamma.grad, 1e-4, "ln_bwd.dgamma")
    _check(dbeta, beta.grad, 1e-4, "ln_bwd.dbeta")


@pytest.mark.parametrize("C", LN_WIDTHS)
@pytest.mark.parametrize("out_bf16", [False, True])
def test_layer_norm_standalone(C, out_bf16):
    """functional.layer_norm (the stage-closing norm_crf, newcrf_layers.py:430-431) vs torch's fp32 LayerNorm:
    forward, dx, dgamma, dbeta; fp32 output within 1e-5, bf16 output / bf16 incoming gradient within 2e-2 (bf16 I/O)."""
    from monocular_depth_estimation_b200 import functional as CF
    torch.manual_seed(C + int(out_bf16))
    dev = torch.device("cuda:0")
    B, T = 3, 331                                   # odd row count: exercises the grid-stride tail
    x = (torch.randn(B, T, C, device=dev) * 1.7 + 0.3).requires_grad_(True)
    w = (1 + 0.2 * torch.randn(C, device=dev)).requires_grad_(True)
    b = (0.1 * torch.randn(C, device=dev)).requires_grad_(True)
    y = CF.layer_norm(x, w, b, 1e-5, out_dtype=torch.bfloat16 if out_bf16 else torch.float32)
    assert y.dtype == (torch.bfloat16 if out_bf16 else torch.float32) and y.shape == x.shape
    gy = torch.randn(B, T, C, device=dev)
    if out_bf16:
        gy = gy.to(torch.bfloat16)
    y.backward(gy)
    xr, wr, br = (t.detach().clone().requires_grad_(True) for t in (x, w, b))
    yr = F.layer_norm(xr, (C,), wr, br, 1e-5)
    yr.backward(gy.float())
    tol = 2e-2 if out_bf16 else 1e-5
    _check(y.float(), yr, tol, "layer_norm y")
    _check(x.grad, xr.grad, 2e-5 if not out_bf16 else 2e-2, "layer_norm dx")
    _check(w.grad, wr.grad, 1e-4, "layer_norm dgamma")
    _check(b.grad, br.grad, 1e-4, "layer_norm dbeta")


@pytest.mark.parametrize("shape", [(2, 1, 37, 53), (1, 1, 2, 2), (3, 1, 3, 5), (2, 1, 120, 160)])
@pytest.mark.parametrize("bf16", [False, True])
def test_depth_loss(shape, bf16):
    """functional.depth_loss (SSIM + 0.1 L1, train.py:94-100 / loss.py:57-88) vs the oracle's composition of torch
    ops evaluated in fp64 on the same (bf16-rounded) prediction: loss value and d loss / d pred."""
    from monocular_depth_estimation_b200 import functional as CF
    from oracle import model_oracle as MO
    torch.manual_seed(sum(shape) + int(bf16))
    dev = torch.device("cuda:0")
    pred = torch.rand(shape, device=dev)
    tgt = (0.5 * pred + 0.5 * torch.rand(shape, device=dev)).clamp(0, 1)
    tgt[..., : shape[-1] // 2] = pred[..., : shape[-1] // 2]      # a region with SSIM ~ 1 (clamp boundary)
    if bf16:
        pred = pred.to(torch.bfloat16)
    pred.requires_grad_(True)
    loss = CF.depth_loss(pred, tgt)
    loss.backward()
    pr = pred.detach().double().cpu().requires_grad_(True)
    lr = MO.ssim_l1_loss(pr, tgt.double().cpu())
    lr.backward()
    assert abs(float(loss) - float(lr)) < 2e-5 * max(1.0, abs(float(lr))), (float(loss), float(lr))
    assert pred.grad.dtype == pred.dtype
    _check(pred.grad.float().reshape(-1, shape[-1]), pr.grad.float().reshape(-1, shape[-1]), 1e-2 if bf16 else 2e-4,
           "depth_loss d pred")


@pytest.mark.parametrize("shape", [(2, 256, 6, 5), (1, 1024, 3, 4), (2, 12, 5, 7), (8, 256, 60, 80)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pixel_shuffle_nhwc_bit_exact(shape, dtype):
    """functional.pixel_shuffle2 on channels-last tensors == F.pixel_shuffle(x, 2), forward and backward, bit-exact
    (a pure permutation: model_mobileV3_large_newCRFs.py:116-120)."""
    from monocular_depth_estimation_b200 import functional as CF
    torch.manual_seed(sum(shape))
    x = torch.randn(shape, device="cuda:0").to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y = CF.pixel_shuffle2(x)
    ref = F.pixel_shuffle(x.detach(), 2)
    assert y.shape == ref.shape and y.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(y, ref)
    g = torch.randn_like(ref)
    y.backward(g)
    assert torch.equal(x.grad, F.pixel_unshuffle(g, 2))


def test_depth_loss_matches_reference_golden():
    """The fused loss kernels against the golden value / gradient of the unmodified reference loss."""
    from monocular_depth_estimation_b200 import functional as CF
    g = load_golden("loss_ssim_l1")
    for tag in ("a", "b", "c"):
        pred = torch.from_numpy(g[f"pred.{tag}"]).to(DEV).requires_grad_(True)
        val = CF.depth_loss(pred, torch.from_numpy(g[f"target.{tag}"]).to(DEV))
        val.backward()
        assert abs(float(val.detach()) - float(g[f"loss.{tag}"][0])) < 2e-5
        _check(pred.grad.reshape(-1, pred.shape[-1]), torch.from_numpy(g[f"dpred.{tag}"]).to(DEV).reshape(-1, pred.shape[-1]),
               2e-4, f"depth_loss d pred ({tag})")


@pytest.mark.parametrize("B,H,W,C", [(2, 5, 7, 64), (2, 15, 20, 1024), (8, 30, 40, 512), (3, 9, 11, 256), (1, 1, 1, 128),
                                     (2, 9, 10, 192), (1, 15, 20, 320), (3, 7, 11, 640), (2, 5, 13, 960)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("aligned", [True, False])
def test_layernorm_pixel_shuffle_fused(B, H, W, C, dtype, aligned):
    """The closing LayerNorm of a decoder stage with the following nn.PixelShuffle(2) folded into its store / load
    (crf_layernorm_ps_fwd / _bwd; model_mobileV3_large_newCRFs.py:116-120): bit-identical to LayerNorm kernel +
    F.pixel_shuffle, forward and backward.  aligned=False hands both backward calls dgamma / dbeta views 4 bytes into
    a larger buffer, which takes the kernels' scalar-atomic path in place of the 16-byte vector reduction."""
    import ctypes as Cc
    L = _L()
    lib = L.lib()
    g = torch.Generator(device="cpu").manual_seed(B * H * W + C)
    T = B * H * W
    x = (torch.randn(T, C, generator=g) * 1.3 + 0.2).to(DEV)
    gam = (1.0 + 0.1 * torch.randn(C, generator=g)).to(DEV)
    bet = (0.1 * torch.randn(C, generator=g)).to(DEV)
    st = Cc.c_void_p(torch.cuda.current_stream().cuda_stream)
    dt = L.CRF_DT_BF16 if dtype == torch.bfloat16 else L.CRF_DT_F32
    # forward
    y_ps = torch.full((B, 2 * H, 2 * W, C // 4), float("nan"), dtype=dtype, device=DEV)
    stats = torch.empty(T, 2, device=DEV)
    L.check(lib.crf_layernorm_ps_fwd(x.data_ptr(), gam.data_ptr(), bet.data_ptr(), 1e-5, y_ps.data_ptr(), dt,
                                     stats.data_ptr(), B, H, W, C, 0, st), "crf_layernorm_ps_fwd")
    y = torch.empty(T, C, dtype=dtype, device=DEV)
    stats2 = torch.empty(T, 2, device=DEV)
    L.check(lib.crf_layernorm_fwd(x.data_ptr(), gam.data_ptr(), bet.data_ptr(), 1e-5, y.data_ptr(), dt, stats2.data_ptr(),
                                  T, C, 0, st), "crf_layernorm_fwd")
    torch.cuda.synchronize()
    ref = F.pixel_shuffle(y.view(B, H, W, C).permute(0, 3, 1, 2), 2)          # (B, C/4, 2H, 2W)
    assert torch.equal(y_ps.permute(0, 3, 1, 2), ref)
    assert torch.equal(stats, stats2)
    _check(y_ps.permute(0, 3, 1, 2).float(), F.pixel_shuffle(
        F.layer_norm(x, (C,), gam, bet, 1e-5).view(B, H, W, C).permute(0, 3, 1, 2), 2), 4e-3 if dtype == torch.bfloat16 else 1e-5,
        "layernorm_ps.y")
    # backward
    gy = torch.randn(B, 2 * H, 2 * W, C // 4, generator=g).to(DEV).to(dtype)        # NHWC gradient of the shuffled map
    def zeros_c(aligned):
        return torch.zeros(C, device=DEV) if aligned else torch.zeros(C + 4, device=DEV)[1:C + 1]

    dx = torch.full((T, C), float("nan"), device=DEV)
    dgam, dbet = zeros_c(aligned), zeros_c(aligned)
    L.check(lib.crf_layernorm_ps_bwd(gy.data_ptr(), dt, x.data_ptr(), stats.data_ptr(), gam.data_ptr(), dx.data_ptr(),
                                     dgam.data_ptr(), dbet.data_ptr(), B, H, W, C, 0, st), "crf_layernorm_ps_bwd")
    g_tok = F.pixel_unshuffle(gy.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1).reshape(T, C).contiguous()

    def layernorm_bwd(aligned):
        dx2 = torch.empty(T, C, device=DEV)
        dgam2, dbet2 = zeros_c(aligned), zeros_c(aligned)
        L.check(lib.crf_layernorm_bwd(g_tok.data_ptr(), dt, x.data_ptr(), stats.data_ptr(), gam.data_ptr(),
                                      dx2.data_ptr(), dgam2.data_ptr(), dbet2.data_ptr(), T, C, 0, st), "crf_layernorm_bwd")
        return dx2, dgam2, dbet2

    dx2, dgam2, dbet2 = layernorm_bwd(aligned)
    torch.cuda.synchronize()
    assert torch.equal(dx, dx2)
    _check(dgam, dgam2, 1e-5, "layernorm_ps.dgamma")
    _check(dbet, dbet2, 1e-5, "layernorm_ps.dbeta")
    if not aligned:  # the scalar-atomic path against the vector reduction
        _, dgam3, dbet3 = layernorm_bwd(True)
        torch.cuda.synchronize()
        for got, what in ((dgam, "layernorm_ps.dgamma"), (dgam2, "layernorm.dgamma")):
            _check(got, dgam3, 1e-5, what + " (unaligned)")
        for got, what in ((dbet, "layernorm_ps.dbeta"), (dbet2, "layernorm.dbeta")):
            _check(got, dbet3, 1e-5, what + " (unaligned)")


def test_colsum_cast_convert():
    ops = _ops()
    for T_, N_ in ((1234, 384), (7, 8), (153600, 128), (38400, 256), (9600, 512), (2401, 1024), (333, 4096)):
        gq = _rand_bf16(T_, N_, seed=11)
        _check(ops.colsum_bf16(gq), gq.float().sum(0), 1e-5, f"colsum {T_}x{N_}")
    src = torch.randn(100003, device=DEV)
    assert torch.equal(ops.cast_bf16(src), src.to(torch.bfloat16))
    v = torch.randn(2, 128, 9, 10, device=DEV).permute(0, 2, 3, 1)  # NCHW view, like newcrf_layers.py:427
    assert torch.equal(ops.convert_v(v), v.reshape(-1, 128).to(torch.bfloat16))
    for Cv in (64, 192, 960):
        v2 = torch.randn(2, 9, 10, Cv, device=DEV)
        assert torch.equal(ops.convert_v(v2), v2.reshape(-1, Cv).to(torch.bfloat16)), Cv
    for Cv in (192, 960):   # NCHW view: the transposing kernel, C / 256 not whole
        v3 = torch.randn(2, Cv, 9, 10, device=DEV).permute(0, 2, 3, 1)
        assert torch.equal(ops.convert_v(v3), v3.reshape(-1, Cv).to(torch.bfloat16)), Cv
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------
# bit-exact index maps against the reference's own outputs (golden) and the oracle
# ---------------------------------------------------------------------------------------------------------
def test_window_index_maps_bit_exact():
    ops = _ops()
    g = load_golden("index_maps")
    for H, W, s in g["cases"]:
        H, W, s = int(H), int(W), int(s)
        tag = f"{H}x{W}s{s}"
        x = torch.arange(1, 2 * H * W * 3 + 1, dtype=torch.float32).reshape(2, H, W, 3).to(DEV)
        win = ops.window_gather(x, 7, s)
        assert np.array_equal(win.cpu().numpy(), g["gather." + tag]), tag
        wv = torch.arange(1, win.numel() + 1, dtype=torch.float32).reshape(win.shape).to(DEV)
        back = ops.window_scatter(wv, 2, H, W, 7, s)
        assert np.array_equal(back.cpu().numpy(), g["scatter." + tag]), tag
        if s == 3:
            assert np.array_equal(ops.shift_mask(H, W, 7, s, DEV).cpu().numpy(), g["mask." + tag]), tag
    # a large, padded, shifted case against the oracle (decoder scale 1/4 of a 480x640 input)
    x = torch.randn(2, 120, 160, 8, device=DEV)
    for s in (0, 3):
        assert torch.equal(ops.window_gather(x, 7, s), O.window_gather(x, 7, s))
        w = torch.randn(2 * 414, 49, 8, device=DEV)
        assert torch.equal(ops.window_scatter(w, 2, 120, 160, 7, s), O.window_scatter(w, 2, 120, 160, 7, s))
    assert np.array_equal(ops.shift_mask(120, 160, 7, 3, DEV).cpu().numpy(), O.shift_mask(120, 160, 7, 3))


# ---------------------------------------------------------------------------------------------------------
# window-attention core
# ---------------------------------------------------------------------------------------------------------
def _attn_reference(qk, vb, qk_bias, table, B, H, W, C, nH, shift):
    """fp32 reference of the attention core on the same bf16-rounded q/k/v, including the zero-pad-token rule
    (k of a pad token = bias, v = 0) and the shift mask.  Differentiable w.r.t. qk, vb, table, qk_bias."""
    N, hd = 49, C // nH
    q = qk[:, :C].reshape(B, H, W, C)
    k = qk[:, C:].reshape(B, H, W, C)
    src = torch.from_numpy(O.window_source_index(H, W, 7, shift)).to(qk.device)
    pad = (src < 0).reshape(1, -1, N, 1)
    qw = O.window_gather(q, 7, shift)
    kw = O.window_gather(k, 7, shift)
    vw = O.window_gather(vb.reshape(B, H, W, C), 7, shift)
    nW = src.shape[0]
    kb = qk_bias[C:].to(torch.bfloat16).float() if not qk_bias.requires_grad else qk_bias[C:]
    kw = torch.where(pad.expand(B, nW, N, C).reshape(B * nW, N, C), kb.expand(B * nW, N, C), kw)
    qh = qw.reshape(-1, N, nH, hd).transpose(1, 2)
    kh = kw.reshape(-1, N, nH, hd).transpose(1, 2)
    vh = vw.reshape(-1, N, nH, hd).transpose(1, 2)
    attn = qh @ kh.transpose(-2, -1)
    idx = torch.from_numpy(O.relative_position_index(7)).to(qk.device)
    attn = attn + table[idx.reshape(-1)].reshape(N, N, nH).permute(2, 0, 1).unsqueeze(0)
    if shift > 0:
        m = torch.from_numpy(O.shift_mask(H, W, 7, shift)).to(qk.device)
        attn = (attn.reshape(B, nW, nH, N, N) + m[None, :, None]).reshape(-1, nH, N, N)
    lse = torch.logsumexp(attn, dim=-1)
    p = torch.softmax(attn, dim=-1)
    ow = (p @ vh).transpose(1, 2).reshape(-1, N, C)
    return O.window_scatter(ow, B, H, W, 7, shift).reshape(-1, C), lse


ATTN_CASES = [(1, 7, 7, 64, 2, 0), (1, 14, 14, 64, 2, 0), (2, 9, 10, 64, 2, 0), (2, 9, 10, 64, 2, 3),
              (1, 15, 20, 128, 4, 3), (3, 30, 40, 128, 4, 3), (2, 15, 20, 256, 8, 0), (1, 21, 16, 1024, 32, 3),
              (2, 9, 10, 64, 4, 3), (1, 15, 20, 128, 8, 0),   # these two: head_dim 16
              # head counts that are not powers of two: head_dim 32 at C = 192 / 320, head_dim 16 at C = 192
              (2, 9, 10, 192, 6, 3), (1, 15, 20, 320, 10, 3), (2, 9, 10, 192, 12, 3)]


@pytest.mark.parametrize("B,H,W,C,nH,shift", ATTN_CASES)
def test_attn_fwd(B, H, W, C, nH, shift):
    ops = _ops()
    T = B * H * W
    qk = _rand_bf16(T, 2 * C, seed=21, scale=0.7)
    vb = _rand_bf16(T, C, seed=22)
    qk_bias = torch.randn(2 * C, device=DEV) * 0.5
    table = torch.randn(169, nH, device=DEV) * 0.5
    d = ops.make_desc(B, H, W, C, nH, shift, device=torch.cuda.current_device())
    o, lse = ops.attn_fwd(d, qk, vb, qk_bias, (C // nH) ** -0.5, table)
    torch.cuda.synchronize()
    ref_o, ref_lse = _attn_reference(qk.float(), vb.float(), qk_bias, table, B, H, W, C, nH, shift)
    _check(o.float(), ref_o, 1e-2, "attn_fwd.o")
    _check(lse[:, :, :49], ref_lse, 1e-4, "attn_fwd.lse")


# head_dim 64 / 128 (crf_attn_wide.cu; BASELINE.json configs[2])
WIDE_CASES = [(1, 7, 7, 64, 1, 0), (2, 9, 10, 64, 1, 3), (1, 14, 14, 128, 2, 0), (1, 15, 20, 128, 1, 3),
              (3, 30, 40, 256, 4, 3), (2, 15, 20, 256, 2, 0), (1, 21, 16, 512, 4, 3), (2, 23, 17, 512, 8, 3),
              # odd head counts: head_dim 64 at C = 192 / 320 / 960, head_dim 128 at C = 384 / 640 / 896
              (2, 9, 10, 192, 3, 3), (1, 15, 20, 320, 5, 3), (1, 15, 20, 960, 15, 3),
              (2, 9, 10, 384, 3, 3), (1, 15, 20, 640, 5, 3), (1, 15, 20, 896, 7, 3)]


@pytest.mark.parametrize("B,H,W,C,nH,shift", WIDE_CASES)
def test_attn_fwd_wide(B, H, W, C, nH, shift):
    test_attn_fwd(B, H, W, C, nH, shift)


@pytest.mark.parametrize("B,H,W,C,nH,shift", WIDE_CASES)
def test_attn_bwd_wide(B, H, W, C, nH, shift):
    test_attn_bwd(B, H, W, C, nH, shift)


@pytest.mark.parametrize("B,H,W,C,nH,shift", [(8, 120, 160, 128, 4, 3), (8, 30, 40, 512, 16, 3), (2, 23, 17, 64, 2, 3)])
def test_attn_repeatable(B, H, W, C, nH, shift):
    """Race hunt for the asynchronous attention pipeline (hardware-made mbarrier arrivals, two MMA-issuing warps,
    accumulator pre-load, transposed stores): every output that involves no floating-point atomics must be bit-identical
    over repeated launches at the full config-2 shape, and untouched by other work running between the launches."""
    ops = _ops()
    T = B * H * W
    qk = _rand_bf16(T, 2 * C, seed=31, scale=0.7)
    vb = _rand_bf16(T, C, seed=32)
    dout = _rand_bf16(T, C, seed=33)
    qk_bias = torch.randn(2 * C, device=DEV) * 0.5
    table = torch.randn(169, nH, device=DEV) * 0.5
    d = ops.make_desc(B, H, W, C, nH, shift, device=torch.cuda.current_device())
    scale = (C // nH) ** -0.5
    o0, lse0 = ops.attn_fwd(d, qk, vb, qk_bias, scale, table)
    dqk0, dv0, dt0, db0 = ops.attn_bwd(d, qk, vb, qk_bias, scale, table, lse0, dout)
    junk = torch.empty(64 << 20, device=DEV)
    for it in range(6):
        junk.normal_()                                    # evict L2, perturb timing
        o, lse = ops.attn_fwd(d, qk, vb, qk_bias, scale, table)
        dqk, dv, dt, db = ops.attn_bwd(d, qk, vb, qk_bias, scale, table, lse, dout)
        assert torch.equal(o, o0) and torch.equal(lse, lse0), f"forward differs on repeat {it}"
        assert torch.equal(dqk, dqk0) and torch.equal(dv, dv0), f"backward differs on repeat {it}"
        _check(dt, dt0, 1e-5, "d_table (atomics: order-dependent rounding only)")
        _check(db, db0, 1e-5, "d_qk_bias (atomics: order-dependent rounding only)")


@pytest.mark.parametrize("B,H,W,C,nH,shift", ATTN_CASES)
def test_attn_bwd(B, H, W, C, nH, shift):
    ops = _ops()
    T = B * H * W
    qk = _rand_bf16(T, 2 * C, seed=31, scale=0.7)
    vb = _rand_bf16(T, C, seed=32)
    dout = _rand_bf16(T, C, seed=33)
    qk_bias = (torch.randn(2 * C, device=DEV) * 0.5).to(torch.bfloat16).float()
    table = torch.randn(169, nH, device=DEV) * 0.5
    scale = (C // nH) ** -0.5
    d = ops.make_desc(B, H, W, C, nH, shift, device=torch.cuda.current_device())
    o, lse = ops.attn_fwd(d, qk, vb, qk_bias, scale, table)
    dqk, dv, d_table, d_bias = ops.attn_bwd(d, qk, vb, qk_bias, scale, table, lse, dout)
    torch.cuda.synchronize()
    qk_r = qk.float().requires_grad_(True)
    vb_r = vb.float().requires_grad_(True)
    tb_r = table.clone().requires_grad_(True)
    bs_r = qk_bias.clone().requires_grad_(True)
    ref_o, _ = _attn_reference(qk_r, vb_r, bs_r, tb_r, B, H, W, C, nH, shift)
    ref_o.backward(dout.float())
    ref_dqk = qk_r.grad.clone()
    ref_dqk[:, :C] *= scale  # the kernel returns d(pre-scale q): q was stored pre-multiplied by scale
    _check(dv, vb_r.grad, 1e-2, "attn_bwd.dv")
    _check(dqk.float()[:, C:], ref_dqk[:, C:], 1.5e-2, "attn_bwd.dk")
    _check(dqk.float()[:, :C], ref_dqk[:, :C], 1.5e-2, "attn_bwd.dq")
    _check(d_table, tb_r.grad, 1.5e-2, "attn_bwd.d_table")
    if bs_r.grad[C:].abs().max() > 0:
        _check(d_bias[C:], bs_r.grad[C:], 1.5e-2, "attn_bwd.d_bias_k")
    assert d_bias[:C].abs().max() == 0


def test_lib_adam_matches_torch_adam():
    """training.LibAdam (crf_adam_step: one launch for all tensors, device-side step counter) against torch.optim.Adam
    on identical parameters / gradients over several steps, including odd sizes, an unaligned view and a state_dict
    round trip into torch's optimizer."""
    from monocular_depth_estimation_b200.training import LibAdam
    torch.manual_seed(0)
    shapes = [(1,), (3,), (169, 4), (128, 128), (512, 128), (16385,), (1024, 1031), (7, 5, 3)]
    base = torch.randn(40, device=DEV)
    ours = [torch.nn.Parameter(torch.randn(s, device=DEV)) for s in shapes]
    ours.append(torch.nn.Parameter(base[1:34]))                    # 4-byte-aligned view: scalar path
    # dense but not "contiguous": channels-last convolution weights (3x3, and 1x1 whose size-1 strides are arbitrary)
    ours.append(torch.nn.Parameter(torch.randn(16, 8, 3, 3, device=DEV).contiguous(memory_format=torch.channels_last)))
    ours.append(torch.nn.Parameter(torch.randn(24, 40, 1, 1, device=DEV).contiguous(memory_format=torch.channels_last)))
    ref = [torch.nn.Parameter(p.detach().clone()) for p in ours]
    oa = LibAdam(ours, lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    ob = torch.optim.Adam(ref, lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    for step in range(6):
        for k, (a, b) in enumerate(zip(ours, ref)):
            g = torch.randn_like(a) * (10.0 ** (step - 3))
            a.grad, b.grad = g.clone(), g.clone()
            if a.dim() == 4 and step % 2 == 1:   # a gradient laid out differently from its parameter is re-laid out
                a.grad = g.contiguous().clone()
        oa.step()
        ob.step()
    torch.cuda.synchronize()
    for a, b in zip(ours, ref):
        assert (a - b).abs().max() <= 3e-7 * max(1.0, float(b.abs().max())), a.shape
        _check(oa.state[a]["exp_avg"], ob.state[b]["exp_avg"], 1e-5, "exp_avg")
        _check(oa.state[a]["exp_avg_sq"], ob.state[b]["exp_avg_sq"], 1e-5, "exp_avg_sq")
    assert float(oa.state[ours[0]]["step"]) == 6.0
    # torch's optimizer accepts our state (same layout), and ours accepts torch's
    sd = oa.state_dict()
    steps = [st["step"] for st in sd["state"].values()]
    assert all(not s.is_cuda and float(s) == 6.0 for s in steps)                       # torch's layout: CPU scalars ...
    assert len({s.data_ptr() for s in steps}) == len(steps)                             # ... one per parameter, no aliases
    assert all("_step" not in grp for grp in sd["param_groups"])
    ob2 = torch.optim.Adam(ref, lr=1e-3)
    ob2.load_state_dict(sd)
    for b in ref:
        b.grad = torch.ones_like(b)
    ob2.step()                                                                          # torch advances each step by ONE
    assert all(float(ob2.state[b]["step"]) == 7.0 for b in ref)
    oa2 = LibAdam(ours, lr=1e-3)
    oa2.load_state_dict(ob.state_dict())
    for a in ours:
        a.grad = torch.ones_like(a)
    oa2.step()
    torch.cuda.synchronize()
    assert float(oa2.state[ours[0]]["step"]) == 7.0


def test_prefetch_loader_cuda():
    """training.prefetch_to_device: same samples, same order, on the device (channels-last images), copies overlapped."""
    from monocular_depth_estimation_b200 import training as TR
    host = list(TR.synthetic_batches(4, 2, 32, 48, seed=3))
    got = list(TR.prefetch_to_device(iter(host), DEV, memory_format=torch.channels_last))
    torch.cuda.synchronize()
    assert len(got) == 4
    for h, g in zip(host, got):
        assert g["image"].is_cuda and g["image"].is_contiguous(memory_format=torch.channels_last)
        assert torch.equal(g["image"].cpu(), h["image"]) and torch.equal(g["depth"].cpu(), h["depth"])
