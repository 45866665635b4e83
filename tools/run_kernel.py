"""Launch individual kernels of the library at BASELINE config-2 shapes (for ncu captures and quick timing).

    python tools/run_kernel.py attn --stage 0 --iters 3
    python tools/run_kernel.py block --stage 0          # one CRFBlock fwd+bwd
Development / profiling tool; prints CUDA-event timings per call."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from monocular_depth_estimation_b200 import _lib as L  # noqa: E402
from monocular_depth_estimation_b200 import ops  # noqa: E402

STAGES = {0: (120, 160, 128, 4), 1: (60, 80, 256, 8), 2: (30, 40, 512, 16), 3: (15, 20, 1024, 32)}


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["attn", "block", "gemm", "gemms", "mlp", "lnbwd", "misc"])
    ap.add_argument("--infer", action="store_true", help="mlp: inference mode (no saved tensors)")
    ap.add_argument("--stage", type=int, default=0)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--shift", type=int, default=3)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--only", default="", help="gemms: run only the shape with this label (e.g. \"d_fc2*gelu'\")")
    a = ap.parse_args()
    H, W, C, nH = STAGES[a.stage]
    B, dev = a.batch, torch.device("cuda:0")
    T = B * H * W
    torch.manual_seed(0)
    if a.what == "mlp":   # fused LN2 + fc1 + GELU + fc2 + residual (csrc/crf_mlp_fused.cu); ops.mlp_fwd allocates outputs
        x1 = torch.randn(T, C, device=dev)
        gam, bet = torch.ones(C, device=dev), torch.zeros(C, device=dev)
        w1 = (torch.randn(4 * C, C, device=dev) * C ** -0.5).to(torch.bfloat16)
        w2 = (torch.randn(C, 4 * C, device=dev) * (4 * C) ** -0.5).to(torch.bfloat16)
        b1, b2 = torch.zeros(4 * C, device=dev), torch.zeros(C, device=dev)
        import ctypes as Cc
        y = torch.empty(T, C, device=dev)
        xn2 = torch.empty(T, C, dtype=torch.bfloat16, device=dev)
        stats = torch.empty(T, 2, device=dev)
        pre = torch.empty(T, 4 * C, dtype=torch.bfloat16, device=dev)
        act = torch.empty(T, 4 * C, dtype=torch.bfloat16, device=dev)
        m = L.MlpArgs()
        m.x1, m.y, m.w1_bf16, m.w2_bf16 = x1.data_ptr(), y.data_ptr(), w1.data_ptr(), w2.data_ptr()
        m.b1, m.b2, m.norm_w, m.norm_b = b1.data_ptr(), b2.data_ptr(), gam.data_ptr(), bet.data_ptr()
        m.xn2, m.stats, m.pre, m.act = xn2.data_ptr(), stats.data_ptr(), pre.data_ptr(), act.data_ptr()
        m.eps, m.T, m.C, m.training, m.device = 1e-5, T, C, 0 if a.infer else 1, 0
        st = Cc.c_void_p(torch.cuda.current_stream().cuda_stream)
        run = lambda: L.check(L.lib().crf_mlp_fwd(Cc.byref(m), st), "crf_mlp_fwd")
        ms = timed(run, a.iters)
        byt = T * C * (8 + (0 if a.infer else 18))
        if os.environ.get("CRF_MLP_PROF") == "1":   # debug timeline of CTA 0 (csrc/crf_mlp_fused.cu MLP_PROF)
            EV, CH = 16, 96
            buf = (Cc.c_longlong * (EV * CH))()
            L.lib().crf_debug_mlp_prof.argtypes = [Cc.POINTER(Cc.c_longlong), Cc.c_int]
            L.lib().crf_debug_mlp_prof(buf, EV * CH)
            t = [[buf[e * CH + c] for c in range(CH)] for e in range(EV)]
            t00 = min(v for row in t for v in row if v > 0)
            names = ["fc1_beg", "fc1_end", "g_pre", "g_math", "g_wait", "g_arr", "fc2_act", "fc2_w2", "fc2_end", "w1_ld", "w2_ld"]
            print("chunk " + " ".join(f"{n:>8s}" for n in names))
            for c in range(40):
                print(f"{c:5d} " + " ".join(f"{(t[e][c] - t00) if t[e][c] else -1:8d}" for e in range(11)))
            print("tile   ln_beg   ln_end  fin_beg  fin_end")
            for c in range(6):
                print(f"{c:4d} " + " ".join(f"{(t[e][c] - t00) if t[e][c] else -1:8d}" for e in (11, 12, 13, 14)))
        print(f"mlp_fused T={T} C={C} {'infer' if a.infer else 'train'}: {ms * 1e3:.1f} us, "
              f"{16.0 * T * C * C / ms / 1e9:.1f} TFLOP/s, {byt / ms / 1e6:.0f} GB/s")
    elif a.what == "attn":
        qk = (torch.randn(T, 2 * C, device=dev) * 0.7).to(torch.bfloat16)
        vb = torch.randn(T, C, device=dev).to(torch.bfloat16)
        dout = torch.randn(T, C, device=dev).to(torch.bfloat16)
        bias = torch.randn(2 * C, device=dev) * 0.5
        table = torch.randn(169, nH, device=dev) * 0.5
        d = ops.make_desc(B, H, W, C, nH, a.shift, device=0)
        o, lse = ops.attn_fwd(d, qk, vb, bias, 32 ** -0.5, table)
        print("attn_fwd ms", timed(lambda: ops.attn_fwd(d, qk, vb, bias, 32 ** -0.5, table), a.iters))
        print("attn_bwd ms", timed(lambda: ops.attn_bwd(d, qk, vb, bias, 32 ** -0.5, table, lse, dout), a.iters))
    elif a.what == "block":
        from monocular_depth_estimation_b200 import CRFBlock
        blk = CRFBlock(C, nH, C, shift_size=a.shift).to(dev)
        blk.H, blk.W = H, W
        x = torch.randn(B, C, H, W, device=dev).flatten(2).transpose(1, 2).requires_grad_(True)
        v = torch.randn(B, C, H, W, device=dev).permute(0, 2, 3, 1).requires_grad_(True)

        def step():
            y = blk(x, v, None)
            y.backward(torch.ones_like(y))
        print("block fwd+bwd ms", timed(step, a.iters))
    elif a.what == "misc":
        # the memory-bound helpers of a stage: LayerNorm backward, conv-bias column sums, weight casts
        g = torch.randn(T, C, device=dev)
        xx = torch.randn(T, C, device=dev)
        stats = torch.stack([xx.mean(1), (xx.var(1, unbiased=False) + 1e-5).rsqrt()], 1).contiguous()
        gam = torch.ones(C, device=dev)
        dres = torch.randn(T, C, device=dev)
        ms = timed(lambda: ops.ln_bwd(g, xx, stats, gam, dres, want_bf16=True), a.iters)
        print(f"ln_bwd  T{T} C{C}: {ms*1e3:7.1f} us  {T*C*18/ms/1e6:7.0f} GB/s")
        gb = torch.randn(T, C, device=dev).to(torch.bfloat16)
        ms = timed(lambda: ops.colsum_bf16(gb), a.iters)
        print(f"colsum  T{T} N{C}: {ms*1e3:7.1f} us  {T*C*2/ms/1e6:7.0f} GB/s")
        w = torch.randn(11 * C * C, device=dev)
        ms = timed(lambda: ops.cast_bf16(w), a.iters)
        print(f"cast    n{w.numel()}: {ms*1e3:7.1f} us  {w.numel()*6/ms/1e6:7.0f} GB/s")
    elif a.what == "lnbwd":
        # d fc1 / d qk + LayerNorm backward: fused kernel against the GEMM + ln_bwd pair
        for name, K in (("d_fc1+LN2'", 4 * C), ("d_qk+LN1'", 2 * C)):
            dy = torch.randn(T, K, device=dev).to(torch.bfloat16)
            Wt = (torch.randn(K, C, device=dev) * K ** -0.5).to(torch.bfloat16)
            xx = torch.randn(T, C, device=dev)
            stats = torch.stack([xx.mean(1), (xx.var(1, unbiased=False) + 1e-5).rsqrt()], 1).contiguous()
            gam = torch.ones(C, device=dev)
            dres = torch.randn(T, C, device=dev)
            gx = torch.empty(T, C, device=dev)
            ms_f = timed(lambda: ops.dgrad_ln_bwd(dy, Wt, xx, stats, gam, dres), a.iters)

            def two():
                ops.gemm(dy, Wt, T, C, K, a_major=0, b_major=1, epilogue=L.EPI_STORE_F32, out0=gx)
                ops.ln_bwd(gx, xx, stats, gam, dres, want_bf16=True)
            ms_2 = timed(two, a.iters)
            mb = T * (2.0 * K + 14.0 * C) / 1e6
            print(f"{name:12s} T{T} C{C} K{K}: fused {ms_f*1e3:7.1f} us ({mb/ms_f/1e3:6.0f} GB/s on {mb:.0f} MB)   "
                  f"GEMM + ln_bwd {ms_2*1e3:7.1f} us")
    elif a.what == "gemms":
        # every fprop / dgrad projection shape of this stage: (label, M, N, K, b_major, epilogue)
        shapes = [("qk", T, 2 * C, C, 0, L.EPI_STORE_BF16), ("proj+res", T, C, C, 0, L.EPI_BIAS_RES_F32),
                  ("fc1+gelu", T, 4 * C, C, 0, L.EPI_BIAS_GELU), ("fc2+res", T, C, 4 * C, 0, L.EPI_BIAS_RES_F32),
                  ("d_fc2*gelu'", T, 4 * C, C, 1, L.EPI_MUL_DGELU), ("d_fc1", T, C, 4 * C, 1, L.EPI_STORE_F32),
                  ("d_proj", T, C, C, 1, L.EPI_STORE_BF16), ("d_qk", T, C, 2 * C, 1, L.EPI_STORE_F32)]
        for name, M, N, K, bmaj, epi in shapes:
            if a.only and name != a.only:
                continue
            A = torch.randn(M, K, device=dev).to(torch.bfloat16)
            Wt = (torch.randn(K, N, device=dev) if bmaj else torch.randn(N, K, device=dev)).to(torch.bfloat16)
            f32 = epi in (L.EPI_STORE_F32, L.EPI_BIAS_RES_F32)
            out0 = torch.empty(M, N, device=dev, dtype=torch.float32 if f32 else torch.bfloat16)
            out1 = torch.empty(M, N, device=dev, dtype=torch.bfloat16) if epi == L.EPI_BIAS_GELU else None
            aux = (torch.randn(M, N, device=dev) if epi == L.EPI_BIAS_RES_F32 else
                   torch.randn(M, N, device=dev).to(torch.bfloat16) if epi == L.EPI_MUL_DGELU else None)
            bias = torch.randn(N, device=dev) if not bmaj else None
            ms = timed(lambda: ops.gemm(A, Wt, M, N, K, b_major=bmaj, epilogue=epi, out0=out0, out1=out1, bias=bias,
                                        aux1=aux), a.iters)
            print(f"{name:12s} M{M} N{N} K{K}: {ms*1e3:8.1f} us  {2.0*M*N*K/ms/1e9:7.1f} TFLOP/s")
    else:
        M, N, K = T, 4 * C, C
        A = torch.randn(M, K, device=dev).to(torch.bfloat16)
        Wt = torch.randn(N, K, device=dev).to(torch.bfloat16)
        pre = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        act = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
        bias = torch.randn(N, device=dev)
        print("fc1+gelu ms", timed(lambda: ops.gemm(A, Wt, M, N, K, epilogue=L.EPI_BIAS_GELU, out0=pre, out1=act,
                                                     bias=bias), a.iters))


if __name__ == "__main__":
    main()
