"""Per-layer timing of the encoder's 15 depthwise convolutions: forward + backward (input and weight gradient) of one
layer at batch 8 and the bench resolution (480 x 640) under bf16 autocast, each captured in a CUDA graph and replayed,
library (DepthwiseConv2d) against torch (nn.Conv2d on cuDNN, with autocast's weight cast).  Prints one line per layer,
and with --out FILE also writes them as JSON.

Bytes and flops are algorithmic: each of the three passes moves 2 (in + out) bytes per channel and pixel (bf16 x or dy
read, y or dx written, or x and dy read) and does k^2 FMAs per output element.  The share of peak is against the larger
of the HBM bound (bench.py's HBM figure) and the CUDA-core fp32 FMA bound (SMs x 128 FMA/clock at --sm-clock-mhz).
Inputs up to about 100 MB stay partly in the 126 MB L2 between replays, so the smaller layers can exceed the HBM rate."""
import argparse
import json
import os
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import load_peaks  # noqa: E402
from tools.bench_batchnorm import graph_time_us  # noqa: E402
from monocular_depth_estimation_b200.model import DepthwiseConv2d, fuse_depthwise  # noqa: E402


def layer_shapes(height, width):
    import torchvision.models as tvm
    m = fuse_depthwise(tvm.mobilenet_v3_large().features)
    shapes = []
    for mod in m.modules():
        if isinstance(mod, DepthwiseConv2d):
            mod.register_forward_hook(lambda mod, i, o: shapes.append(
                (mod.in_channels, i[0].shape[2], i[0].shape[3], mod.kernel_size[0], mod.stride[0])))
    with torch.no_grad():
        m.eval()(torch.zeros(1, 3, height, width))
    return shapes


class Autocast(nn.Module):
    def __init__(self, mod):
        super().__init__()
        self.mod = mod

    def forward(self, x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return self.mod(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--sm-clock-mhz", type=float, default=1965.0, help="SM clock of the FMA bound (B200 maximum)")
    ap.add_argument("--out", default="", help="also write the per-layer results as JSON to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_depthwise.py needs a CUDA device")
    os.environ["CRF_DEBUG_GUARD"] = "0"
    dev = torch.device("cuda:0")
    hbm = load_peaks()["hbm_gbs"]
    fma_gflops = torch.cuda.get_device_properties(dev).multi_processor_count * 128 * 2 * a.sm_clock_mhz / 1e3
    rows, tot_lib, tot_torch = [], 0.0, 0.0
    print(f"{'layer':>26} {'lib us':>8} {'torch us':>9} {'MB':>7} {'lib GB/s':>9} {'bound':>6} {'of bound':>9}")
    for i, (C, H, W, k, s) in enumerate(layer_shapes(a.height, a.width)):
        torch.manual_seed(i)
        conv = nn.Conv2d(C, C, k, s, k // 2, groups=C, bias=False)
        ref = Autocast(conv).to(dev).to(memory_format=torch.channels_last)
        ours = Autocast(DepthwiseConv2d.from_conv(conv)).to(dev).to(memory_format=torch.channels_last)
        x = torch.randn(a.batch, C, H, W, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
        dy = torch.randn(a.batch, C, Ho, Wo, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        t_lib = graph_time_us(ours, x, dy, a.iters)
        assert ours.mod._tickets is not None, "the library path was not taken"
        t_torch = graph_time_us(ref, x, dy, a.iters)
        n_in, n_out = a.batch * H * W * C, a.batch * Ho * Wo * C
        nbytes = 3 * 2.0 * (n_in + n_out)
        flops = 3 * 2.0 * k * k * n_out
        t_hbm, t_fma = nbytes / hbm / 1e3, flops / fma_gflops / 1e3   # µs
        bound = "hbm" if t_hbm >= t_fma else "fma"
        frac = max(t_hbm, t_fma) / t_lib
        gbs = nbytes / t_lib / 1e3
        name = f"{i:2d} C{C} {H}x{W} k{k} s{s}"
        print(f"{name:>26} {t_lib:8.1f} {t_torch:9.1f} {nbytes / 1e6:7.1f} {gbs:9.0f} {bound:>6} {frac:9.2f}")
        rows.append({"layer": i, "C": C, "H": H, "W": W, "k": k, "stride": s, "us_lib": t_lib, "us_torch": t_torch,
                     "bytes": nbytes, "flops": flops, "gbs_lib": gbs, "bound": bound, "frac_of_bound": frac,
                     "frac_hbm_peak": gbs / hbm})
        tot_lib += t_lib
        tot_torch += t_torch
    print(f"total fwd+bwd of the 15 layers: library {tot_lib / 1e3:.3f} ms, torch {tot_torch / 1e3:.3f} ms")
    if not a.out:
        return
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"device": torch.cuda.get_device_name(dev), "hbm_peak_gbs": hbm, "fma_peak_gflops": fma_gflops,
                   "batch": a.batch, "total_ms_lib": tot_lib / 1e3, "total_ms_torch": tot_torch / 1e3, "layers": rows},
                  f, indent=1)


if __name__ == "__main__":
    main()
