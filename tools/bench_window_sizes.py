"""One CRFBlock forward + backward at every window size the kernels implement (2..8), at the four decoder scales of
BASELINE.json configs[1] (batch 8, 480 x 640 input: 120x160 C128, 60x80 C256, 30x40 C512, 15x20 C1024; shifted
block, shift = window // 2, bf16 tier).

    python tools/bench_window_sizes.py [--out-dir DIR] [--iters 20] [--warmup 3]

Per (window, scale):
  * block_ms: CUDA-event time of one forward + backward, replayed from a CUDA graph (captured after a warm-up; eager
    launches with events if the capture fails, flagged "graph": false), over --iters replays;
  * windows/s and ns per token of that time;
  * algorithmic TFLOP/s: SURVEY section 8d's per-window flops of a block with N = ws^2 in place of 49,
    (22 N C^2 + 4 N^2 C) x 3 for forward + backward, over block_ms;
  * the attention kernels alone (library KernelTimer events, eager run): forward / backward time, their algorithmic
    bytes (8 resp. 16 bytes per token-channel: q|k, v in bf16, o / dq|dk, dv out) as GB/s and as a fraction of the
    7.7 TB/s HBM3e of NVIDIA's HGX B200 data sheet.
Writes <out-dir>/r03_window_sizes.json and .md (default: profiles/) with the device name and power limit beside the
numbers.  Inputs are device resident; writes nothing else.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from monocular_depth_estimation_b200 import _lib  # noqa: E402
from monocular_depth_estimation_b200.model import CRF_DIMS, NUM_HEADS  # noqa: E402
from monocular_depth_estimation_b200.newcrf_layers import CRFBlock  # noqa: E402

HBM_PEAK_GBS = 7700.0   # NVIDIA HGX B200 data sheet, one GPU
WINDOWS = range(2, 9)


def block_flops(ws, C):
    N = ws * ws
    return (22 * N * C * C + 4 * N * N * C) * 3


def device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_clock_max"] = [s.strip() for s in q.split(",")]
    except Exception as exc:  # noqa: BLE001
        info["power_limit"] = f"unknown ({type(exc).__name__})"
    return info


def kernel_times(lib, fn, iters):
    lib.crf_timing_enable(1)
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    lib.crf_timing_enable(0)
    need = lib.crf_timing_report(None, 0)
    buf = ctypes.create_string_buffer(need + 16)
    lib.crf_timing_report(buf, need + 16)
    return json.loads(buf.value.decode())


def run_case(lib, ws, B, H, W, C, nH, iters, warmup):
    dev = torch.device("cuda:0")
    torch.manual_seed(ws * 1000 + C)
    blk = CRFBlock(C, nH, C, window_size=ws, shift_size=ws // 2).to(dev)
    blk.H, blk.W = H, W
    x = torch.randn(B, C, H, W, device=dev).flatten(2).transpose(1, 2).requires_grad_(True)
    v = torch.randn(B, C, H, W, device=dev).permute(0, 2, 3, 1).requires_grad_(True)
    dy = torch.randn(B, H * W, C, device=dev)

    def step():
        blk(x, v, None).backward(dy)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warmup):
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = None
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step()
        graph = g
    except Exception as exc:  # noqa: BLE001
        print(f"bench_window_sizes: graph capture failed at ws {ws} ({type(exc).__name__}: {exc}); eager timing",
              file=sys.stderr)
    run = graph.replay if graph is not None else step
    for _ in range(warmup):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters

    kt = kernel_times(lib, step, max(3, iters // 4))
    att = {}
    for k in kt:
        for tag in ("attn_fwd", "attn_bwd"):
            if k["kernel"].startswith(tag + "_"):
                avg = k["total_ms"] / max(k["launches"], 1)
                att[tag] = {"us": avg * 1e3, "gbs": k["bytes"] / avg / 1e6,
                            "frac_hbm_peak": k["bytes"] / avg / 1e6 / HBM_PEAK_GBS}
    nwin = B * (-(-H // ws)) * (-(-W // ws))
    T = B * H * W
    return {"window": ws, "N": ws * ws, "B": B, "H": H, "W": W, "C": C, "heads": nH, "shift": ws // 2,
            "windows": nwin, "graph": graph is not None, "block_ms": ms,
            "windows_per_s": nwin / (ms * 1e-3), "ns_per_token": ms * 1e6 / T,
            "tile_rows_used": f"{ws * ws}/64",
            "algorithmic_tflops": block_flops(ws, C) * nwin / (ms * 1e-3) / 1e12, "attention": att}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_window_sizes: needs a CUDA device (sm_100a); there is no CPU path")
    lib = _lib.lib()
    info = device_info()
    rows = []
    for s, (C, nH) in enumerate(zip(CRF_DIMS, NUM_HEADS)):
        H, W = 480 // (4 << s), 640 // (4 << s)
        for ws in WINDOWS:
            r = run_case(lib, ws, args.batch, H, W, C, nH, args.iters, args.warmup)
            rows.append(r)
            print(json.dumps(r), flush=True)
    out = {"device": info, "hbm_peak_gbs": HBM_PEAK_GBS,
           "what": "one CRFBlock forward+backward (shift ws//2, bf16 tier), BASELINE configs[1] decoder scales, batch "
                   f"{args.batch}; CUDA-graph replay, {args.iters} replays after {args.warmup} warm-up steps",
           "rows": rows}
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "r03_window_sizes.json"), "w") as f:
        json.dump(out, f, indent=1)
    md = [f"# CRF block forward + backward by window size ({info['name']}, power limit {info.get('power_limit')})", "",
          out["what"] + ".", "",
          "| scale | C | ws | N/64 rows | windows | block ms | windows/s | ns/token | TFLOP/s (alg.) | attn fwd us | "
          "attn fwd GB/s | attn bwd us | attn bwd GB/s |", "|---|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|---:|"]
    for r in rows:
        a, b = r["attention"].get("attn_fwd", {}), r["attention"].get("attn_bwd", {})
        md.append(f"| {r['H']}x{r['W']} | {r['C']} | {r['window']} | {r['tile_rows_used']} | {r['windows']} | "
                  f"{r['block_ms']:.3f} | {r['windows_per_s']:.3g} | {r['ns_per_token']:.2f} | "
                  f"{r['algorithmic_tflops']:.1f} | {a.get('us', 0):.1f} | {a.get('gbs', 0):.0f} | "
                  f"{b.get('us', 0):.1f} | {b.get('gbs', 0):.0f} |")
    with open(os.path.join(args.out_dir, "r03_window_sizes.md"), "w") as f:
        f.write("\n".join(md) + "\n")


if __name__ == "__main__":
    main()
