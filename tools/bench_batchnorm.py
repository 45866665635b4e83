"""Per-layer timing of the encoder's 46 training-mode BatchNorm + activation layers: forward + backward of one layer at
batch 8 and the bench resolution (480 x 640), each captured in a CUDA graph and replayed, library (BatchNormAct2d)
against torch (nn.BatchNorm2d followed by the inplace ReLU / Hardswish module).  Prints one line per layer, and with
--out FILE also writes them as JSON.

Bytes are algorithmic: forward reads x twice and writes y, backward reads x and dy twice and writes dx, all bf16:
16 T C bytes per layer (T = B H W).  Inputs of 78 MB and less stay partly in the 126 MB L2 between replays, so the
smaller layers can exceed the HBM rate; the fraction of peak is against bench.py's HBM figure."""
import argparse
import json
import os
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import load_peaks  # noqa: E402
from monocular_depth_estimation_b200.model import BatchNormAct2d, fuse_batchnorm_act  # noqa: E402


def layer_shapes(height, width):
    import torchvision.models as tvm
    m = fuse_batchnorm_act(tvm.mobilenet_v3_large().features)
    shapes = []
    for mod in m.modules():
        if isinstance(mod, BatchNormAct2d):
            mod.register_forward_hook(lambda mod, i, o: shapes.append((mod.num_features, i[0].shape[2], i[0].shape[3],
                                                                       mod.act)))
    with torch.no_grad():
        m.eval()(torch.zeros(1, 3, height, width))
    return shapes


def graph_time_us(mod, x, dy, iters):
    """Mean time of one forward + backward, replayed from a CUDA graph (µs)."""
    xg = x.clone().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            mod(xg).backward(dy)
    torch.cuda.current_stream().wait_stream(side)
    for p in mod.parameters():
        p.grad = None
    xg.grad = None
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        mod(xg).backward(dy)
    for _ in range(3):
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def step_breakdown(batch, height, width, steps):
    """Library BatchNorm kernel time per training step of the bench workload, from the library's per-kernel timing (the
    bench's kernel breakdown: CUDA events around every library launch of eager steps)."""
    import ctypes
    from monocular_depth_estimation_b200 import _lib
    from monocular_depth_estimation_b200.model import PTModel
    from monocular_depth_estimation_b200.training import LibAdam, train_step
    dev = torch.device("cuda:0")
    model = PTModel().to(dev).train().to(memory_format=torch.channels_last)
    opt = LibAdam([p for p in model.parameters() if p.requires_grad], 1e-4)
    img = torch.rand(batch, 3, height, width, device=dev).contiguous(memory_format=torch.channels_last)
    dep = torch.rand(batch, 1, height, width, device=dev)
    for _ in range(3):
        train_step(model, opt, img, dep)
    lib = _lib.lib()
    lib.crf_timing_enable(1)
    for _ in range(steps):
        train_step(model, opt, img, dep)
    torch.cuda.synchronize()
    lib.crf_timing_enable(0)
    need = lib.crf_timing_report(None, 0)
    buf = ctypes.create_string_buffer(need + 16)
    lib.crf_timing_report(buf, need + 16)
    kernels = json.loads(buf.value.decode())
    per = {}
    for k in kernels:
        if k["kernel"].startswith("bn_"):
            kind = k["kernel"].split("_C")[0]
            per[kind] = per.get(kind, 0.0) + k["total_ms"] / steps
    return {"ms_per_step": sum(per.values()), "by_kernel": per,
            "launches_per_step": sum(k["launches"] for k in kernels if k["kernel"].startswith("bn_")) / steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default="", help="also write the per-layer results as JSON to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_batchnorm.py needs a CUDA device")
    os.environ["CRF_DEBUG_GUARD"] = "0"
    dev = torch.device("cuda:0")
    peak = load_peaks()["hbm_gbs"]
    acts = {"relu": nn.ReLU(inplace=True), "hardswish": nn.Hardswish(inplace=True), None: nn.Identity()}
    rows, tot_lib, tot_torch = [], 0.0, 0.0
    print(f"{'layer':>28} {'lib us':>8} {'torch us':>9} {'lib GB/s':>9} {'of peak':>8}")
    for i, (C, H, W, act) in enumerate(layer_shapes(a.height, a.width)):
        torch.manual_seed(i)
        x = torch.randn(a.batch, C, H, W, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        dy = torch.randn_like(x)
        ours = BatchNormAct2d(C, eps=1e-3, momentum=0.01, act=act).to(dev).train()
        ref = nn.Sequential(nn.BatchNorm2d(C, eps=1e-3, momentum=0.01), acts[act]).to(dev).train()
        t_lib = graph_time_us(ours, x, dy, a.iters)
        t_torch = graph_time_us(ref, x, dy, a.iters)
        nbytes = 16.0 * a.batch * H * W * C
        gbs = nbytes / t_lib / 1e3
        name = f"{i:2d} C{C} {H}x{W} {act}"
        print(f"{name:>28} {t_lib:8.1f} {t_torch:9.1f} {gbs:9.0f} {gbs / peak:8.2f}")
        rows.append({"layer": i, "C": C, "H": H, "W": W, "act": act, "us_lib": t_lib, "us_torch": t_torch,
                     "bytes": nbytes, "gbs_lib": gbs, "frac_hbm_peak": gbs / peak})
        tot_lib += t_lib
        tot_torch += t_torch
    print(f"total fwd+bwd of the 46 layers: library {tot_lib / 1e3:.3f} ms, torch {tot_torch / 1e3:.3f} ms")
    step = step_breakdown(a.batch, a.height, a.width, 5)
    print("library BatchNorm kernels in the training step's per-kernel breakdown:", json.dumps(step))
    if not a.out:
        return
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"device": torch.cuda.get_device_name(dev), "hbm_peak_gbs": peak, "batch": a.batch,
                   "total_ms_lib": tot_lib / 1e3, "total_ms_torch": tot_torch / 1e3, "step_breakdown": step,
                   "layers": rows}, f, indent=1)


if __name__ == "__main__":
    main()
