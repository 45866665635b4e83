#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on its own config: 480x640 training img/s of MobileNetV3-large + NeWCRFs decoder
(configs[1]: batch 8 per GPU, bf16 autocast for encoder/convs, CRF blocks on the sm_100a library), with the
per-kernel tensor-core / HBM roofline of the dominant CRF kernel and the host-CPU baseline beside it.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps K --warmup W     # the reference's CPU path (oracle port), host cores
    python bench.py --steps K --warmup W --dump-outputs DIR   # also write what the timed step computes (.npy)

A "step" is one iteration of the reference training loop (src/train.py:86-114): forward, SSIM + 0.1 L1 loss,
backward, Adam.  Data is synthetic (rand image / depth of NYU shape), weights are random-init (no network).
One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "train_images_per_sec_480x640"
UNIT = "img/s"


_REAL_STDOUT = None


def emit(line):
    """Write the ONE JSON line to the process's real stdout (see main(): fd 1 is pointed at stderr while working so
    that banners printed by native libraries, e.g. 'NCCL version ...', cannot end up in front of it)."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="images per GPU (weak scaling)")
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--ref-batch", type=int, default=0,
                    help="images per CPU reference step; 0 (default): the same batch as our arm (--batch)")
    ap.add_argument("--regions", type=int, default=5,
                    help="timed regions of exactly --steps steps each; `value` is the MEDIAN region (step time is bimodal "
                         "across repetitions, DESIGN.md 8), all regions are listed in `regions_ms_per_step`")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--breakdown", default="", help="write the per-kernel timing table (JSON) to this file")
    ap.add_argument("--cuda-graph", type=int, default=2,
                    help="1: capture the whole training step (fwd+loss+bwd+Adam) in a CUDA graph at N=1 and replay it; "
                         "2: also at N>1 (DDP all-reduce captured in the graph); 0: eager")
    ap.add_argument("--profile-range", action="store_true",
                    help="bracket the timed region with cudaProfilerStart/Stop (for `ncu --profile-from-start off`)")
    ap.add_argument("--cudnn-benchmark", type=int, default=0,
                    help="1: torch.backends.cudnn.benchmark (cuDNN autotunes the stock convolutions during warm-up)")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="BASELINE configs[3]: fixed global batch (64) sharded over the ranks, i.e. strong scaling; "
                         "0 (default): --batch images per GPU, weak scaling")
    ap.add_argument("--no-gpu-eager-baseline", action="store_true",
                    help="N=1: skip timing the reference's eager PyTorch path on this GPU (gpu_eager_baseline / "
                         "vs_gpu_eager; SURVEY.md 8d, BASELINE.md 3)")
    ap.add_argument("--lib-adam", action="store_true", default=True,
                    help="the library's multi-tensor Adam step (crf_adam_step, training.LibAdam): the default since it was "
                         "measured (13.89 against 14.15-14.5 ms per step with torch's fused Adam, same loss trajectory)")
    ap.add_argument("--torch-adam", dest="lib_adam", action="store_false",
                    help="use torch.optim.Adam(fused=True) instead of the library's Adam step")
    ap.add_argument("--bucket-mb", type=int, default=64, help="N>1: DDP gradient bucket size (MB)")
    ap.add_argument("--no-comm-breakdown", action="store_true",
                    help="N>1: skip the all-reduce measurements (alone / exposed / overlapped) and the config-4 strong-scaling block")
    ap.add_argument("--ddp-grad-bf16", action="store_true",
                    help="N>1: exchange the gradient buckets in bf16 (90 MB instead of 180 MB per step); off by default")
    ap.add_argument("--memory-format", default="channels_last", choices=["contiguous", "channels_last"],
                    help="memory format of the model and the images (host-side choice; math is identical)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed regions, run the timed step twice from the seeded initial model and "
                         "optimizer state and write its losses and first gradients to DIR/<name>.npy (dump_outputs), "
                         "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.tmp = gpu_index, None, None

    def start(self):
        try:
            self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            self.tmp.flush()
            self.tmp.seek(0)
            rows = [[c.strip() for c in ln.split(",")] for ln in self.tmp.read().splitlines() if ln.count(",") >= 8]
            sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
            busy = [v for v in sm if v > 0.5 * max(sm)] if sm else []
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            reasons = sorted({names[i] for r in rows for i in range(4) if r[5 + i].lower().startswith("active")})
            out = {"sm_mhz": statistics.median(busy) if busy else None,
                   "sm_max_mhz": float(rows[0][2]) if rows else None, "reasons": reasons, "samples": len(rows)}
        except Exception:
            pass
        finally:
            try:
                os.unlink(self.tmp.name)
            except Exception:
                pass
        return out


DUMP_SAMPLE = 1 << 20   # elements of the gradient sample: 4 MB in float32


def reset_state(model, optimizer, state0):
    """Put the model back into `state0` (a clone of its state_dict) and the optimizer into the state a fresh Adam starts
    from (moments and step counters at zero), in place: a captured CUDA graph keeps reading the same tensors."""
    import torch
    with torch.no_grad():
        for k, t in model.state_dict().items():
            t.copy_(state0[k])
        for st in optimizer.state.values():
            for t in st.values():
                if torch.is_tensor(t):
                    t.zero_()


def grad_sample(model):
    """A fixed sample (seeded, DUMP_SAMPLE elements) of the model's gradients, float32 on the host, flattened in
    model.named_parameters() order and in logical element order, so it does not depend on the memory format."""
    import numpy as np
    import torch
    params = [p for _, p in model.named_parameters() if p.requires_grad]
    n = sum(p.numel() for p in params)
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
    return flat[torch.from_numpy(idx).to(flat.device)].float().cpu().numpy()


def dump_outputs(out_dir, losses, grads):
    """`loss.npy`: the losses train_step returned (float64), `grads.npy`: a grad_sample (float32).

    Two runs of the same build (`--steps 10 --warmup 3`, B200 at its 1000 W power limit) agreed to rel 6e-7 in the
    losses and rel-L2 1.7e-3 in the gradient sample (every element within rtol 1e-2, atol 1e-6): the bf16 path's
    rounding under a varying summation order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array(losses, dtype=np.float64))
    np.save(os.path.join(out_dir, "grads.npy"), grads)


# --------------------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the path (oracle port; the Python reference cannot travel)
# --------------------------------------------------------------------------------------------------------------
def cpu_reference_run(batch, height, width, steps, warmup):
    import torch
    from oracle import model_oracle as MO
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    # the unmodified reference model when its sources are reachable (build container), else its restatement
    kind, make_model = "port", MO.OraclePTModel
    try:
        from oracle import ref_import
        ref_cls = ref_import.reference_ptmodel()
        if ref_cls is not None:
            kind, make_model = "reference", ref_cls
    except Exception:
        pass
    model = make_model().train()
    opt = torch.optim.Adam(model.parameters(), 1e-4)
    image = torch.rand(batch, 3, height, width)
    depth = torch.rand(batch, 1, height, width)
    for _ in range(warmup):
        MO.train_step(model, opt, image, depth)
    t0 = time.perf_counter()
    for _ in range(steps):
        MO.train_step(model, opt, image, depth)
    dt = time.perf_counter() - t0
    what = ("the unmodified reference model (shim-imported)" if kind == "reference"
            else "oracle port of the reference PyTorch path")
    return {"value": batch * steps / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{steps} fp32 train steps (fwd+loss+bwd+Adam) of batch {batch} at {height}x{width} on the host CPU, "
                      f"{what}, torch.set_num_threads({cores})",
            "ms_per_step": 1e3 * dt / steps}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    ref_batch = args.ref_batch or args.batch
    r = cpu_reference_run(ref_batch, args.height, args.width, steps, warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "MobileNetV3-large + NeWCRFs decoder train step (fwd+loss+bwd+Adam), "
                                   f"{args.height}x{args.width}, host CPU, batch {ref_batch} per step "
                                   "(BASELINE.json configs[1])",
                       "global_batch": ref_batch, "parallelism": "host CPU, 1 process",
                       "arm": ("the unmodified reference model, shim-imported" if r["kind"] == "reference" else
                               "oracle port of the reference's PyTorch CPU path (the Python reference cannot travel to "
                               "the GPU box; the port is pinned to the unmodified reference by tests/test_oracle_golden.py)")},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                             "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# --------------------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from monocular_depth_estimation_b200 import _lib
    from monocular_depth_estimation_b200.model import PTModel
    from monocular_depth_estimation_b200.training import init_distributed, train_step, wrap_ddp

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sm_100a path has no CPU fallback "
                         "(use --impl reference for the CPU reference arm)")
    lib = _lib.lib()  # fail loudly if the extension is missing
    graph_multi = bool(args.cuda_graph >= 2 and int(os.environ.get("WORLD_SIZE", "1")) > 1)
    if graph_multi:  # whole-step capture with DDP (PyTorch CUDA-graph notes): no async NCCL error handling
        os.environ["TORCH_NCCL_ASYNC_ERROR_HANDLING"] = "0"
    rank, local_rank, world, device = init_distributed()
    torch.cuda.set_device(device)
    torch.manual_seed(1234 + rank)
    torch.backends.cudnn.benchmark = bool(args.cudnn_benchmark)
    B, H, W = args.batch, args.height, args.width
    if args.global_batch:   # BASELINE.json configs[3]: a fixed global batch sharded over the ranks (strong scaling)
        if args.global_batch % world:
            raise SystemExit(f"bench.py: --global-batch {args.global_batch} is not divisible by {world} ranks")
        B = args.global_batch // world

    model = PTModel().to(device).train()
    mf = torch.channels_last if args.memory_format == "channels_last" else torch.contiguous_format
    model = model.to(memory_format=mf)
    use_graph = bool(args.cuda_graph and (world == 1 or graph_multi))
    grad_dtype = torch.bfloat16 if args.ddp_grad_bf16 else None
    if graph_multi:  # DDP must be constructed on the side stream the warm-up and capture will use
        side0 = torch.cuda.Stream()
        side0.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side0):
            net = wrap_ddp(model, device, world, grad_dtype=grad_dtype, bucket_cap_mb=args.bucket_mb)
        torch.cuda.current_stream().wait_stream(side0)
    else:
        net = wrap_ddp(model, device, world, grad_dtype=grad_dtype, bucket_cap_mb=args.bucket_mb)
    # same update as train.py:41 in one fused kernel; capturable so the step can live in a CUDA graph
    if args.lib_adam:   # training.LibAdam: same update as torch.optim.Adam (test_lib_adam_matches_torch_adam, 1e-5), fewer / shorter launches
        from monocular_depth_estimation_b200.training import LibAdam
        opt = LibAdam([p for p in model.parameters() if p.requires_grad], 1e-4)
    else:
        opt = torch.optim.Adam(model.parameters(), 1e-4, fused=True, capturable=use_graph)
    # --dump-outputs: the state the dumped steps start from (taken after DDP gave every rank rank 0's parameters)
    state0 = {k: t.detach().clone() for k, t in model.state_dict().items()} if args.dump_outputs else None

    image_h = torch.rand(B, 3, H, W).contiguous(memory_format=mf).pin_memory()
    depth_h = torch.rand(B, 1, H, W).pin_memory()
    image_d, depth_d = image_h.to(device), depth_h.to(device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    def step_eager():
        return train_step(net, opt, image_d, depth_d)

    for _ in range(max(args.warmup, 3)):
        step_eager()

    # Whole-step CUDA graph (single GPU): ~1600 launches per step are replayed from one graph, which removes the
    # CPU launch gaps (the GPU is otherwise idle ~10 % of the step).  The captured work is the same eager step.
    graph, static_loss, launches_per_replay = None, None, 0
    if use_graph:
        try:
            side = side0 if graph_multi else torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(11 if graph_multi else 2):  # DDP needs >= 11 eager iterations before capture
                    step_eager()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            opt.zero_grad(set_to_none=True)
            n_before = lib.crf_kernel_launches()
            with torch.cuda.graph(g):
                static_loss = step_eager()
            launches_per_replay = lib.crf_kernel_launches() - n_before
            g.replay()
            torch.cuda.synchronize()
            graph = g
        except Exception as exc:  # keep the eager path if capture is not possible on this build
            print(f"bench.py: CUDA-graph capture failed ({type(exc).__name__}: {exc}); running eagerly", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()

    resident_loss = [static_loss]

    def step_resident():
        if graph is not None:
            graph.replay()
        else:
            resident_loss[0] = step_eager()

    last_loss = [0.0]
    # End-to-end input pipeline (what a pinned-memory loader with prefetch does): every step's image + depth are copied
    # host -> device from pinned memory on a copy stream into a staging pair while the PREVIOUS step computes; the step
    # itself starts with a device-to-device move into the graph's static input tensors.  The first step of a timed
    # region copies its own batch un-overlapped, so K steps make exactly K host -> device copies, all consumed.
    copy_stream = torch.cuda.Stream()
    image_s, depth_s = torch.empty_like(image_d), torch.empty_like(depth_d)
    ev_h2d, ev_d2d = torch.cuda.Event(), torch.cuda.Event()
    e2e_k = [0]

    def prefetch():
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_d2d)          # the staging pair has been consumed
            image_s.copy_(image_h, non_blocking=True)
            depth_s.copy_(depth_h, non_blocking=True)
            ev_h2d.record(copy_stream)

    def step_e2e():
        if graph is not None:  # the graph reads its inputs from image_d / depth_d
            cur = torch.cuda.current_stream()
            if e2e_k[0] % args.steps == 0:
                prefetch()                          # first step of a region: its own batch, not overlapped
            cur.wait_event(ev_h2d)
            image_d.copy_(image_s, non_blocking=True)
            depth_d.copy_(depth_s, non_blocking=True)
            ev_d2d.record(cur)
            if (e2e_k[0] + 1) % args.steps != 0:
                prefetch()                          # next step's batch travels while this step computes
            e2e_k[0] += 1
            graph.replay()
            last_loss[0] = float(static_loss.item())
        else:
            img = image_h.to(device, non_blocking=True)
            dep = depth_h.to(device, non_blocking=True)
            loss = train_step(net, opt, img, dep)
            last_loss[0] = float(loss.item())  # device -> host read of the step's result

    for _ in range(3):
        step_resident()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n0 = lib.crf_kernel_launches()
    if args.profile_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
    regions = [timed(step_resident, args.steps) for _ in range(max(1, args.regions))]
    ms = statistics.median(regions)   # every region is exactly --steps steps; the median region is reported
    if args.profile_range:
        torch.cuda.profiler.stop()
    launches = (lib.crf_kernel_launches() - n0) // max(1, args.regions)
    if graph is not None:
        launches = launches_per_replay * args.steps  # replayed from the graph: counted once at capture time
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # The state reached after the timed regions differs from run to run (float atomics in the library and cuDNN's
        # convolutions vary the summation order, and the Adam steps amplify that), so the timed step runs twice more
        # from the seeded initial state, on every rank (a DDP step all-reduces): rank 0 writes both losses and the
        # first step's gradients.  With the same arguments, these depend on the arguments only, up to rounding.
        reset_state(model, opt, state0)
        step_resident()
        losses, grads = [resident_loss[0].detach().item()], grad_sample(model)
        step_resident()
        losses.append(resident_loss[0].detach().item())
        if rank == 0:
            dump_outputs(args.dump_outputs, losses, grads)
        state0 = None

    for _ in range(args.steps):   # one full untimed region (keeps the prefetch phase aligned with the step counter)
        step_e2e()
    regions_e2e = [timed(step_e2e, args.steps) for _ in range(max(1, args.regions))]
    ms_e2e = statistics.median(regions_e2e)

    # per-kernel timing pass: same step loop, every library kernel bracketed by CUDA events on its own stream
    lib.crf_timing_enable(1)
    ms_probe = timed(step_eager, args.steps)
    lib.crf_timing_enable(0)
    need = lib.crf_timing_report(None, 0)
    buf = ctypes.create_string_buffer(need + 16)
    lib.crf_timing_report(buf, need + 16)
    kernels = json.loads(buf.value.decode())

    # ---- N > 1: what the gradient exchange costs (all ranks take part; eager steps, CUDA events, max over ranks) ----
    comm, config4 = None, None
    if world > 1 and not args.no_comm_breakdown:
        k = max(3, min(args.steps, 10))
        ms_with = timed(step_eager, k) / k

        def step_nosync():     # the same step without the all-reduce (gradients stay rank-local)
            with net.no_sync():
                return train_step(net, opt, image_d, depth_d)
        for _ in range(2):
            step_nosync()
        ms_without = timed(step_nosync, k) / k
        with torch.no_grad():  # the un-synchronised steps let the replicas drift apart: re-align them with rank 0
            for p_ in model.parameters():
                dist.broadcast(p_.data, 0)
        step_eager()
        nbytes = sum(p.numel() for p in model.parameters() if p.requires_grad) * (2 if args.ddp_grad_bf16 else 4)
        flat = torch.empty(nbytes // 4, dtype=torch.float32, device=device)

        def allreduce_alone():
            dist.all_reduce(flat)
        for _ in range(3):
            allreduce_alone()
        ms_alone = timed(allreduce_alone, 10) / 10
        exposed = max(0.0, ms_with - ms_without)
        comm = {"gradient_bytes": nbytes, "allreduce_alone_ms": ms_alone,
                "allreduce_alone_busbw_gbs": 2.0 * (world - 1) / world * nbytes / (ms_alone * 1e-3) / 1e9,
                "step_ms_eager_with_allreduce": ms_with, "step_ms_eager_without_allreduce": ms_without,
                "exposed_ms": exposed, "overlapped_fraction": max(0.0, 1.0 - exposed / ms_alone) if ms_alone else None,
                "bucket_mb": args.bucket_mb, "how": "eager steps (no CUDA graph): DDP step vs the same step under no_sync(), "
                "and one all-reduce of the whole gradient volume alone; CUDA events, max over ranks"}
        # BASELINE.json configs[3]: global batch 64 sharded over the ranks (strong scaling), eager DDP steps
        gb = 64
        if not args.global_batch and gb % world == 0:
            Bs = gb // world
            try:
                img_s = torch.rand(Bs, 3, H, W, device=device).contiguous(memory_format=mf)
                dep_s = torch.rand(Bs, 1, H, W, device=device)

                def step_strong():
                    return train_step(net, opt, img_s, dep_s)
                for _ in range(3):
                    step_strong()
                ks = max(3, min(args.steps, 6))
                ms_s = timed(step_strong, ks) / ks
                config4 = {"global_batch": gb, "per_gpu_batch": Bs, "n_gpus": world, "ms_per_step": ms_s,
                           "value": gb / (ms_s * 1e-3), "unit": UNIT, "scaling": "strong", "cuda_graph": False,
                           "what": "BASELINE.json configs[3]: global batch 64 at 480x640 sharded over the ranks, "
                                   "eager DDP steps (fwd + loss + bwd + NCCL all-reduce + Adam)"}
                del img_s, dep_s
            except Exception as exc:
                config4 = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()

    def finish():
        # Orderly exit: drop the captured graph (it references the NCCL communicator) before the process group goes.
        # A watchdog ends the process if destroy_process_group() does not return (observed once with a captured DDP
        # step in round 1; the result line has been printed by then).
        nonlocal graph
        torch.cuda.synchronize()
        if world > 1:
            import gc
            import threading
            graph = None
            gc.collect()
            torch.cuda.synchronize()
            sys.stdout.flush()
            sys.stderr.flush()
            dog = threading.Timer(20.0, lambda: os._exit(0))
            dog.daemon = True
            dog.start()
            dist.barrier()
            dist.destroy_process_group()
            dog.cancel()

    if rank != 0:
        finish()
        return

    peaks = load_peaks()
    tot = sum(k["total_ms"] for k in kernels) or 1.0
    kernels.sort(key=lambda k: -k["total_ms"])
    breakdown = [{"kernel": k["kernel"], "launches": k["launches"], "ms_per_step": k["total_ms"] / args.steps,
                  "share": k["total_ms"] / tot,
                  "tflops": k["flops"] * k["launches"] / (k["total_ms"] * 1e-3) / 1e12 if k["total_ms"] else 0.0,
                  "gbs": k["bytes"] * k["launches"] / (k["total_ms"] * 1e-3) / 1e9 if k["total_ms"] else 0.0}
                 for k in kernels]
    if args.breakdown:
        with open(args.breakdown, "w") as f:
            json.dump(breakdown, f, indent=1)

    # ---- roofline: the CRF BLOCK against SURVEY.md 8(d) --------------------------------------------------------
    # Algorithmic work of one CRFBlock: (22*49*C^2 + 4*49^2*C) flops per 49-token window forward, x3 with backward;
    # minimum HBM bytes of a fully fused block: 8*C*2 per token forward+backward (x, v -> y; x, v, dy -> dx, dv in bf16).
    # `roofline` is the step-level figure: all eight blocks' algorithmic flops / the CUDA-event time of the library's
    # block kernels inside the step, against the measured SUSTAINED bf16 peak (the kernels are timed inside a long step).
    STAGES = ((4, 128, 4), (8, 256, 8), (16, 512, 16), (32, 1024, 32))

    def n_windows(Hs, Ws):
        return B * (-(-Hs // 7)) * (-(-Ws // 7))

    def block_flops(Hs, Ws, Cd):
        # SURVEY.md 8(d): qk / attention / proj act on the padded tokens Tp = 49 * windows, LayerNorm / MLP on the real
        # tokens T; forward = Tp * (6 C^2 + 196 C) + T * 16 C^2, x3 with backward (60.29 GFLOP forward at 120x160, C = 128,
        # B = 8; all eight blocks of the step: 1454.6 GFLOP)
        Tp, T_ = 49.0 * n_windows(Hs, Ws), float(B * Hs * Ws)
        return 3.0 * (Tp * (6 * Cd * Cd + 196 * Cd) + T_ * 16 * Cd * Cd)

    def block_min_bytes(Hs, Ws, Cd, nH):
        # fully fused block, bf16 activations: per window 49 * 8 C * 2 B forward+backward (x, v -> y; x, v, dy -> dx, dv),
        # plus the fp32 parameters read once per direction and their gradients written once
        params = 11 * Cd * Cd + 12 * Cd + 169 * nH
        return n_windows(Hs, Ws) * 49 * 8 * Cd * 2 + 3 * params * 4

    BLOCK_PREFIXES = ("gemm_", "gemm2", "dgrad_lnbwd", "attn_", "ln_fwd", "ln_bwd", "cast4", "cast_bf16", "convert_bf16", "mlp_fused", "splitk_reduce")
    blk_k = [k for k in kernels if k["kernel"].startswith(BLOCK_PREFIXES)]
    blk_ms = sum(k["total_ms"] for k in blk_k) / args.steps                       # per step, all eight blocks
    blk_bytes = sum(k["bytes"] * k["launches"] for k in blk_k) / args.steps       # sum of per-kernel algorithmic bytes
    step_flops = sum(2 * block_flops(H // sc, W // sc, Cd) for sc, Cd, _ in STAGES)
    step_min_bytes = sum(2 * block_min_bytes(H // sc, W // sc, Cd, nH_) for sc, Cd, nH_ in STAGES)
    tf = step_flops / (blk_ms * 1e-3) / 1e12 if blk_ms else 0.0
    traffic, traffic_src = None, None
    try:   # DRAM bytes of the block kernels from the committed `ncu --set full` captures, where all of them were captured
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            ent = json.load(f).get("crf_blocks_step")
        if ent:
            traffic, traffic_src = ent["dram_bytes"], ent.get("source")
    except Exception:
        pass
    roof = {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
            "frac": tf / peaks["bf16_tflops_sustained"], "traffic": traffic, "traffic_source": traffic_src,
            "what": "all 8 CRF blocks of the step (fwd+bwd): algorithmic flops of SURVEY.md 8(d) / CUDA-event time of the "
                    "library's block kernels inside the step",
            "algorithmic_gflop_per_step": step_flops / 1e9, "block_kernel_ms_per_step": blk_ms,
            "peak_source": peaks["source"] + " (bf16 peak: sustained figure, kernels timed inside the step)",
            "hbm": {"min_bytes_fused_MB": step_min_bytes / 1e6, "sum_kernel_algorithmic_bytes_MB": blk_bytes / 1e6,
                    "bytes_ratio_vs_fused_minimum": blk_bytes / step_min_bytes if step_min_bytes else None,
                    "achieved_gbs_on_kernel_bytes": blk_bytes / (blk_ms * 1e-3) / 1e9 if blk_ms else 0.0,
                    "frac_of_hbm_peak_on_kernel_bytes": blk_bytes / (blk_ms * 1e-3) / 1e9 / peaks["hbm_gbs"] if blk_ms else 0.0,
                    "hbm_peak_gbs": peaks["hbm_gbs"]},
            "share_of_step": blk_ms / (ms / args.steps), "library_kernel_ms_per_step": tot / args.steps,
            "step_ms_with_events": ms_probe / args.steps}

    # per-scale: ONE CRFBlock forward+backward (shifted windows) replayed from a CUDA graph (so the small scales are not
    # launch-bound), windows/s, algorithmic TFLOP/s against the bf16 peak, and the attention-core kernels' algorithmic
    # HBM rate (8 resp. 16 bytes per token-channel) against the HBM peak (KernelTimer labels of the step above).
    crf_blocks = None
    if world == 1:
        from monocular_depth_estimation_b200 import CRFBlock
        crf_blocks = []
        for scale, Cd, nH in STAGES:
            Hs, Ws = H // scale, W // scale
            blk = CRFBlock(Cd, nH, Cd, shift_size=3).to(device)
            blk.H, blk.W = Hs, Ws
            xb = torch.randn(B, Hs * Ws, Cd, device=device, requires_grad=True)
            vb = torch.randn(B, Hs, Ws, Cd, device=device, requires_grad=True)
            gy = torch.randn(B, Hs * Ws, Cd, device=device)

            def blk_step():
                blk(xb, vb, None).backward(gy)
                xb.grad = vb.grad = None
                for p_ in blk.parameters():
                    p_.grad = None
            for _ in range(3):
                blk_step()
            ms_eager = timed(blk_step, 10) / 10
            ms_b, graphed = ms_eager, False
            try:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    blk_step()
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                gb = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gb):
                    blk_step()
                gb.replay()
                ms_b, graphed = timed(gb.replay, 20) / 20, True
                del gb
            except Exception as exc:
                print(f"bench.py: block graph capture failed ({type(exc).__name__}: {exc})", file=sys.stderr)
                torch.cuda.synchronize()
            nwin = n_windows(Hs, Ws)
            fl = block_flops(Hs, Ws, Cd)
            ent = {"stage": f"1/{scale}", "H": Hs, "W": Ws, "C": Cd, "heads": nH, "windows": nwin,
                   "ms_fwd_bwd": ms_b, "ms_fwd_bwd_eager": ms_eager, "cuda_graph": graphed,
                   "windows_per_s": nwin / (ms_b * 1e-3), "algorithmic_tflops": fl / (ms_b * 1e-3) / 1e12,
                   "frac_of_bf16_peak": fl / (ms_b * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
                   "min_bytes_MB": block_min_bytes(Hs, Ws, Cd, nH) / 1e6,
                   "frac_of_hbm_peak_on_min_bytes": block_min_bytes(Hs, Ws, Cd, nH) / (ms_b * 1e-3) / 1e9 / peaks["hbm_gbs"]}
            for k in kernels:
                for tag in ("attn_fwd", "attn_bwd"):
                    if k["kernel"] == f"{tag}_B{B}_{Hs}x{Ws}_C{Cd}_s3" and k["total_ms"] > 0:
                        us = k["total_ms"] / k["launches"] * 1e3
                        ent[tag] = {"avg_us": us, "gbs": k["bytes"] / us / 1e3, "frac_of_hbm_peak": k["bytes"] / us / 1e3 / peaks["hbm_gbs"],
                                    "tensor_tflops": k["flops"] / us / 1e6}
            try:   # the same block in the fp32 precision mode (rel 1e-3 tier: split-operand GEMMs, fp32 attention)
                blk.precision = "fp32"
                for _ in range(2):
                    blk_step()
                ms_f = timed(blk_step, 5) / 5
                ent["fp32_mode"] = {"ms_fwd_bwd": ms_f, "windows_per_s": nwin / (ms_f * 1e-3),
                                    "algorithmic_tflops": fl / (ms_f * 1e-3) / 1e12,
                                    "slowdown_vs_bf16_mode": ms_f / ms_eager}
            except Exception as exc:
                ent["fp32_mode"] = {"error": f"{type(exc).__name__}: {exc}"}
            crf_blocks.append(ent)
            del blk, xb, vb, gy
        roof["per_scale"] = [{"stage": e["stage"], "C": e["C"], "ms_fwd_bwd": e["ms_fwd_bwd"],
                              "frac_of_bf16_peak": e["frac_of_bf16_peak"]} for e in crf_blocks]

    # ---- reported baselines -------------------------------------------------------------------------------------
    gpu_eager = None
    if world == 1 and not args.no_gpu_eager_baseline:
        # The reference's real GPU path is eager PyTorch (BASELINE.md 3, SURVEY.md 8d).  The unmodified reference is
        # imported with its three shims when /root/reference (or baseline/_ref) is present; on the GPU box it is not
        # (the Python reference cannot travel), so its restatement with the same torch ops (oracle/model_oracle.py) is
        # timed instead: same config, stock PyTorch kernels only, fused Adam, no CUDA graph.
        from oracle import model_oracle as MO
        ref_kind = "oracle port of the reference's PyTorch path"
        make_model = MO.OraclePTModel
        try:
            from oracle import ref_import
            ref_cls = ref_import.reference_ptmodel()
            if ref_cls is not None:
                make_model, ref_kind = ref_cls, "unmodified reference model (shim-imported)"
        except Exception:
            pass
        gpu_eager = {"kind": ref_kind + ", eager on this GPU: stock PyTorch kernels, channels-last, fused Adam, no CUDA graph",
                     "unit": UNIT, "batch": B}
        for tag, autocast in (("bf16_autocast", True), ("fp32", False)):
            try:
                torch.manual_seed(0)
                ref_model = make_model().to(device).train().to(memory_format=mf)
                ref_opt = torch.optim.Adam(ref_model.parameters(), 1e-4, fused=True)

                def ref_step():
                    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                        pred = ref_model(image_d)
                    loss_r = MO.ssim_l1_loss(pred.float(), MO.depth_norm(depth_d))
                    ref_opt.zero_grad(set_to_none=True)
                    loss_r.backward()
                    ref_opt.step()

                for _ in range(3):
                    ref_step()
                k = max(3, min(args.steps, 5))
                ms_ref = timed(ref_step, k)
                gpu_eager[tag] = {"value": B * k / (ms_ref * 1e-3), "ms_per_step": ms_ref / k, "steps": k}
                del ref_model, ref_opt
            except Exception as exc:
                gpu_eager[tag] = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_run(args.ref_batch or B, H, W, steps=2, warmup=1)
        cpu.pop("ms_per_step", None)

    imgs = B * world * args.steps
    line = {
        "metric": METRIC, "value": imgs / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.global_batch else "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"MobileNetV3-large + NeWCRFs decoder train step (fwd + SSIM/L1 loss + bwd + Adam), "
                               f"{H}x{W}, batch {B} per GPU (BASELINE.json configs[1])",
                   "global_batch": B * world, "parallelism": f"dp{world}", "memory_format": args.memory_format,
                   "gradient_exchange": "none (1 GPU)" if world == 1 else
                   ("NCCL all-reduce, bf16 buckets" if args.ddp_grad_bf16 else "NCCL all-reduce, fp32 buckets"),
                   "cuda_graph": graph is not None,
                   "optimizer": "library Adam (crf_adam_step)" if args.lib_adam else "torch.optim.Adam(fused=True)",
                   "l2": "per-step working set (GBs of activations) far exceeds the 126 MB L2; no explicit flush",
                   "timing": f"median of {len(regions)} regions of exactly {args.steps} steps each (CUDA events, max over ranks)",
                   "precision": "bf16 tensor-core operands + bf16 intermediates, fp32 accumulate/softmax/LN/residual; "
                                "encoder and convs under torch bf16 autocast"},
        "regions_ms_per_step": [r_ / args.steps for r_ in regions],
        "clocks": clocks,
        "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": image_h.numel() * 4 + depth_h.numel() * 4, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps, "regions_ms_per_step": [r_ / args.steps for r_ in regions_e2e],
                "last_loss": last_loss[0],
                "input_pipeline": ("pinned host -> staging copy of step i+1 on a copy stream while step i computes "
                                   "(K copies for K steps, the first one not overlapped); loss read back every step")
                if graph is not None else "copies and step on one stream"},
        "gpu_launches": int(launches),
        "roofline": roof,
        "kernel_breakdown": breakdown[:10],
    }
    if crf_blocks is not None:
        line["crf_blocks"] = crf_blocks
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if comm is not None:
        line["allreduce"] = comm
    if config4 is not None:
        line["config4_strong"] = config4
    if gpu_eager is not None:
        line["gpu_eager_baseline"] = gpu_eager
        best = max((v["value"] for v in gpu_eager.values() if isinstance(v, dict) and "value" in v), default=None)
        if best:
            line["vs_gpu_eager"] = {"value_over_best_eager": line["value"] / best,
                                    "e2e_over_best_eager": line["e2e"]["value"] / best}
    emit(line)
    finish()


def main():
    args = parse_args()
    # rank 0 must print exactly ONE line on stdout: keep NCCL's "NCCL version ..." banner (NCCL_DEBUG=VERSION) off it
    # (NCCL's levels nest: WARN would still print the banner, so the variable is removed unless INFO/TRACE was asked for)
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
        del os.environ["NCCL_DEBUG"]
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
