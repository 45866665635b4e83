"""Training-step plumbing around the hot path: the reference loop's loss (src/train.py:89-100: SSIM + 0.1 * L1 on
min-max-normalised depth; SSIM from src/loss.py:57-88) and the data-parallel wrapper the reference lacks
(one process per GPU, NCCL gradient all-reduce over NVLink).  Windows never cross images, so sharding the batch
needs no data-path collective; the only exchange is the parameter-gradient average, which DDP overlaps with backward.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn
import torch.nn.functional as F


def depth_norm(depth):
    """src/utils.py:7-8 -- per-batch min-max normalisation."""
    return (depth - depth.min()) / (depth.max() - depth.min())


def ssim_loss(x, y):
    """monodepth2-style SSIM on 3x3 average pools with reflection padding (src/loss.py:57-88)."""
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    x, y = F.pad(x, (1, 1, 1, 1), mode="reflect"), F.pad(y, (1, 1, 1, 1), mode="reflect")
    mu_x, mu_y = F.avg_pool2d(x, 3, 1), F.avg_pool2d(y, 3, 1)
    sx = F.avg_pool2d(x * x, 3, 1) - mu_x * mu_x
    sy = F.avg_pool2d(y * y, 3, 1) - mu_y * mu_y
    sxy = F.avg_pool2d(x * y, 3, 1) - mu_x * mu_y
    n = (2 * mu_x * mu_y + c1) * (2 * sxy + c2)
    d = (mu_x * mu_x + mu_y * mu_y + c1) * (sx + sy + c2)
    return torch.clamp((1 - n / d) / 2, 0, 1).mean()


def depth_loss(pred, depth_n):
    """loss = 1.0 * SSIM + 0.1 * L1 (src/train.py:94-100).  CUDA tensors go through the library's two-kernel
    forward / backward (functional.depth_loss); the composition of torch ops below is what it replaces and remains
    the CPU path of the gloo tests."""
    if pred.is_cuda:
        from .functional import depth_loss as _fused
        return _fused(pred, depth_n)
    return ssim_loss(pred, depth_n) + 0.1 * F.l1_loss(pred, depth_n)


def init_distributed():
    """One process per GPU (torchrun): returns (rank, local_rank, world_size, device)."""
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    device = torch.device("cuda", local_rank) if torch.cuda.is_available() else torch.device("cpu")
    if world > 1 and not dist.is_initialized():
        if device.type == "cuda":
            torch.cuda.set_device(device)
            dist.init_process_group("nccl", device_id=device)
        else:
            dist.init_process_group("gloo")
    return rank, local_rank, world, device


def wrap_ddp(model, device, world, grad_dtype=None, bucket_cap_mb=64):
    """The DDP wrapper `train.py` lacks: gradients are averaged with an NCCL all-reduce, bucketed and launched while
    backward is still running (crf3's 29 M parameters become ready first and are reduced under the rest).

    grad_dtype=torch.bfloat16 exchanges the buckets in bf16 -- 90 MB instead of 180 MB per
    step (SURVEY.md 8e) -- through DDP's stock bf16_compress_hook: each rank's gradient is divided by the world size,
    rounded to bf16, summed by the all-reduce in bf16 and widened back to fp32.  Off by default: the averaged gradient
    then carries a bf16 rounding (rel ~ 2^-9) the fp32 exchange does not have."""
    if world <= 1:
        return model
    if grad_dtype not in (None, torch.float32, torch.bfloat16):
        raise ValueError(f"wrap_ddp: grad_dtype must be None, torch.float32 or torch.bfloat16 (got {grad_dtype})")
    from torch.nn.parallel import DistributedDataParallel as DDP
    # The reference keeps torchvision's ImageNet classifier head inside the encoder module although forward() never
    # uses it (model_mobileV3_large_newCRFs.py:176-182).  DDP requires every trainable parameter to receive a
    # gradient, so those parameters are frozen (they never get a gradient in the reference either).
    for name, p in model.named_parameters():
        if ".original_model.classifier." in name:
            p.requires_grad_(False)
    if device.type == "cuda":
        # broadcast_buffers=False: BatchNorm running statistics stay rank-local (46 BN layers would otherwise add a
        # broadcast of ~140 small buffers to every forward); gradients are what is averaged.
        net = DDP(model, device_ids=[device.index], bucket_cap_mb=bucket_cap_mb, broadcast_buffers=False,
                  gradient_as_bucket_view=True)
    else:
        net = DDP(model)
    if grad_dtype == torch.bfloat16:
        import torch.distributed as dist
        from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
        net.register_comm_hook(dist.group.WORLD, default_hooks.bf16_compress_hook)
    return net


def train_step(model, optimizer, image, depth, autocast_dtype=torch.bfloat16):
    """One iteration of the reference loop (src/train.py:86-114): forward, loss, zero_grad, backward, Adam step."""
    depth_n = depth_norm(depth)
    use_amp = autocast_dtype is not None and image.is_cuda
    with torch.autocast("cuda", dtype=autocast_dtype, enabled=use_amp):
        pred = model(image)
    loss = depth_loss(pred if pred.is_cuda else pred.float(), depth_n)
    optimizer.zero_grad(set_to_none=True)
    loss.backward()
    optimizer.step()
    return loss


def _unwrap(model):
    return model.module if hasattr(model, "module") and isinstance(model.module, nn.Module) else model


def save_checkpoint(path, model, optimizer, epoch, loss):
    """The reference loop's checkpoint (src/train.py:143-155): a dict with `epoch`, `model_state_dict`,
    `optimizer_state_dict`, `loss`.  A DDP-wrapped model is unwrapped first, so the keys are the reference's
    (`Unet.0...`, `Unet.1...`, never `module.`-prefixed) and the file loads into the reference, a single-GPU run or
    another DDP run alike.  Under torchrun call it on rank 0 only (parameters are replicated)."""
    loss_t = loss.detach().cpu() if torch.is_tensor(loss) else torch.tensor(float(loss))
    torch.save({"epoch": int(epoch), "model_state_dict": _unwrap(model).state_dict(),
                "optimizer_state_dict": optimizer.state_dict(), "loss": loss_t}, path)


def load_checkpoint(path, model, optimizer=None, map_location="cpu", trusted_pickle=False):
    """Resume as src/train.py:56-67 does: returns (epoch, loss).  Accepts checkpoints written by the reference loop
    (same format and keys) and ones whose keys carry a DDP `module.` prefix.  The format holds tensors, ints and plain
    dicts only, so the file is read with weights_only=True (no arbitrary unpickling); trusted_pickle=True is the explicit
    opt-in for legacy files that need the full unpickler."""
    ck = torch.load(path, map_location=map_location, weights_only=not trusted_pickle)
    sd = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in ck["model_state_dict"].items()}
    _unwrap(model).load_state_dict(sd, strict=True)
    if optimizer is not None and "optimizer_state_dict" in ck:
        optimizer.load_state_dict(ck["optimizer_state_dict"])
    return int(ck.get("epoch", 0)), ck.get("loss")


def synthetic_batches(n_batches, batch, height=480, width=640, seed=0, pin=None):
    """Stand-in for the reference's loader (src/data.py:179, consumed at src/train.py:86-89): yields dicts
    {'image': (B, 3, H, W) in [0, 1], 'depth': (B, 1, H, W)} of host tensors, NYU-shaped, pinned when CUDA is present."""
    gen = torch.Generator().manual_seed(seed)
    pin = torch.cuda.is_available() if pin is None else pin
    for _ in range(n_batches):
        sample = {"image": torch.rand(batch, 3, height, width, generator=gen),
                  "depth": torch.rand(batch, 1, height, width, generator=gen) * 9.0 + 1.0}
        yield {k: (t.pin_memory() if pin else t) for k, t in sample.items()}


def prefetch_to_device(batches, device, memory_format=torch.contiguous_format):
    """Iterate `batches` (dicts of host tensors, as the reference loop's `sample_batched`) one step ahead: the
    host -> device copy of batch i+1 runs on a copy stream while the caller computes on batch i (what bench.py's `e2e`
    measures).  On a CPU device the samples pass through unchanged."""
    device = torch.device(device)
    if device.type != "cuda":
        for sample in batches:
            yield sample
        return
    copy_stream = torch.cuda.Stream(device)

    def stage(sample):
        with torch.cuda.stream(copy_stream):
            out = {}
            for k, t in sample.items():
                fmt = memory_format if t.dim() == 4 and t.shape[1] > 1 else torch.contiguous_format
                out[k] = t.to(device, non_blocking=True, memory_format=fmt)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return out, ev

    it = iter(batches)
    nxt = None
    for sample in it:
        nxt = stage(sample)
        break
    while nxt is not None:
        cur, ev = nxt
        nxt = None
        for sample in it:
            nxt = stage(sample)
            break
        torch.cuda.current_stream(device).wait_event(ev)
        for t in cur.values():   # the consumer's stream now owns these buffers
            t.record_stream(torch.cuda.current_stream(device))
        yield cur


def _dense(t):
    """Non-overlapping and dense in memory (any permutation of a contiguous layout, e.g. channels-last)."""
    if t.is_contiguous() or (t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last)):
        return True
    sizes_strides = sorted(((st, sz) for sz, st in zip(t.size(), t.stride()) if sz > 1))
    expect = 1
    for st, sz in sizes_strides:
        if st != expect:
            return False
        expect *= sz
    return True


def _same_layout(a, b):
    """Same element order in memory: equal strides on every dimension longer than 1."""
    return a.size() == b.size() and all(sa == sb for n, sa, sb in zip(a.size(), a.stride(), b.stride()) if n > 1)


class LibAdam(torch.optim.Optimizer):
    """torch.optim.Adam(params, lr) of the reference loop (src/train.py:41, :108) as the library's multi-tensor step
    (crf_adam_step: 80 tensors per launch, pointers passed as launch arguments) instead of torch's multi-tensor launches;
    same update, same state layout (`exp_avg`, `exp_avg_sq`, `step` per parameter), so optimizer_state_dict entries of
    the reference's checkpoints load.  The step counter lives on the device, hence a CUDA graph that captured the step
    keeps counting on replay.  CUDA fp32 parameters only.

    Status: the element update is verified on the host against torch.optim.Adam (tests/test_adam_host.py) and on a B200
    against torch.optim.Adam over several steps incl. channels-last weights, an unaligned view and state_dict round trips
    (tests/test_gpu_stages.py::test_lib_adam_matches_torch_adam, 1e-5); measured in the training step (round 2): 0.28 ms
    for the model's 302 tensors, 13.9 ms per step against 14.15-14.5 with torch's fused Adam, same loss trajectory --
    `bench.py` uses it by default (`--torch-adam` for torch's)."""

    CHUNK = 16384   # elements per CTA (64 KB of each of p, g, m, v)

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        if lr < 0 or eps < 0 or not (0 <= betas[0] < 1 and 0 <= betas[1] < 1) or weight_decay < 0:
            raise ValueError("LibAdam: invalid hyper-parameters")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    @staticmethod
    def chunk_counts(numels, chunk):
        """CTAs per tensor: crf_adam_step gives CTA c of a tensor the elements [c * chunk, min(n, (c + 1) * chunk))."""
        return [(int(n) + chunk - 1) // chunk for n in numels]

    def _init_group(self, group):
        ps = [p for p in group["params"] if p.requires_grad]
        for p in ps:
            if not (p.is_cuda and p.dtype == torch.float32 and _dense(p)):
                raise RuntimeError("LibAdam: parameters must be dense CUDA fp32 tensors (there is no CPU path)")
        missing = [p for p in ps if "exp_avg" not in self.state[p]]
        if missing:
            dev = missing[0].device
            sizes = [(p.numel() + 3) // 4 * 4 for p in missing]           # keep every view 16-byte aligned
            flat_m = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
            flat_v = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
            if group.get("_step") is None:
                group["_step"] = torch.zeros((), dtype=torch.float32, device=dev)
            o = 0
            for p, n in zip(missing, sizes):
                self.state[p]["step"] = group["_step"]
                # the update is element-wise over memory: the moments take the parameter's own (dense) strides, so a
                # channels-last convolution weight keeps its layout
                self.state[p]["exp_avg"] = flat_m[o:o + p.numel()].as_strided(p.size(), p.stride())
                self.state[p]["exp_avg_sq"] = flat_v[o:o + p.numel()].as_strided(p.size(), p.stride())
                o += n
        return ps

    def state_dict(self):
        """torch.optim.Adam's layout: an independent CPU fp32 scalar `step` per parameter (here all parameters of a
        group share ONE device counter, which must not leak into a checkpoint as ~300 aliases of the same storage: a
        torch.optim.Adam resumed from it would advance the shared tensor once per parameter) and no private keys in
        param_groups.  A checkpoint written here therefore resumes in torch.optim.Adam (the reference loop) and here."""
        sd = super().state_dict()
        for st in sd["state"].values():
            if "step" in st:
                st["step"] = torch.tensor(float(st["step"]), dtype=torch.float32)
        for grp in sd["param_groups"]:
            grp.pop("_step", None)
        return sd

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        for group in self.param_groups:   # one device counter per group again (torch keeps one per parameter)
            have = [p for p in group["params"] if p in self.state and "step" in self.state[p]]
            if have:
                step = torch.as_tensor(float(self.state[have[0]]["step"]), dtype=torch.float32)
                group["_step"] = step.to(have[0].device).reshape(())
                for p in have:
                    self.state[p]["step"] = group["_step"]
                    for k in ("exp_avg", "exp_avg_sq"):
                        t = self.state[p][k].to(device=p.device, dtype=torch.float32)
                        if not _same_layout(t, p):
                            t = torch.empty_strided(p.size(), p.stride(), dtype=torch.float32, device=p.device).copy_(t)
                        self.state[p][k] = t

    @torch.no_grad()
    def step(self, closure=None):
        import ctypes as C
        from . import _lib as L
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for group in self.param_groups:
            ps = [p for p in self._init_group(group) if p.grad is not None]
            if not ps:
                continue
            dev = ps[0].device
            recs = (L.AdamTensor * len(ps))()
            for r, p in zip(recs, ps):
                g = p.grad
                if g.dtype != torch.float32 or g.device != dev:
                    raise RuntimeError("LibAdam: gradients must be fp32 tensors on the parameters' device")
                if not _same_layout(g, p):   # rare: re-lay the gradient out like the parameter (element-wise update)
                    g = torch.empty_strided(p.size(), p.stride(), dtype=torch.float32, device=dev).copy_(g)
                st = self.state[p]
                r.p, r.g, r.m, r.v, r.n = p.data_ptr(), g.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), p.numel()
            b1, b2 = group["betas"]
            L.check(L.lib().crf_adam_step(recs, len(ps), self.CHUNK, float(group["lr"]), float(b1), float(b2),
                                          float(group["eps"]), float(group["weight_decay"]), group["_step"].data_ptr(),
                                          dev.index, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
                    "crf_adam_step")
        return loss
