"""N>1 host logic on CPU (gloo, world_size 2): the data-parallel wrapper shards the batch with no data-path collective
and averages parameter gradients; the averaged gradients must equal the single-process gradients of the concatenated
batch (SURVEY.md 8e).  The CRF math here is the oracle's (CPU); the CUDA path is covered by the -m gpu tests."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

from monocular_depth_estimation_b200 import training as T


class _TinyDepthNet(nn.Module):
    """A NewCRF stage (oracle math) between two convs: same structure as one decoder stage + head."""

    def __init__(self):
        super().__init__()
        from oracle.model_oracle import OracleNewCRF
        self.stem = nn.Conv2d(3, 16, 3, padding=1)
        self.crf = OracleNewCRF(input_dim=16, embed_dim=64, v_dim=16, num_heads=2)
        self.head = nn.Conv2d(64, 1, 3, padding=1)

    def forward(self, img):
        f = self.stem(img)
        return torch.sigmoid(self.head(self.crf(f, f)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _data(n):
    g = torch.Generator().manual_seed(7)
    # pre-normalised depth: DepthNorm is a per-batch min-max, so per-rank normalisation would differ from global
    return torch.rand(n, 3, 9, 10, generator=g), torch.rand(n, 1, 9, 10, generator=g)


def _worker(rank, world, port, out_path, grad_dtype=None):
    # the CPU / gloo path also on a host with GPUs: this spawned process has not initialised CUDA yet, so hiding the
    # devices here makes init_distributed() choose the CPU (with GPUs it would take cuda:<local rank> and NCCL)
    os.environ.update({"RANK": str(rank), "LOCAL_RANK": str(rank), "WORLD_SIZE": str(world),
                       "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(port), "CUDA_VISIBLE_DEVICES": ""})
    torch.set_num_threads(1)
    r, lr, w, device = T.init_distributed()
    assert (r, w, device.type) == (rank, world, "cpu")
    torch.manual_seed(0)
    model = _TinyDepthNet()
    net = T.wrap_ddp(model, device, w, grad_dtype=grad_dtype)
    img, dep = _data(4)
    shard = slice(rank * 2, rank * 2 + 2)                     # batch-sharded: whole images per rank
    loss = T.depth_loss(net(img[shard]), dep[shard])
    loss.backward()
    if rank == 0:
        torch.save({k: p.grad.clone() for k, p in model.named_parameters()}, out_path)
    dist.barrier()
    dist.destroy_process_group()


def test_ddp_gradients_equal_full_batch_gradients(tmp_path):
    out = str(tmp_path / "grads.pt")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = torch.load(out)
    torch.manual_seed(0)
    model = _TinyDepthNet()
    img, dep = _data(4)
    # mean over ranks of per-shard losses == loss terms averaged over equal shards
    loss = 0.5 * (T.depth_loss(model(img[:2]), dep[:2]) + T.depth_loss(model(img[2:]), dep[2:]))
    loss.backward()
    for k, p in model.named_parameters():
        assert torch.allclose(got[k], p.grad, rtol=1e-4, atol=1e-6), k


def test_ddp_bf16_gradient_exchange(tmp_path):
    """Optional bf16 bucket exchange (wrap_ddp(grad_dtype=torch.bfloat16)): same averaged gradients up to the bf16
    rounding of the exchanged values."""
    out = str(tmp_path / "grads_bf16.pt")
    mp.spawn(_worker, args=(2, _free_port(), out, torch.bfloat16), nprocs=2, join=True)
    got = torch.load(out)
    torch.manual_seed(0)
    model = _TinyDepthNet()
    img, dep = _data(4)
    loss = 0.5 * (T.depth_loss(model(img[:2]), dep[:2]) + T.depth_loss(model(img[2:]), dep[2:]))
    loss.backward()
    for k, p in model.named_parameters():
        assert got[k].dtype == torch.float32
        err = float((got[k] - p.grad).norm() / p.grad.norm().clamp_min(1e-30))
        assert err < 1e-2, (k, err)
    assert any(not torch.equal(got[k], p.grad) for k, p in model.named_parameters())   # the hook really ran


def test_loss_matches_oracle_loss():
    from oracle import model_oracle as MO
    torch.manual_seed(1)
    a, b = torch.rand(2, 1, 24, 32), torch.rand(2, 1, 24, 32)
    assert torch.allclose(T.depth_loss(a, b), MO.ssim_l1_loss(a, b), rtol=1e-6)
    assert torch.equal(T.depth_norm(b), MO.depth_norm(b))
