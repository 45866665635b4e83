"""The caller of the hot path: MobileNetV3-large encoder + NeWCRFs decoder, same module tree (and therefore the same
state_dict keys) as /root/reference/src/model_mobileV3_large_newCRFs.py:60-193, with the four `NewCRF` stages backed
by the sm_100a CRF block.  Encoder and the plain convolutions stay on stock PyTorch/cuDNN (SURVEY.md 8f: "next" rows).

Decoder wiring (model_mobileV3_large_newCRFs.py:113-124):
    bridge = conv0(feats[17]);  e3 = crf3(feats[16], bridge);  e2 = crf2(feats[13], PixelShuffle2(e3));
    e1 = crf1(feats[7], PixelShuffle2(e2));  e0 = crf0(feats[4], PixelShuffle2(e1));
    depth = upsample x4 (sigmoid(conv1(e0)))
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from .newcrf_layers import NewCRF

CRF_DIMS = (128, 256, 512, 1024)      # embed dim per scale 1/4 .. 1/32
V_DIMS = (64, 128, 256, 512)          # depth-feature channels entering each stage
NUM_HEADS = (4, 8, 16, 32)
ENC_CHANNELS = (24, 40, 112, 160, 960)
ENC_TAPS = (4, 7, 13, 16, 17)         # indices into the encoder feature list


class Decoder(nn.Module):
    def __init__(self, window_size=7):
        super().__init__()
        self.conv0 = nn.Conv2d(ENC_CHANNELS[4], V_DIMS[3], kernel_size=1, stride=1)
        for s in (3, 2, 1, 0):
            setattr(self, f"crf{s}", NewCRF(input_dim=ENC_CHANNELS[s], embed_dim=CRF_DIMS[s], window_size=window_size,
                                            v_dim=V_DIMS[s], num_heads=NUM_HEADS[s]))
        self.conv1 = nn.Conv2d(CRF_DIMS[0], 1, 3, padding=1)
        self.sigmoid = nn.Sigmoid()

    def forward(self, feats):
        e = self.conv0(feats[ENC_TAPS[4]])
        for s in (3, 2, 1, 0):
            # nn.PixelShuffle(2) between the stages (model_mobileV3_large_newCRFs.py:116-120) is folded into the store of
            # the producing stage's closing LayerNorm (no separate permutation pass)
            e = getattr(self, f"crf{s}")(feats[ENC_TAPS[s]], e, pixel_shuffle=(s != 0))
        d = self.sigmoid(self.conv1(e))
        return F.interpolate(d, scale_factor=4, mode="bilinear", align_corners=False)


_ACTS = {"relu": nn.ReLU, "hardswish": nn.Hardswish}
_ACT_FNS = {"relu": F.relu, "hardswish": F.hardswish}


class BatchNormAct2d(nn.BatchNorm2d):
    """nn.BatchNorm2d followed by an activation (act: None, "relu" or "hardswish"), with nn.BatchNorm2d's parameters,
    buffers and state_dict.  In training mode on a CUDA bf16 channels-last map with C % 8 == 0 it runs on the library's
    BatchNorm kernels (functional.batch_norm_act: two launches each way, only x and the statistics saved for the
    backward); every other case runs act(nn.BatchNorm2d.forward(x)) unchanged."""

    def __init__(self, num_features, eps=1e-5, momentum=0.1, affine=True, track_running_stats=True, act=None,
                 device=None, dtype=None):
        super().__init__(num_features, eps, momentum, affine, track_running_stats, device, dtype)
        if act not in (None, *_ACTS):
            raise ValueError(f"act must be None, 'relu' or 'hardswish' (got {act!r})")
        self.act = act
        self._tickets = None   # the kernels' per-launch counters (not state: always zero between launches)

    @classmethod
    def from_batchnorm(cls, bn, act=None):
        """A BatchNormAct2d that holds bn's own parameter and buffer tensors (shared, not copied)."""
        m = cls(bn.num_features, bn.eps, bn.momentum, bn.affine, bn.track_running_stats, act=act, device="meta")
        m._parameters.update(bn._parameters)
        m._buffers.update(bn._buffers)
        m.train(bn.training)
        return m

    def _library(self, x):
        return (self.training and self.track_running_stats and self.affine and isinstance(self.momentum, float)
                and x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 4
                and x.is_contiguous(memory_format=torch.channels_last) and x.data_ptr() % 16 == 0
                and x.shape[1] % 8 == 0 and x.shape[0] * x.shape[2] * x.shape[3] >= 2
                and self.weight.dtype == torch.float32 and self.running_mean.dtype == torch.float32)

    def forward(self, x):
        if self._library(x):
            from .functional import batch_norm_act
            if self._tickets is None or self._tickets.device != x.device:
                self._tickets = torch.zeros(self.num_features // 8, dtype=torch.int32, device=x.device)
            return batch_norm_act(x, self.weight, self.bias, self.running_mean, self.running_var,
                                  self.num_batches_tracked, self._tickets, self.eps, self.momentum, self.act)
        y = super().forward(x)
        return y if self.act is None else _ACT_FNS[self.act](y, inplace=True)   # as torchvision's inplace modules

    def extra_repr(self):
        return super().extra_repr() + f", act={self.act}"


def fuse_batchnorm_act(features):
    """Replaces, inside every torchvision Conv2dNormActivation of `features`, the BatchNorm2d (index 1) by a
    BatchNormAct2d holding the same tensors and the ReLU / Hardswish after it (index 2) by nn.Identity.  Keys, shapes and
    dtypes of the state_dict stay torchvision's."""
    from torchvision.ops.misc import Conv2dNormActivation
    for mod in features.modules():
        if not isinstance(mod, Conv2dNormActivation) or type(mod[1]) is not nn.BatchNorm2d:
            continue
        act = None
        if len(mod) > 2:
            act = next((k for k, cls in _ACTS.items() if type(mod[2]) is cls), None)
            if act is None:
                continue
            mod[2] = nn.Identity()
        mod[1] = BatchNormAct2d.from_batchnorm(mod[1], act)
    return features


class Encoder(nn.Module):
    """torchvision MobileNetV3-large feature stack; keeps every intermediate map (18 tensors incl. the input).  Its 46
    BatchNorm layers, with the activation that follows each, are BatchNormAct2d modules."""

    def __init__(self, pretrained=False):
        super().__init__()
        import torchvision.models as tvm
        weights = tvm.MobileNet_V3_Large_Weights.IMAGENET1K_V1 if pretrained else None
        self.original_model = tvm.mobilenet_v3_large(weights=weights)
        fuse_batchnorm_act(self.original_model.features)

    def forward(self, x):
        feats = [x]
        for layer in self.original_model.features:
            feats.append(layer(feats[-1]))
        return feats


class PTModel(nn.Module):
    def __init__(self, pretrained_encoder=False):
        super().__init__()
        self.Unet = nn.Sequential(Encoder(pretrained_encoder), Decoder())

    def forward(self, x):
        return self.Unet(x)
