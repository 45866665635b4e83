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


class Encoder(nn.Module):
    """torchvision MobileNetV3-large feature stack; keeps every intermediate map (18 tensors incl. the input)."""

    def __init__(self, pretrained=False):
        super().__init__()
        import torchvision.models as tvm
        weights = tvm.MobileNet_V3_Large_Weights.IMAGENET1K_V1 if pretrained else None
        self.original_model = tvm.mobilenet_v3_large(weights=weights)

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
