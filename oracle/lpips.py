"""Oracle restatement of ``lpips.LPIPS(net='vgg')`` (lpips v0.1, ``normalize=False``) - the distance of the reference's
``apply_lpips`` regulariser (src/attr_functions.py) and of ``metrics.lpips``.

TEST INFRASTRUCTURE (see oracle/__init__.py).  PARITY UNPINNED: the ``lpips`` package is neither vendored nor installed
and the reference holds no golden vectors for it; this file restates the published algorithm and is the normative spec
for the native engine (b200edit.lpips):

    x' = (x - shift) / scale, shift = (-.030, -.088, -.188), scale = (.458, .448, .450)
    VGG-16 features[0:30] in five slices [0:4], [4:9], [9:16], [16:23], [23:30]; taps relu1_2 .. relu5_3
    per tap: u = f / (sqrt(sum_c f_c^2) + 1e-10); d = lin_k((u0 - u1)^2) (1x1 conv, no bias); spatial mean
    result: sum over the taps, (B, 1, 1, 1); in1 may have batch 1 (broadcast)

State-dict names follow ``lpips.LPIPS().state_dict()`` (``net.slice1.0.weight`` .. ``net.slice5.28.bias``,
``lin0.model.1.weight`` .. ``lin4.model.1.weight``, ``scaling_layer.shift`` / ``.scale``).  Any dtype and device.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torchvision

SLICES = ((0, 4), (4, 9), (9, 16), (16, 23), (23, 30))
CHANNELS = (64, 128, 256, 512, 512)


class ScalingLayer(nn.Module):
    def __init__(self):
        super().__init__()
        self.register_buffer("shift", torch.tensor([-.030, -.088, -.188])[None, :, None, None])
        self.register_buffer("scale", torch.tensor([.458, .448, .450])[None, :, None, None])

    def forward(self, x):
        return (x - self.shift) / self.scale


class VGG16Slices(nn.Module):
    def __init__(self):
        super().__init__()
        features = torchvision.models.vgg16(weights=None).features
        for k, (a, b) in enumerate(SLICES):
            s = nn.Sequential()
            for i in range(a, b):
                s.add_module(str(i), features[i])
            setattr(self, f"slice{k + 1}", s)

    def forward(self, x):
        outs = []
        for k in range(5):
            x = getattr(self, f"slice{k + 1}")(x)
            outs.append(x)
        return outs


class NetLinLayer(nn.Module):
    def __init__(self, chn_in):
        super().__init__()
        self.model = nn.Sequential(nn.Dropout(), nn.Conv2d(chn_in, 1, 1, stride=1, padding=0, bias=False))

    def forward(self, x):
        return self.model(x)


def normalize_tensor(x, eps=1e-10):
    norm_factor = torch.sqrt(torch.sum(x ** 2, dim=1, keepdim=True))
    return x / (norm_factor + eps)


class LPIPS(nn.Module):
    def __init__(self, net="vgg"):
        super().__init__()
        if net != "vgg":
            raise ValueError("oracle LPIPS: net='vgg' only")
        self.scaling_layer = ScalingLayer()
        self.net = VGG16Slices()
        for k, c in enumerate(CHANNELS):
            setattr(self, f"lin{k}", NetLinLayer(c))
        self.eval()
        for p in self.parameters():
            p.requires_grad_(False)

    def forward(self, in0, in1, normalize=False):
        if normalize:
            raise ValueError("oracle LPIPS: normalize=True is out of scope")
        outs0, outs1 = self.net(self.scaling_layer(in0)), self.net(self.scaling_layer(in1))
        val = 0
        for k in range(5):
            diff = (normalize_tensor(outs0[k]) - normalize_tensor(outs1[k])) ** 2
            val = val + getattr(self, f"lin{k}")(diff).mean(dim=(2, 3), keepdim=True)
        return val
