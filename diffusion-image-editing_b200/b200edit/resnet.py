"""Native classifier network: torchvision ResNet (the attribute predictor of src/models.py:69-77, ``resnet50`` with an
80-way ``fc``) on libb200edit.so, differentiable w.r.t. its input - what ``ClassifierAttrFunc.loss``
(src/attr_functions.py:237-257) needs from it: ``predictor(image)`` inside an autograd graph.

Eval-mode BatchNorm is folded into the convolution weights / biases when a torchvision ``state_dict`` is loaded; every
convolution runs on the tcgen05 implicit-GEMM kernel (bf16 operands, fp32 accumulation) with ReLU in the epilogue and
the block shortcut fused as a K segment; the input gradient runs on the dgrad twins of the same kernel."""
from __future__ import annotations

from types import SimpleNamespace

import torch

from . import _C
from ._C import ResNetConfig, lib
from .engine import Engine

RESNET50_LAYERS = (3, 4, 6, 3)


class ResNet(Engine):
    """``logits = net(image)``; image (B, C, S, S) fp32 CUDA, S a power of two >= 64."""

    def __init__(self, block="bottleneck", layers=RESNET50_LAYERS, num_classes=80, input_size=256, in_channels=3, width=64,
                 max_batch=8, device="cuda", precision=None):
        """precision: None / "fp16" - f16 operands throughout; "fp32" - fp32-accurate FORWARD (split f16 operands, three
        tensor-core products per GEMM) so that the ReLU / max-pool masks of the input gradient agree with an fp32 evaluation
        of the network; the backward pass stays on f16 operands."""
        _C.require_device()
        self.precision, precision_cfg = _C.resolve_precision(precision, "ResNet")
        if block not in ("bottleneck", "basic"):
            raise ValueError("ResNet: block must be 'bottleneck' or 'basic'")
        self.config = SimpleNamespace(block=block, layers=tuple(layers), num_classes=num_classes, input_size=input_size,
                                      in_channels=in_channels, sample_size=input_size, out_channels=num_classes, width=width)
        cfg = ResNetConfig()
        cfg.input_size, cfg.in_channels, cfg.bottleneck = input_size, in_channels, int(block == "bottleneck")
        for i in range(4):
            cfg.layers[i] = layers[i]
        cfg.width, cfg.num_classes = width, num_classes
        cfg.precision = precision_cfg
        self._create(lib.b2e_resnet_create, cfg, max_batch, device)

    # ------------------------------------------------------------------ parameters
    @staticmethod
    def fold_batchnorm(sd, eps=1e-5):
        """torchvision ResNet state_dict (conv without bias + BatchNorm running statistics) -> folded convolution
        weights / biases under the convolution names the engine uses."""
        out = {}
        for k, w in sd.items():
            if k.endswith(".weight") and w.dim() == 4:
                conv = k[:-len(".weight")]
                if conv.endswith("downsample.0"):
                    bn = conv[:-1] + "1"
                else:
                    head, last = conv.rsplit("conv", 1) if "conv" in conv else (None, None)
                    bn = f"{head}bn{last}"
                g, b = sd[bn + ".weight"].double(), sd[bn + ".bias"].double()
                mu, var = sd[bn + ".running_mean"].double(), sd[bn + ".running_var"].double()
                s = g / torch.sqrt(var + eps)
                out[conv + ".weight"] = (w.double() * s.view(-1, 1, 1, 1)).float()
                out[conv + ".bias"] = (b - mu * s).float()
        out["fc.weight"], out["fc.bias"] = sd["fc.weight"].float(), sd["fc.bias"].float()
        return out

    def load_torchvision_state_dict(self, sd, eps=1e-5):
        return self.load_state_dict(self.fold_batchnorm(sd, eps))

    # ------------------------------------------------------------------ forward / backward
    _backward_fn = lib.b2e_resnet_backward

    def _out_shape(self, B):
        return (B, self.config.num_classes)

    def _check_input(self, image):
        if not image.is_cuda:
            raise _C.B2EError("ResNet: image must be a CUDA tensor (no CPU fallback)")
        cfg = self.config
        if tuple(image.shape[1:]) != (cfg.in_channels, cfg.input_size, cfg.input_size):
            raise ValueError(f"ResNet: expected (B,{cfg.in_channels},{cfg.input_size},{cfg.input_size}), got {tuple(image.shape)}")
        if image.shape[0] > self.max_batch:
            raise ValueError(f"ResNet: batch {image.shape[0]} > max_batch {self.max_batch}")

    def forward_keep(self, image):
        """``net(image)`` with the activations kept in the engine's workspace for ``input_grad`` (no autograd graph)."""
        self._check_input(image)
        return self._keep(image.detach().to(torch.float32).contiguous())

    def input_grad(self, d_logits):
        """d(loss)/d(image) of the last ``forward_keep`` given d(loss)/d(logits) (native dgrad of the whole network)."""
        return self._keep_grad(d_logits)

    def __call__(self, image):
        self._check_input(image)
        x = image if (image.dtype == torch.float32 and image.is_contiguous()) else image.to(torch.float32).contiguous()
        if x.requires_grad and torch.is_grad_enabled():
            return self._keep_node(x)
        return self._forward(x.detach())

    forward = __call__

    def profile(self, image):
        x = image.detach().to(torch.float32).contiguous()
        return self._profile(x, None, torch.empty(self._out_shape(x.shape[0]), dtype=torch.float32, device=x.device))


def resnet50_predictor(num_classes=80, input_size=256, max_batch=8, state_dict=None, seed=0, precision=None):
    """The attribute predictor of src/models.py:69-77 (``models.resnet50()`` with ``fc = Linear(2048, 40 * 2)``)."""
    net = ResNet("bottleneck", RESNET50_LAYERS, num_classes, input_size, max_batch=max_batch, precision=precision)
    if state_dict is not None:
        net.load_torchvision_state_dict(state_dict)
    else:
        net.init_random(seed)
    return net
