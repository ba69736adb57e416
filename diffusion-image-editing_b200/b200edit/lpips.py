"""Native LPIPS distance (lpips v0.1, ``lpips.LPIPS(net='vgg')``) on libb200edit.so, differentiable w.r.t. its first
input - the regulariser of the masked-prediction guidance (``AttrFunc(..., use_lpips=True)``: ``loss(mask * x0') +
lambda_ * LPIPS(1 - mask * x0', x_0)``) and the ``metrics.lpips`` distance.

The VGG-16 trunk runs on the tcgen05 implicit-GEMM kernel with ReLU in the epilogue (conv1_1 as a 1x1 GEMM over an
im2col tensor that the input packer forms from the scaled input), the distance head and the max pools on their own
kernels, the input gradient on the dgrad twins of the same convolutions.  The second input is constant for a whole edit:
its normalised features are computed once and cached in the engine (re-run only when that tensor changes)."""
from __future__ import annotations

from types import SimpleNamespace

import torch

from . import _C
from ._C import LpipsConfig, lib
from .engine import Engine, _ptr, _stream

# (slice, index in vgg16().features, in channels, out channels) of the thirteen convolutions
VGG16_CONVS = ((1, 0, 3, 64), (1, 2, 64, 64), (2, 5, 64, 128), (2, 7, 128, 128), (3, 10, 128, 256), (3, 12, 256, 256),
               (3, 14, 256, 256), (4, 17, 256, 512), (4, 19, 512, 512), (4, 21, 512, 512), (5, 24, 512, 512),
               (5, 26, 512, 512), (5, 28, 512, 512))
LIN_CHANNELS = (64, 128, 256, 512, 512)
SCALING_SHIFT = (-.030, -.088, -.188)
SCALING_SCALE = (.458, .448, .450)


class LPIPS(Engine):
    """``d = LPIPS(...)(in0, in1)``: (B, 1, 1, 1), like ``lpips.LPIPS.forward``; in0 (B, 3, S, S) and in1 (1 | B, 3, S, S)
    fp32 CUDA tensors in [-1, 1].  Autograd node in ``in0`` only; parameters under ``lpips.LPIPS().state_dict()`` names."""

    _ref = None             # the reference tensor whose features the engine holds (kept alive: identity check)
    _mask = None            # the mask the engine reads in the backward of the last forward (kept alive)

    def __init__(self, net="vgg", input_size=256, max_batch=1, device="cuda", precision="fp32"):
        """precision: "fp32" (default) - fp32-accurate FORWARD (split 16-bit operands, three tensor-core products per
        GEMM), so that the ReLU / max-pool masks of the input gradient agree with an fp32 evaluation; None / "fp16" - 16-bit
        operands throughout.  The backward pass runs on 16-bit operands either way."""
        if net != "vgg":
            raise ValueError(f"LPIPS: only net='vgg' is implemented (got {net!r})")
        _C.require_device()
        self.precision, precision_cfg = _C.resolve_precision(precision, "LPIPS")
        self.config = SimpleNamespace(net=net, input_size=input_size, sample_size=input_size, in_channels=3, out_channels=1)
        cfg = LpipsConfig()
        cfg.input_size, cfg.precision = input_size, precision_cfg
        self._create(lib.b2e_lpips_create, cfg, max_batch, device)

    # ------------------------------------------------------------------ parameters
    def load_state_dict(self, sd, strict=True):
        """The full ``lpips.LPIPS(net='vgg').state_dict()``: ``net.slice*``, ``lin*.model.1.weight`` and the scaling
        layer's constants, which are checked (they are built into the engine, not parameters)."""
        sd = dict(sd)
        for name, ref in (("scaling_layer.shift", SCALING_SHIFT), ("scaling_layer.scale", SCALING_SCALE)):
            v = sd.pop(name, None)
            if v is not None and not torch.allclose(v.detach().float().cpu().reshape(-1), torch.tensor(ref), atol=1e-6):
                raise ValueError(f"LPIPS: {name} = {v.reshape(-1).tolist()} differs from lpips v0.1's {list(ref)}")
        missing, unexpected = super().load_state_dict(sd, strict)
        self._ref = None
        return missing, unexpected

    load_lpips_state_dict = load_state_dict

    @staticmethod
    def from_vgg16_features(features_sd, lin_weights):
        """A torchvision ``vgg16().features`` state dict (keys "<index>.weight" / "<index>.bias") plus five lin weight
        tensors -> an lpips state dict (names mapped by index)."""
        sd = {}
        for s, i, _, _ in VGG16_CONVS:
            for p in ("weight", "bias"):
                sd[f"net.slice{s}.{i}.{p}"] = features_sd[f"{i}.{p}"]
        for k, w in enumerate(lin_weights):
            sd[f"lin{k}.model.1.weight"] = w.reshape(1, LIN_CHANNELS[k], 1, 1)
        return sd

    def random_state_dict(self, seed=0):
        """Seeded weights in lpips' layout: convolutions as torchvision initialises VGG (Kaiming normal, fan_out, ReLU
        gain) with small random biases; lin weights non-negative, as in trained LPIPS."""
        return lpips_random_state_dict(seed)

    # ------------------------------------------------------------------ forward / backward
    _backward_fn = lib.b2e_lpips_backward

    def enable_grad(self, enable: bool = True):
        self._enable_grad(enable)
        self._ref = None                # the engine dropped the cached reference with the workspace
        return self

    def _check(self, x, what, batch_ok):
        if not torch.is_tensor(x) or not x.is_cuda:
            raise _C.B2EError(f"LPIPS: {what} must be a CUDA tensor (no CPU fallback)")
        S = self.config.input_size
        if x.dim() != 4 or tuple(x.shape[1:]) != (3, S, S) or not batch_ok(x.shape[0]):
            raise ValueError(f"LPIPS: {what} must be (B <= {self.max_batch}, 3, {S}, {S}) (got {tuple(x.shape)})")
        return x if (x.dtype == torch.float32 and x.is_contiguous()) else x.to(torch.float32).contiguous()

    def set_reference(self, in1):
        """Normalised features of ``in1`` (1 or B images) into the engine's cache; skipped when ``in1`` is the very tensor
        of the last call, unmodified since (identity and version counter; the wrapper holds a reference to it, so its
        memory cannot be reused by another tensor)."""
        if self._ref is not None and in1 is self._ref[0] and in1._version == self._ref[1]:
            return
        x = self._check(in1, "in1", lambda b: 1 <= b <= self.max_batch).detach()
        self._ref = None
        self._launch(lib.b2e_lpips_set_reference, _ptr(x), x.shape[0], _stream())
        self._ref = (in1, in1._version)

    def _forward(self, x, mask=None):
        self._mask = mask           # the backward's -mask chain reads this memory: it lives until the next forward
        B = x.shape[0]
        dist = torch.empty((B, 1, 1, 1), dtype=torch.float32, device=x.device)
        self._launch(lib.b2e_lpips_forward, _ptr(x), _ptr(mask), 0 if mask is None else mask.shape[0], _ptr(dist), B,
                     _stream())
        return dist

    def __call__(self, in0, in1, normalize=False, mask=None):
        """LPIPS(in0, in1) (B, 1, 1, 1).  ``mask`` (extension, 1 | B, 3, S, S): the distance of ``1 - mask * in0`` -
        the regulariser's input transform, formed inside the input packer (autograd flows to ``in0``)."""
        if normalize:
            raise ValueError("LPIPS: normalize=True (inputs in [0, 1]) is not implemented; pass inputs in [-1, 1]")
        if torch.is_tensor(in1) and in1.requires_grad:
            raise _C.B2EError("LPIPS: no gradient w.r.t. in1 (the reference image); detach it")
        x = self._check(in0, "in0", lambda b: 1 <= b <= self.max_batch)
        B = x.shape[0]
        if not torch.is_tensor(in1) or in1.dim() != 4 or in1.shape[0] not in (1, B):
            raise ValueError(f"LPIPS: in1 must have batch 1 or {B} (got {tuple(in1.shape) if torch.is_tensor(in1) else in1})")
        if mask is not None:
            mask = self._check(mask.expand(mask.shape[0], 3, *mask.shape[2:]) if mask.dim() == 4 and mask.shape[1] == 1
                               else mask, "mask", lambda b: b in (1, B)).detach()
        self.set_reference(in1)
        if x.requires_grad and torch.is_grad_enabled():
            return self._keep_node(x, mask)
        return self._keep(x.detach(), mask)

    forward = __call__

    def input_grad(self, d_dist):
        """d(sum_b d_dist[b] * dist[b]) / d(in0) of the last forward (through its mask transform), without autograd."""
        return self._keep_grad(d_dist)

    def profile(self, in0):
        x = self._check(in0, "in0", lambda b: 1 <= b <= self.max_batch).detach()
        self._mask = None           # profiling forwards run without a mask
        return self._profile(x, None, torch.empty((x.shape[0],), dtype=torch.float32, device=x.device))


def lpips_random_state_dict(seed=0):
    """Seeded LPIPS (vgg) state dict with lpips' names and shapes (CPU fp32)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for s, i, cin, cout in VGG16_CONVS:
        std = (2.0 / (cout * 9)) ** 0.5
        sd[f"net.slice{s}.{i}.weight"] = torch.randn(cout, cin, 3, 3, generator=g) * std
        sd[f"net.slice{s}.{i}.bias"] = (torch.rand(cout, generator=g) * 2 - 1) * 0.05
    for k, c in enumerate(LIN_CHANNELS):
        sd[f"lin{k}.model.1.weight"] = torch.rand(1, c, 1, 1, generator=g) * (2.0 / c) ** 0.5
    sd["scaling_layer.shift"] = torch.tensor(SCALING_SHIFT).view(1, 3, 1, 1)
    sd["scaling_layer.scale"] = torch.tensor(SCALING_SCALE).view(1, 3, 1, 1)
    return sd
