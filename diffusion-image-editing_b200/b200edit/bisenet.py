"""Native face parser: the reference's ``BiSeNet`` (src/Segmentation/model.py:234-262 on the ResNet-18 of
src/Segmentation/resnet.py) on libb200edit.so - the network behind ``SegmentationModel`` (src/models.py:80-118), whose
parsing map feeds the mask path (``prepare_for_edit``, src/SegDiffEditPipeline.py:79-97), and ``NetAttrFunc.loss``
(src/attr_functions.py:213-219), which differentiates through it.  ``net(x)[0]`` = logits (B, n_classes, S, S) like the
reference's first output; after ``enable_grad()`` the call is an autograd node backed by the native input gradient.

Eval-mode BatchNorm is folded into the convolutions when the reference's ``state_dict`` is loaded; convolutions run on
the tcgen05 implicit-GEMM kernel with ReLU in the epilogue, the channel-attention branches (global pooling -> 1x1
convolutions -> sigmoid) as small fp32 kernels, the final align_corners bilinear upsampling as one kernel."""
from __future__ import annotations

from types import SimpleNamespace

import torch

from . import _C
from ._C import ResNetConfig, lib
from .engine import Engine, _ptr, _stream


def _fold(w, sd, bn, eps=1e-5):
    g, b = sd[bn + ".weight"].double(), sd[bn + ".bias"].double()
    mu, var = sd[bn + ".running_mean"].double(), sd[bn + ".running_var"].double()
    s = g / torch.sqrt(var + eps)
    return (w.double() * s.view(-1, 1, 1, 1)).float(), (b - mu * s).float()


class BiSeNet(Engine):
    differentiable = False

    def __init__(self, n_classes=19, input_size=512, max_batch=1, device="cuda", precision=None, grad_precision=None):
        """precision: None / "fp16" - f16 operands throughout; "fp32" - fp32-accurate FORWARD (split f16 operands), so
        the ReLU / max-pool masks the backward pass routes gradients with are those of the fp32 network.  grad_precision:
        None - 16-bit backward; "fp32" (needs precision="fp32") - fp32-accurate backward (see b200edit.resnet.ResNet)."""
        self.precision, precision_cfg = _C.resolve_precision(precision, "BiSeNet")
        grad_cfg = _C.resolve_grad_precision(grad_precision, self.precision, "BiSeNet")
        _C.require_device()
        self.grad_precision = grad_precision
        self.config = SimpleNamespace(n_classes=n_classes, input_size=input_size, in_channels=3, sample_size=input_size,
                                      out_channels=n_classes)
        cfg = ResNetConfig()
        cfg.input_size, cfg.in_channels, cfg.bottleneck, cfg.width, cfg.num_classes, cfg.head = input_size, 3, 0, 64, n_classes, 1
        for i in range(4):
            cfg.layers[i] = 2
        cfg.precision, cfg.grad_precision = precision_cfg, grad_cfg
        self._create(lib.b2e_resnet_create, cfg, max_batch, device)

    def enable_grad(self, enable: bool = True):
        """Gradient mode: ``net(x)[0]`` becomes differentiable w.r.t. the image (native dgrad of the whole parser;
        batches <= max_batch).  Costs workspace: the backward pass has its own buffers."""
        self._enable_grad(enable)
        self.differentiable = bool(enable)
        return self

    _backward_fn = lib.b2e_resnet_backward

    def _out_shape(self, B):
        cfg = self.config
        return (B, cfg.n_classes, cfg.input_size, cfg.input_size)

    @staticmethod
    def fold_reference_state_dict(sd, eps=1e-5):
        """The reference's BiSeNet ``state_dict`` -> the engine's parameters (BatchNorm folded; the auxiliary heads
        conv_out16 / conv_out32 are training-time outputs and are dropped)."""
        out = {}
        for k, w in sd.items():
            if not k.endswith(".weight") or w.dim() != 4 or k.startswith(("conv_out16.", "conv_out32.")):
                continue
            name = k[:-len(".weight")]
            if name.startswith("cp.resnet."):
                if name.endswith("downsample.0"):
                    bn = name[:-1] + "1"
                else:
                    head, last = name.rsplit("conv", 1)
                    bn = f"{head}bn{last}"
                out[name + ".weight"], out[name + ".bias"] = _fold(w, sd, bn, eps)
            elif name.endswith(".conv") and (name + ".weight") in sd and (name[:-len(".conv")] + ".bn.weight") in sd:
                # ConvBNReLU: <block>.conv + <block>.bn -> <block>
                blk = name[:-len(".conv")]
                fw, fb = _fold(w, sd, blk + ".bn", eps)
                if blk == "cp.conv_avg":         # acts on the pooled vector: an fp32 matrix
                    fw = fw.reshape(fw.shape[0], -1)
                out[blk + ".weight"], out[blk + ".bias"] = fw, fb
            elif name.endswith(".conv_atten"):
                fw, fb = _fold(w, sd, name[:-len("conv_atten")] + "bn_atten", eps)
                out[name + ".weight"], out[name + ".bias"] = fw.reshape(fw.shape[0], -1), fb
            elif name in ("ffm.conv1", "ffm.conv2"):
                out[name + ".weight"] = w.float().reshape(w.shape[0], -1)
            elif name == "conv_out.conv_out":
                out[name + ".weight"], out[name + ".bias"] = w.float(), torch.zeros(w.shape[0])
        return out

    def load_reference_state_dict(self, sd, eps=1e-5):
        return self.load_state_dict(self.fold_reference_state_dict(sd, eps))

    def _check_input(self, image, keep=False):
        if not image.is_cuda:
            raise _C.B2EError("BiSeNet: image must be a CUDA tensor (no CPU fallback)")
        cfg = self.config
        if tuple(image.shape[1:]) != (3, cfg.input_size, cfg.input_size):
            raise ValueError(f"BiSeNet: expected (B,3,{cfg.input_size},{cfg.input_size}), got {tuple(image.shape)}")
        if keep and not self.differentiable:
            raise _C.B2EError("BiSeNet: call enable_grad() before differentiating through the native face parser")
        if keep and image.shape[0] > self.max_batch:
            raise ValueError(f"BiSeNet with gradient: batch {image.shape[0]} > max_batch {self.max_batch}")

    def forward_keep(self, image):
        """Logits (B, n_classes, S, S) - ``net(image)[0]`` - with the activations kept in the engine's workspace for
        ``input_grad`` (no autograd graph).  Needs gradient mode (``enable_grad()``) and B <= max_batch."""
        self._check_input(image, keep=True)
        return self._keep(image.detach().to(torch.float32).contiguous())

    def input_grad(self, d_logits):
        """d(loss)/d(image) of the last ``forward_keep`` given d(loss)/d(logits) (native dgrad of the whole parser)."""
        return self._keep_grad(d_logits)

    def __call__(self, image):
        grad = image.requires_grad and torch.is_grad_enabled()
        self._check_input(image, keep=grad)
        if grad:
            xx = image if (image.dtype == torch.float32 and image.is_contiguous()) else image.to(torch.float32).contiguous()
            return (self._keep_node(xx), None, None)
        return (self._forward_sliced(image.detach().to(torch.float32).contiguous()), None, None)

    def labels(self, image):
        """Parsing map (B, S, S) int64 = ``net(image)[0].argmax(1)``, bit for bit: the last kernel upsamples the logits
        and takes their argmax per pixel, so no (B, n_classes, S, S) logits are written.  Batches above max_batch run
        in slices.  The call overwrites the activations, so a gradient of an earlier kept forward is refused after it."""
        self._check_input(image)
        x = image.detach().to(torch.float32).contiguous()
        S = self.config.input_size
        out = torch.empty((x.shape[0], S, S), dtype=torch.int64, device=x.device)
        for b0 in range(0, x.shape[0], self.max_batch):
            xs, ls = x[b0:b0 + self.max_batch], out[b0:b0 + self.max_batch]
            self._launch(lib.b2e_resnet_forward_labels, _ptr(xs), _ptr(ls), xs.shape[0], _stream())
        return out

    def profile(self, image, timestep=None):
        """Per-op CUDA-event timings of one forward (``timestep`` is ignored: the face parser has none)."""
        x = image.detach().to(torch.float32).contiguous()
        return self._profile(x, None, torch.empty(self._out_shape(x.shape[0]), dtype=torch.float32, device=x.device))


class MultiResBiSeNet:
    """ONE face parser for every square input resolution - the reference's BiSeNet is fully convolutional, and its
    workflow shares one ``SegmentationModel`` between mask creation (512x512, src/models.py:113-118) and ``NetAttrFunc``
    (the decoded 256x256 image goes straight into ``segmentation_model.net``, src/attr_functions.py:213-215).  The
    engine plans its buffers per resolution, so this wrapper keeps one engine per input size (built on first use, same
    weights); differentiated calls get their own engine with the native input gradient enabled.

    ``precision``: None - forward-only engines (mask creation: an argmax) run f16 operands, the differentiated engines
    the fp32-accurate forward ("fp32"), so the guidance gradient has the fp32 network's ReLU / max-pool masks;
    "fp16" / "fp32" force one mode for both.  ``grad_precision`` applies to the differentiated engines only: None - their
    backward runs on 16-bit operands; "fp32" - fp32-accurate backward (needs their forward to be fp32-accurate, i.e.
    ``precision`` None or "fp32")."""

    def __init__(self, n_classes=19, max_batch=1, device="cuda", seed=0, precision=None, grad_precision=None):
        self.n_classes, self.max_batch, self.device, self.seed = n_classes, int(max_batch), device, seed
        if precision not in (None, "fp16", "fp32"):
            raise ValueError(f"MultiResBiSeNet: precision must be None, 'fp16' or 'fp32' (got {precision!r})")
        _C.resolve_grad_precision(grad_precision, precision or "fp32", "MultiResBiSeNet")
        self.precision, self.grad_precision = precision, grad_precision
        self._folded = None      # engine-format state dict (BatchNorm folded); None -> seeded random init
        self._engines = {}

    def load_reference_state_dict(self, sd, eps=1e-5):
        self._folded = BiSeNet.fold_reference_state_dict(sd, eps)
        for e in self._engines.values():
            e.load_state_dict(self._folded)
        return self

    def engine(self, size: int, grad: bool = False) -> BiSeNet:
        grad = bool(grad)
        e = self._engines.get((size, grad))
        if e is None:
            if size % 32 or size < 64:
                raise ValueError(f"BiSeNet: input resolution must be a multiple of 32 and >= 64 (got {size})")
            precision = self.precision or ("fp32" if grad else "fp16")
            e = BiSeNet(self.n_classes, size, max_batch=self.max_batch, device=self.device, precision=precision,
                        grad_precision=self.grad_precision if grad else None)
            if self._folded is not None:
                e.load_state_dict(self._folded)
            else:
                e.init_random(self.seed)
            if grad:
                e.enable_grad()
            self._engines[(size, grad)] = e
        return e

    @staticmethod
    def _check_shape(image):
        if image.dim() != 4 or image.shape[1] != 3 or image.shape[-1] != image.shape[-2]:
            raise ValueError(f"BiSeNet: expected (B,3,S,S), got {tuple(image.shape)}")

    def __call__(self, image):
        self._check_shape(image)
        return self.engine(int(image.shape[-1]), grad=image.requires_grad and torch.is_grad_enabled())(image)

    def labels(self, image):
        """Parsing map (B, S, S) int64 on the forward-only engine of the input's resolution (``BiSeNet.labels``)."""
        self._check_shape(image)
        return self.engine(int(image.shape[-1])).labels(image)

    def eval(self):
        return self

    def to(self, *a, **k):
        return self
