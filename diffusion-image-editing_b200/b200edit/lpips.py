"""Native LPIPS distance (lpips v0.1, ``lpips.LPIPS(net='vgg')``) on libb200edit.so, differentiable w.r.t. its first
input - the regulariser of the masked-prediction guidance (``AttrFunc(..., use_lpips=True)``: ``loss(mask * x0') +
lambda_ * LPIPS(1 - mask * x0', x_0)``) and the ``metrics.lpips`` distance.

The VGG-16 trunk runs on the tcgen05 implicit-GEMM kernel with ReLU in the epilogue (conv1_1 as a 1x1 GEMM over an
im2col tensor that the input packer forms from the scaled input), the distance head and the max pools on their own
kernels, the input gradient on the dgrad twins of the same convolutions.  The second input is constant for a whole edit:
its normalised features are computed once and cached in the engine (re-run only when that tensor changes)."""
from __future__ import annotations

import ctypes as C
from types import SimpleNamespace

import torch

from . import _C
from ._C import LpipsConfig, check, lib
from .unet import UNet2DModel

# (slice, index in vgg16().features, in channels, out channels) of the thirteen convolutions
VGG16_CONVS = ((1, 0, 3, 64), (1, 2, 64, 64), (2, 5, 64, 128), (2, 7, 128, 128), (3, 10, 128, 256), (3, 12, 256, 256),
               (3, 14, 256, 256), (4, 17, 256, 512), (4, 19, 512, 512), (4, 21, 512, 512), (5, 24, 512, 512),
               (5, 26, 512, 512), (5, 28, 512, 512))
LIN_CHANNELS = (64, 128, 256, 512, 512)
SCALING_SHIFT = (-.030, -.088, -.188)
SCALING_SCALE = (.458, .448, .450)


class _LPIPSFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, in0, model, mask):
        ctx.model, ctx.shape = model, tuple(in0.shape)
        out = model._forward(in0, mask)
        ctx.gen = model._fwd_gen      # the activations of THIS forward live in the engine's single workspace
        return out

    @staticmethod
    def backward(ctx, d_out):
        m = ctx.model
        if m._fwd_gen != ctx.gen:
            raise _C.B2EError("LPIPS backward: the engine ran another forward since this graph was built (its activations "
                              "were overwritten); differentiate before the next call on the same network")
        return m._backward(d_out.reshape(ctx.shape[0])), None, None


class LPIPS(UNet2DModel):
    """``d = LPIPS(...)(in0, in1)``: (B, 1, 1, 1), like ``lpips.LPIPS.forward``; in0 (B, 3, S, S) and in1 (1 | B, 3, S, S)
    fp32 CUDA tensors in [-1, 1].  Autograd node in ``in0`` only.  Shares parameter loading / profiling with the UNet
    wrapper (same engine handle type); parameters under ``lpips.LPIPS().state_dict()`` names."""

    def __init__(self, net="vgg", input_size=256, max_batch=1, device="cuda", precision="fp32"):
        """precision: "fp32" (default) - fp32-accurate FORWARD (split 16-bit operands, three tensor-core products per
        GEMM), so that the ReLU / max-pool masks of the input gradient agree with an fp32 evaluation; None / "fp16" - 16-bit
        operands throughout.  The backward pass runs on 16-bit operands either way."""
        if net != "vgg":
            raise ValueError(f"LPIPS: only net='vgg' is implemented (got {net!r})")
        _C.require_device()
        self.precision, precision_cfg = _C.resolve_precision(precision, "LPIPS")
        self.config = SimpleNamespace(net=net, input_size=input_size, sample_size=input_size, in_channels=3, out_channels=1)
        self.device = torch.device(device)
        self.dtype = torch.float32
        self.max_batch = int(max_batch)
        cfg = LpipsConfig()
        cfg.input_size, cfg.precision = input_size, precision_cfg
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(lib.b2e_lpips_create(C.byref(cfg), self.max_batch, C.byref(h)), "lpips_create")
            self._h = h
            nbytes = lib.b2e_unet_workspace_bytes(h)
            self._ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
            base = (self._ws.data_ptr() + 255) // 256 * 256
            check(lib.b2e_unet_bind_workspace(h, C.c_void_p(base), nbytes), "unet_bind_workspace")
        self._t_cache = {}
        self._ref = None            # the reference tensor whose features the engine holds (kept alive: identity check)
        self._mask = None           # the mask the engine reads in the backward of the last forward (kept alive)

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
    _fwd_gen = 0   # bumped by every forward: a backward over a stale workspace is detected (see _LPIPSFn)

    def enable_grad(self, enable: bool = True):
        with torch.cuda.device(self.device):
            check(lib.b2e_unet_enable_grad(self._h, int(enable)), "unet_enable_grad")
            nbytes = lib.b2e_unet_workspace_bytes(self._h)
            self._ws = None
            self._ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
            base = (self._ws.data_ptr() + 255) // 256 * 256
            check(lib.b2e_unet_bind_workspace(self._h, C.c_void_p(base), nbytes), "unet_bind_workspace")
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
        self._fwd_gen += 1
        check(lib.b2e_lpips_set_reference(self._h, C.c_void_p(x.data_ptr()), x.shape[0],
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream)), "lpips_set_reference")
        self._ref = (in1, in1._version)

    def _forward(self, x, mask=None):
        self._fwd_gen += 1
        self._mask = mask           # the backward's -mask chain reads this memory: it lives until the next forward
        B = x.shape[0]
        dist = torch.empty((B, 1, 1, 1), dtype=torch.float32, device=x.device)
        mp, mb = (None, 0) if mask is None else (C.c_void_p(mask.data_ptr()), mask.shape[0])
        check(lib.b2e_lpips_forward(self._h, C.c_void_p(x.data_ptr()), mp, mb, C.c_void_p(dist.data_ptr()), B,
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream)), "lpips_forward")
        return dist

    def _backward(self, d_dist):
        g = d_dist.to(torch.float32).contiguous()
        B = g.shape[0]
        S = self.config.input_size
        dx = torch.empty((B, 3, S, S), dtype=torch.float32, device=g.device)
        check(lib.b2e_lpips_backward(self._h, C.c_void_p(g.data_ptr()), C.c_void_p(dx.data_ptr()), B,
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream)), "lpips_backward")
        return dx

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
            return _LPIPSFn.apply(x, self, mask)
        return self._forward(x.detach(), mask)

    forward = __call__

    def input_grad(self, d_dist):
        """d(sum_b d_dist[b] * dist[b]) / d(in0) of the last forward (through its mask transform), without autograd."""
        return self._backward(d_dist.reshape(-1))

    def profile(self, in0):
        x = self._check(in0, "in0", lambda b: 1 <= b <= self.max_batch).detach()
        B = x.shape[0]
        out = torch.empty((B,), dtype=torch.float32, device=x.device)
        self._fwd_gen += 1          # profiling forwards overwrite the activations (and run without a mask)
        self._mask = None
        cap = 1024
        n = C.c_int()
        ms, fl, by, kd = (C.c_float * cap)(), (C.c_double * cap)(), (C.c_double * cap)(), (C.c_int * cap)()
        check(lib.b2e_unet_profile(self._h, C.c_void_p(x.data_ptr()), None, C.c_void_p(out.data_ptr()), B,
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream), cap, C.byref(n), ms, fl, by, kd),
              "lpips_profile")
        names = {0: "conv_igemm", 1: "groupnorm", 2: "attention", 3: "other"}
        return [dict(kind=names[kd[i]], ms=ms[i], flops=fl[i], bytes=by[i],
                     desc=lib.b2e_unet_op_desc(self._h, i).decode()) for i in range(n.value)]


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
