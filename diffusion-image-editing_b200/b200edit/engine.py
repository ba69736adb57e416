"""Base class of the native network wrappers: one ``b2e_unet`` handle of libb200edit.so (every network of the engine,
UNet, decoders, encoder, classifier, face parser, LPIPS and CLIP, is this handle type), the workspace bound to it, its
parameters, and the one rule of its single workspace: a backward pass runs only over the activations of the forward it
belongs to."""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _C
from ._C import check, lib

_OP_KINDS = {0: "conv_igemm", 1: "groupnorm", 2: "attention", 3: "other"}


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class _KeptForwardFn(torch.autograd.Function):
    """A kept forward as an autograd node: backward = the engine's native input gradient over this forward's activations,
    refused once another call has overwritten them."""

    @staticmethod
    def forward(ctx, x, model, *args):
        ctx.model, ctx.n_args = model, len(args)
        out = model._keep(x, *args)
        ctx.gen = model._keep_gen
        return out

    @staticmethod
    def backward(ctx, d_out):
        return (ctx.model._keep_grad(d_out, ctx.gen), None) + (None,) * ctx.n_args


class Engine:
    _h = None
    _fwd_gen = 0        # generation of the activations in the workspace (see _launch)
    _keep_gen = None    # generation of the last kept forward

    def _create(self, create, cfg, max_batch, device):
        """``create(&cfg, max_batch, &handle)`` (a ``b2e_*_create``), then allocate and bind the workspace."""
        self.device = torch.device(device)
        self.dtype = torch.float32
        self.max_batch = int(max_batch)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(create(C.byref(cfg), self.max_batch, C.byref(h)), create.__name__)
        self._h = h
        self._rebind_workspace()

    def _rebind_workspace(self):
        """Allocate the workspace the engine's current plan needs (256-byte aligned) and bind it."""
        with torch.cuda.device(self.device):
            nbytes = lib.b2e_unet_workspace_bytes(self._h)
            self._ws = None                 # free the old workspace before allocating the new one
            self._ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
            base = (self._ws.data_ptr() + 255) // 256 * 256
            self._launch(lib.b2e_unet_bind_workspace, C.c_void_p(base), nbytes)

    def _enable_grad(self, enable):
        """Gradient mode on / off: the plan changes, so the workspace is re-queried and re-bound."""
        with torch.cuda.device(self.device):
            check(lib.b2e_unet_enable_grad(self._h, int(enable)), "b2e_unet_enable_grad")
        self._rebind_workspace()

    def __del__(self):
        if self._h:
            lib.b2e_unet_destroy(self._h)
            self._h = None

    # ------------------------------------------------------------------ parameters
    def param_info(self):
        out = []
        name, numel, fan = C.c_char_p(), C.c_int64(), C.c_int64()
        for i in range(lib.b2e_unet_num_params(self._h)):
            check(lib.b2e_unet_param_info(self._h, i, C.byref(name), C.byref(numel), C.byref(fan)))
            out.append((name.value.decode(), numel.value, fan.value))
        return out

    def load_state_dict(self, sd, strict=True):
        """sd: mapping diffusers-name -> fp32 tensor (any device)."""
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        names = {n for n, _, _ in self.param_info()}
        missing = sorted(names - set(sd))
        unexpected = sorted(set(sd) - names)
        if strict and (missing or unexpected):
            raise KeyError(f"load_state_dict: missing {missing[:5]}..., unexpected {unexpected[:5]}...")
        with torch.cuda.device(self.device):
            for k in names & set(sd):
                t = sd[k].detach().to(self.device, torch.float32).contiguous()
                check(lib.b2e_unet_set_param(self._h, k.encode(), C.c_void_p(t.data_ptr()), t.numel(), stream),
                      f"set_param({k})")
            torch.cuda.current_stream().synchronize()   # temporaries above must outlive the copies
        return missing, unexpected

    def init_random(self, seed=0):
        """PyTorch-default-style init (U(-1/sqrt(fan_in), 1/sqrt(fan_in)); norm scale 1, shift 0)."""
        self.load_state_dict(self.random_state_dict(seed))
        return self

    def random_state_dict(self, seed=0):
        """The state dict ``init_random(seed)`` loads (so that a second engine can be given the same weights)."""
        g = torch.Generator().manual_seed(seed)
        sd = {}
        for name, numel, fan in self.param_info():
            if fan == 0:
                sd[name] = torch.ones(numel) if name.endswith(".weight") else torch.zeros(numel)
            elif fan < 0:   # codebook: U(-1/n, 1/n) with n = -fan (diffusers VectorQuantizer init)
                sd[name] = (torch.rand(numel, generator=g) * 2 - 1) / float(-fan)
            else:
                bound = 1.0 / math.sqrt(fan)
                sd[name] = (torch.rand(numel, generator=g) * 2 - 1) * bound
        return sd

    def to(self, *a, **k):
        return self

    def eval(self):
        return self

    @property
    def flops_per_sample(self) -> float:
        return float(lib.b2e_unet_flops(self._h, 1))

    @property
    def launches_per_forward(self) -> int:
        return int(lib.b2e_unet_launches_per_forward(self._h))

    # ------------------------------------------------------------------ forward
    def _launch(self, fn, *args):
        """``fn(handle, *args)``: every library call that overwrites the activations in the workspace (a forward, a
        profiled forward, LPIPS's reference pass, a workspace re-bind) goes through here and starts a new generation, so
        the input gradient of any earlier kept forward is refused instead of computed over the wrong activations."""
        self._fwd_gen += 1
        check(fn(self._h, *args), fn.__name__)

    def _out_shape(self, B):
        raise NotImplementedError

    def _forward(self, x):
        """One forward of a batch <= max_batch (no timesteps)."""
        out = torch.empty(self._out_shape(x.shape[0]), dtype=torch.float32, device=x.device)
        self._launch(lib.b2e_unet_forward, _ptr(x), None, _ptr(out), x.shape[0], _stream())
        return out

    def _forward_sliced(self, x):
        """The forward of any batch, in slices of max_batch."""
        outs = [self._forward(x[b0:b0 + self.max_batch]) for b0 in range(0, x.shape[0], self.max_batch)]
        return outs[0] if len(outs) == 1 else torch.cat(outs)

    def _profile(self, x, t, out):
        """Per-op CUDA-event timings of one forward: list of dicts(kind, ms, flops, bytes, desc)."""
        cap = 1024
        n = C.c_int()
        ms, fl, by, kd = (C.c_float * cap)(), (C.c_double * cap)(), (C.c_double * cap)(), (C.c_int * cap)()
        self._launch(lib.b2e_unet_profile, _ptr(x), _ptr(t), _ptr(out), x.shape[0], _stream(), cap, C.byref(n), ms, fl,
                     by, kd)
        return [dict(kind=_OP_KINDS[kd[i]], ms=ms[i], flops=fl[i], bytes=by[i],
                     desc=lib.b2e_unet_op_desc(self._h, i).decode()) for i in range(n.value)]

    # ------------------------------------------------------------------ kept forward / input gradient
    _backward_fn = None     # the b2e_*_backward of a differentiable network

    def _keep(self, x, *args):
        """``_forward`` whose activations the workspace keeps for ``_keep_grad`` (no autograd graph)."""
        out = self._forward(x, *args)
        self._keep_gen, self._keep_shape, self._keep_numel = self._fwd_gen, tuple(x.shape), out.numel()
        return out

    def _keep_grad(self, d_out, gen=None):
        """d(loss)/d(input) of the kept forward of generation ``gen`` (default: the last one) given d(loss)/d(output)."""
        if (self._keep_gen if gen is None else gen) != self._fwd_gen:
            raise _C.B2EError(f"{type(self).__name__}: the engine ran another forward since the one being differentiated "
                              "(its activations were overwritten); differentiate before the next call on the same network")
        g = d_out.detach().to(torch.float32).contiguous()
        if g.numel() != self._keep_numel:
            raise _C.B2EError(f"{type(self).__name__}: the output gradient has {g.numel()} elements, the output of the "
                              f"forward being differentiated {self._keep_numel}")
        dx = torch.empty(self._keep_shape, dtype=torch.float32, device=g.device)
        fn = self._backward_fn
        check(fn(self._h, _ptr(g), _ptr(dx), self._keep_shape[0], _stream()), fn.__name__)
        return dx

    def _keep_node(self, x, *args):
        """``_keep`` as an autograd node differentiable w.r.t. ``x``."""
        return _KeptForwardFn.apply(x, self, *args)
