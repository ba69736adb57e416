"""Native UNet2DModel: same call contract as ``diffusers.UNet2DModel`` on the reference's path
(``unet(sample, timestep)["sample"]``, ``unet.config.in_channels/sample_size`` and the deprecated
direct attributes - src/diffusion_utils.py:72, src/utils.py:68-70, src/ddpm_inversion.py:39-41),
executed by libb200edit.so: bf16 tcgen05 implicit-GEMM convolutions, fp32 accumulation."""
from __future__ import annotations

from types import SimpleNamespace
from typing import Dict, Optional

import torch

from . import _C
from ._C import UNetConfig, lib
from .engine import Engine, _ptr, _stream

DDPM256_CONFIG = dict(
    sample_size=256, in_channels=3, out_channels=3,
    block_out_channels=(128, 128, 256, 256, 512, 512), layers_per_block=2,
    down_block_types=("DownBlock2D",) * 4 + ("AttnDownBlock2D", "DownBlock2D"),
    up_block_types=("UpBlock2D", "AttnUpBlock2D") + ("UpBlock2D",) * 4,
    norm_num_groups=32, norm_eps=1e-6, attention_head_dim=None,
    flip_sin_to_cos=False, freq_shift=1, downsample_padding=0,
)

# CompVis/ldm-celebahq-256 `unet` (UNet2DModel on the 64x64x3 VQ latent, ~274 M parameters)
LDM_CELEBAHQ_CONFIG = dict(
    sample_size=64, in_channels=3, out_channels=3,
    block_out_channels=(224, 448, 672, 896), layers_per_block=2,
    down_block_types=("DownBlock2D", "AttnDownBlock2D", "AttnDownBlock2D", "AttnDownBlock2D"),
    up_block_types=("AttnUpBlock2D", "AttnUpBlock2D", "AttnUpBlock2D", "UpBlock2D"),
    norm_num_groups=32, norm_eps=1e-6, attention_head_dim=32,
    flip_sin_to_cos=True, freq_shift=0, downsample_padding=1,
)


class UNetOutput(dict):
    @property
    def sample(self):
        return self["sample"]


class UNet2DModel(Engine):
    def __init__(self, sample_size=256, in_channels=3, out_channels=3,
                 block_out_channels=(128, 128, 256, 256, 512, 512), layers_per_block=2,
                 down_block_types=None, up_block_types=None, norm_num_groups=32, norm_eps=1e-6,
                 attention_head_dim=None, flip_sin_to_cos=False, freq_shift=1, downsample_padding=0,
                 max_batch=8, device="cuda", precision=None):
        """precision: None / "fp16" (default: fp16 operands, fp32 accumulation) or "fp32" (fp32-accurate mode: split-f16
        operands hi + lo on the same tcgen05 kernels, three products per GEMM; meets the 1e-4 bar of the fp32
        reference at about a third of the fp16 throughput)."""
        _C.require_device()
        self.precision, self._precision_cfg = _C.resolve_precision(precision, "UNet2DModel")
        n = len(block_out_channels)
        down_block_types = tuple(down_block_types or ("DownBlock2D",) * n)
        up_block_types = tuple(up_block_types or ("UpBlock2D",) * n)
        self.config = SimpleNamespace(
            sample_size=sample_size, in_channels=in_channels, out_channels=out_channels,
            block_out_channels=tuple(block_out_channels), layers_per_block=layers_per_block,
            down_block_types=down_block_types, up_block_types=up_block_types,
            norm_num_groups=norm_num_groups, norm_eps=norm_eps, attention_head_dim=attention_head_dim,
            flip_sin_to_cos=flip_sin_to_cos, freq_shift=freq_shift, downsample_padding=downsample_padding)
        self.in_channels, self.sample_size = in_channels, sample_size   # deprecated aliases
        cfg = UNetConfig()
        cfg.sample_size, cfg.in_channels, cfg.out_channels, cfg.n_blocks = sample_size, in_channels, out_channels, n
        for i in range(n):
            cfg.block_out_channels[i] = block_out_channels[i]
            cfg.down_attn[i] = int(down_block_types[i].startswith("Attn"))
            cfg.up_attn[i] = int(up_block_types[i].startswith("Attn"))
        cfg.layers_per_block, cfg.norm_num_groups, cfg.norm_eps = layers_per_block, norm_num_groups, norm_eps
        cfg.attention_head_dim = int(attention_head_dim or 0)
        cfg.flip_sin_to_cos, cfg.freq_shift = int(flip_sin_to_cos), float(freq_shift)
        cfg.downsample_padding = int(downsample_padding)
        cfg.precision = self._precision_cfg
        self._create(lib.b2e_unet_create, cfg, max_batch, device)
        self._t_cache: Dict[tuple, torch.Tensor] = {}

    def _out_shape(self, B):
        cfg = self.config
        return (B, cfg.out_channels, cfg.sample_size, cfg.sample_size)

    def profile(self, sample, timestep):
        """Per-op CUDA-event timings of one forward: list of dicts(kind, ms, flops, bytes)."""
        x = sample.to(torch.float32).contiguous()
        B = x.shape[0]
        eps = torch.empty(self._out_shape(B), dtype=torch.float32, device=x.device)
        return self._profile(x, self._timesteps(timestep, B), eps)

    # ------------------------------------------------------------------ forward
    def _timesteps(self, timestep, B):
        if torch.is_tensor(timestep) and timestep.is_cuda:
            t = timestep.to(torch.int64)
            return (t.reshape(1).expand(B) if t.numel() == 1 else t.reshape(B)).contiguous()
        if torch.is_tensor(timestep) and timestep.numel() > 1:
            return timestep.to(self.device, torch.int64).contiguous()
        key = (int(timestep), B)
        if key not in self._t_cache:
            self._t_cache[key] = torch.full((B,), int(timestep), dtype=torch.int64, device=self.device)
        return self._t_cache[key]

    def __call__(self, sample, timestep, out: Optional[torch.Tensor] = None, **_):
        if not sample.is_cuda:
            raise _C.B2EError("UNet2DModel: sample must be a CUDA tensor (no CPU fallback)")
        x = sample.to(torch.float32).contiguous()
        B = x.shape[0]
        cfg = self.config
        if tuple(x.shape[1:]) != (cfg.in_channels, cfg.sample_size, cfg.sample_size):
            raise ValueError(f"UNet2DModel: expected (B,{cfg.in_channels},{cfg.sample_size},{cfg.sample_size}), "
                             f"got {tuple(x.shape)}")
        t = self._timesteps(timestep, B)
        eps = out if out is not None else torch.empty(self._out_shape(B), dtype=torch.float32, device=x.device)
        if self._graph_on and B == self.max_batch and not torch.cuda.is_current_stream_capturing():
            return UNetOutput(sample=self._replay(x, t, eps))
        if self._graph_on and self._graphs:
            self._graphs.clear()      # an eager forward at another batch re-plans the workspace: captured launches are stale
        self._launch(lib.b2e_unet_forward, _ptr(x), _ptr(t), _ptr(eps), B, _stream())
        return UNetOutput(sample=eps)

    # ------------------------------------------------------------------ CUDA-graph replay (launch-bound regime)
    _graph_on = False

    def enable_cuda_graph(self, enable: bool = True):
        """Replay the forward's ~225 launches as ONE captured CUDA graph for calls at batch == max_batch (the launch-bound
        regime: at batch 1 the forward is 225 kernels of ~10 us).  The plan has fixed buffers, no allocation and no host
        synchronisation, so it captures as is (programmatic-dependent-launch edges included); inputs / timesteps / output go
        through static buffers.  Captured on first use; any eager call at another batch size re-plans the workspace and
        drops the capture."""
        self._graph_on = bool(enable)
        self._graphs = {}
        return self

    def _replay(self, x, t, eps):
        B = x.shape[0]
        g = self._graphs.get(B)
        if g is None:
            sx, st, se = torch.empty_like(x), torch.empty_like(t), torch.empty_like(eps)
            sx.copy_(x); st.copy_(t)
            # warm-up outside capture (plan rebuild for this batch, lazy function attributes), then capture
            self._launch(lib.b2e_unet_forward, _ptr(sx), _ptr(st), _ptr(se), B, _stream())
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                self._launch(lib.b2e_unet_forward, _ptr(sx), _ptr(st), _ptr(se), B, _stream())
            g = self._graphs[B] = (graph, sx, st, se)
        graph, sx, st, se = g
        sx.copy_(x)
        st.copy_(t)
        graph.replay()
        eps.copy_(se)
        return eps
