"""Native ``UNet2DConditionModel`` (Stable Diffusion 1.x layout): the call contract of the reference's CFG branch,
``unet(cat([latent] * 2), t, encoder_hidden_states=text_emb)["sample"]`` (src/diffusion_utils.py:61-70), executed by
libb200edit.so.  ResNet blocks and down/up-sampling are the UNet2DModel ones; attention blocks are Transformer2DModel
(GroupNorm, 1x1 proj_in, LayerNorm + 8-head self-attention, LayerNorm + cross-attention over <= 128 text tokens,
LayerNorm + GEGLU feed-forward, 1x1 proj_out), all linear layers and attention products on the tcgen05 GEMM kernel."""
from __future__ import annotations

from types import SimpleNamespace

import torch

from . import _C
from ._C import UNetConfig, lib
from .engine import _ptr, _stream
from .unet import UNet2DModel, UNetOutput

SD15_CONFIG = dict(sample_size=64, in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280),
                   layers_per_block=2, cross_attention_dim=768, attention_head_dim=8, norm_num_groups=32, norm_eps=1e-5)


class UNet2DConditionModel(UNet2DModel):
    def __init__(self, sample_size=64, in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280),
                 layers_per_block=2, cross_attention_dim=768, attention_head_dim=8, norm_num_groups=32, norm_eps=1e-5,
                 down_block_types=None, up_block_types=None, max_batch=2, device="cuda", precision=None):
        _C.require_device()
        self.precision, self._precision_cfg = _C.resolve_precision(precision, "UNet2DConditionModel")
        n = len(block_out_channels)
        down_block_types = tuple(down_block_types or ("CrossAttnDownBlock2D",) * (n - 1) + ("DownBlock2D",))
        up_block_types = tuple(up_block_types or ("UpBlock2D",) + ("CrossAttnUpBlock2D",) * (n - 1))
        self.config = SimpleNamespace(
            sample_size=sample_size, in_channels=in_channels, out_channels=out_channels,
            block_out_channels=tuple(block_out_channels), layers_per_block=layers_per_block,
            cross_attention_dim=cross_attention_dim, attention_head_dim=attention_head_dim,
            norm_num_groups=norm_num_groups, norm_eps=norm_eps, down_block_types=down_block_types,
            up_block_types=up_block_types)
        self.in_channels, self.sample_size = in_channels, sample_size
        cfg = UNetConfig()
        cfg.sample_size, cfg.in_channels, cfg.out_channels, cfg.n_blocks = sample_size, in_channels, out_channels, n
        for i in range(n):
            cfg.block_out_channels[i] = block_out_channels[i]
            cfg.down_attn[i] = int("Attn" in down_block_types[i])
            cfg.up_attn[i] = int("Attn" in up_block_types[i])
        cfg.layers_per_block, cfg.norm_num_groups, cfg.norm_eps = layers_per_block, norm_num_groups, norm_eps
        cfg.attention_head_dim = 0
        cfg.flip_sin_to_cos, cfg.freq_shift, cfg.downsample_padding = 1, 0.0, 1
        cfg.cross_attention_dim, cfg.num_attention_heads = cross_attention_dim, attention_head_dim   # SD 1.x: 8 heads
        cfg.precision = self._precision_cfg   # 1: fp32-accurate mode (split-f16 operands, fp32 attention)
        self._create(lib.b2e_unet_create, cfg, max_batch, device)
        self._t_cache = {}

    def __call__(self, sample, timestep, encoder_hidden_states=None, out=None, **_):
        if encoder_hidden_states is None:
            raise ValueError("UNet2DConditionModel: encoder_hidden_states is required")
        if not sample.is_cuda:
            raise _C.B2EError("UNet2DConditionModel: sample must be a CUDA tensor (no CPU fallback)")
        x = sample.to(torch.float32).contiguous()
        B = x.shape[0]
        cfg = self.config
        if tuple(x.shape[1:]) != (cfg.in_channels, cfg.sample_size, cfg.sample_size):
            raise ValueError(f"UNet2DConditionModel: expected (B,{cfg.in_channels},{cfg.sample_size},{cfg.sample_size}), "
                             f"got {tuple(x.shape)}")
        ctx = encoder_hidden_states.to(x.device, torch.float32)
        if ctx.dim() != 3 or ctx.shape[2] != cfg.cross_attention_dim or ctx.shape[1] > 128:
            raise ValueError(f"encoder_hidden_states must be (B, L <= 128, {cfg.cross_attention_dim}), got {tuple(ctx.shape)}")
        if ctx.shape[0] != B:
            # the reference's CFG call doubles ONE latent and passes (2, L, D) = [first, second]; for a batch of latents
            # cat([latent] * 2) is [all firsts, all seconds], so every context row serves B / n consecutive samples
            if B % ctx.shape[0] != 0:
                raise ValueError(f"encoder_hidden_states batch {ctx.shape[0]} does not divide the sample batch {B}")
            ctx = ctx.repeat_interleave(B // ctx.shape[0], dim=0)
        ctx = ctx.contiguous()
        t = self._timesteps(timestep, B)
        eps = out if out is not None else torch.empty_like(x[:, :cfg.out_channels]) if cfg.out_channels == cfg.in_channels \
            else torch.empty((B, cfg.out_channels, cfg.sample_size, cfg.sample_size), dtype=torch.float32, device=x.device)
        self._launch(lib.b2e_unet_forward_cond, _ptr(x), _ptr(t), _ptr(ctx), ctx.shape[1], _ptr(eps), B, _stream())
        return UNetOutput(sample=eps)
