"""Native CLIP text encoder: the call contract the reference uses is ``model.text_encoder(input_ids)[0]``
(``encode_text`` / ``prep_text``, src/diffusion_utils.py:34-52) = ``transformers.CLIPTextModel(...).last_hidden_state``.
Token + position embedding, pre-LayerNorm transformer layers (causal multi-head self-attention on the fused tcgen05
attention kernel, quick-GELU MLP, every linear layer on the implicit-GEMM kernel), final LayerNorm - in libb200edit.so.
Parameters load from a transformers ``state_dict`` unchanged.  The tokenizer (BPE files) stays the caller's.

``precision="fp32"`` builds the fp32-accurate forward (split hi + lo 16-bit operands, three products per GEMM; the
embedding sum, LayerNorm, quick-GELU and the causal attention in fp32 on the CUDA cores), the text conditioning an
fp32-accurate noise predictor wants; ``None`` (default) is the build's 16-bit type."""
from __future__ import annotations

from types import SimpleNamespace

import torch

from . import _C
from ._C import ClipConfig, lib
from .engine import Engine, _ptr, _stream

# openai/clip-vit-large-patch14 text tower (the text encoder of Stable Diffusion 1.x)
SD15_CLIP_CONFIG = dict(vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12,
                        num_attention_heads=12, max_position_embeddings=77)


class TextEncoderOutput(tuple):
    @property
    def last_hidden_state(self):
        return self[0]


class CLIPTextModel(Engine):
    def __init__(self, vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12,
                 num_attention_heads=12, max_position_embeddings=77, max_batch=2, device="cuda", precision=None):
        _C.require_device()
        self.precision, precision_cfg = _C.resolve_precision(precision, type(self).__name__)
        self.config = SimpleNamespace(vocab_size=vocab_size, hidden_size=hidden_size, intermediate_size=intermediate_size,
                                      num_hidden_layers=num_hidden_layers, num_attention_heads=num_attention_heads,
                                      max_position_embeddings=max_position_embeddings, in_channels=1, sample_size=8,
                                      out_channels=1)
        cfg = ClipConfig()
        cfg.vocab_size, cfg.hidden_size, cfg.intermediate_size = vocab_size, hidden_size, intermediate_size
        cfg.num_layers, cfg.num_heads, cfg.max_positions = num_hidden_layers, num_attention_heads, max_position_embeddings
        cfg.precision = precision_cfg
        self._create(lib.b2e_clip_create, cfg, max_batch, device)

    def load_state_dict(self, sd, strict=True):
        sd = {k: v for k, v in sd.items() if not k.endswith("position_ids")}   # a buffer of older transformers versions
        return super().load_state_dict(sd, strict)

    def _forward(self, ids):
        ids = ids.contiguous()
        o = torch.empty((ids.shape[0], ids.shape[1], self.config.hidden_size), dtype=torch.float32, device=self.device)
        self._launch(lib.b2e_clip_forward, _ptr(ids), ids.shape[1], _ptr(o), ids.shape[0], _stream())
        return o

    def __call__(self, input_ids, **_):
        ids = input_ids.to(self.device, torch.int64).contiguous()
        if ids.dim() != 2 or ids.shape[1] > self.config.max_position_embeddings:
            raise ValueError(f"CLIPTextModel: input_ids must be (B, L <= {self.config.max_position_embeddings}), got {tuple(ids.shape)}")
        return TextEncoderOutput((self._forward_sliced(ids),))

    forward = __call__
