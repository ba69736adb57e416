"""Native decode path of ``diffusers.VQModel`` (the ``vqvae`` of CompVis/ldm-celebahq-256): the call contract the
reference uses is ``vqvae.decode(latent).sample`` (src/diffusion_classes.py:62-70).  Nearest-code quantisation,
post_quant_conv and the decoder run in libb200edit.so (bf16 tcgen05 implicit-GEMM convolutions, fp32 accumulation).

``decode`` is forward-only by default (post-loop decoding of the final sample and of the x0-prediction history);
``enable_grad()`` makes it an autograd node backed by the native decoder dgrad, which is what guidance THROUGH the
decoder (AttrFunc.apply with no_grad=False) uses.  ``with_encoder=True`` adds the native encoder + quant_conv
(``vqvae.encode(img).latents`` / ``vae.encode(img).latent_dist.mode()``, src/diffusion_classes.py:27-30, 55-60).
``precision`` selects the decoder's operands, ``encoder_precision`` the encoder's (``"fp32"``: the fp32-accurate split
forward; ``None``: the build's 16-bit type - it does not follow ``precision``).  A ``precision="fp32"`` decoder in gradient
mode also differentiates at the fp32 bar: split gradients through split dgrad weights, fp32 GroupNorm / upsample /
attention backward kernels; its forward is the same as in forward-only mode."""
from __future__ import annotations

from types import SimpleNamespace

import torch

from . import _C
from ._C import VQDecConfig, VQEncConfig, lib
from .engine import Engine

LDM_VQ_CONFIG = dict(latent_channels=3, out_channels=3, block_out_channels=(128, 256, 512), layers_per_block=2,
                     norm_num_groups=32, norm_eps=1e-6, num_vq_embeddings=8192, sample_size=64)


class _EncoderEngine(Engine):
    """diffusers ``Encoder`` + ``quant_conv`` on the engine (b2e_vqenc_create): image (B, C, S, S) -> (B, Q, s, s)."""

    def __init__(self, image_size, in_channels, latent_channels, block_out_channels, layers_per_block, norm_num_groups,
                 norm_eps, double_z, max_batch, device, precision=None):
        self.precision, precision_cfg = _C.resolve_precision(precision, "encoder")
        n = len(block_out_channels)
        self.image_size, self.q = image_size, latent_channels * (2 if double_z else 1)
        self.out_size = image_size >> (n - 1)
        self.config = SimpleNamespace(in_channels=in_channels, sample_size=image_size, out_channels=self.q)
        cfg = VQEncConfig()
        cfg.sample_size, cfg.in_channels, cfg.latent_channels, cfg.n_blocks = image_size, in_channels, latent_channels, n
        for i in range(n):
            cfg.block_out_channels[i] = block_out_channels[i]
        cfg.layers_per_block, cfg.norm_num_groups, cfg.norm_eps = layers_per_block, norm_num_groups, norm_eps
        cfg.double_z = int(double_z)
        cfg.precision = precision_cfg      # 1: fp32-accurate encode (split-f16 operands); quant_conv is fp32 either way
        self._create(lib.b2e_vqenc_create, cfg, max_batch, device)

    def _out_shape(self, B):
        return (B, self.q, self.out_size, self.out_size)

    def __call__(self, image):
        if not image.is_cuda:
            raise _C.B2EError("encode: image must be a CUDA tensor (no CPU fallback)")
        x = image.detach().to(torch.float32).contiguous()
        if tuple(x.shape[1:]) != (self.config.in_channels, self.image_size, self.image_size):
            raise ValueError(f"encode: expected (B,{self.config.in_channels},{self.image_size},{self.image_size}), "
                             f"got {tuple(x.shape)}")
        return self._forward_sliced(x)


class DiagonalGaussianDistribution:
    """``vae.encode(x).latent_dist``: moments = [mean | logvar] from the native encoder; the reference only takes
    ``mode()`` (src/diffusion_classes.py:29)."""

    def __init__(self, moments: torch.Tensor):
        self.mean, logvar = torch.chunk(moments, 2, dim=1)
        self.logvar = torch.clamp(logvar, -30.0, 20.0)
        self.std = torch.exp(0.5 * self.logvar)

    def mode(self) -> torch.Tensor:
        return self.mean

    def sample(self, generator=None) -> torch.Tensor:
        noise = torch.randn(self.mean.shape, generator=generator).to(self.mean.device)   # host RNG stream, as utils.py
        return self.mean + self.std * noise


def _is_encoder_key(k: str) -> bool:
    return k.startswith("encoder.") or k.startswith("quant_conv.")


class VQModel(Engine):

    forward_only = True   # until enable_grad(): no autograd graph through decode (see LDM.decode)

    def __init__(self, latent_channels=3, out_channels=3, block_out_channels=(128, 256, 512), layers_per_block=2,
                 norm_num_groups=32, norm_eps=1e-6, num_vq_embeddings=8192, sample_size=64, max_batch=8,
                 device="cuda", with_encoder=False, precision=None, encoder_precision=None):
        _C.require_device()
        self.precision, self._precision_cfg = _C.resolve_precision(precision, type(self).__name__)
        # the encoder's own precision (None: the 16-bit type, whatever the decoder's), checked with or without an encoder
        self.encoder_precision = _C.resolve_precision(encoder_precision, f"{type(self).__name__} encoder")[0]
        n = len(block_out_channels)
        self._enc = None
        self.config = SimpleNamespace(latent_channels=latent_channels, out_channels=out_channels,
                                      block_out_channels=tuple(block_out_channels), layers_per_block=layers_per_block,
                                      norm_num_groups=norm_num_groups, norm_eps=norm_eps,
                                      num_vq_embeddings=num_vq_embeddings, sample_size=sample_size,
                                      in_channels=latent_channels)
        self.out_size = sample_size << (n - 1)
        cfg = VQDecConfig()
        cfg.sample_size, cfg.latent_channels, cfg.out_channels, cfg.n_blocks = sample_size, latent_channels, out_channels, n
        for i in range(n):
            cfg.block_out_channels[i] = block_out_channels[i]
        cfg.layers_per_block, cfg.norm_num_groups, cfg.norm_eps = layers_per_block, norm_num_groups, norm_eps
        cfg.num_vq_embeddings = num_vq_embeddings
        cfg.precision = self._precision_cfg      # 1: fp32-accurate decode and, in gradient mode, latent gradient (split-f16)
        self._create(lib.b2e_vqdec_create, cfg, max_batch, device)
        if with_encoder:
            self._enc = _EncoderEngine(self.out_size, out_channels, latent_channels, block_out_channels, layers_per_block,
                                       norm_num_groups, norm_eps, num_vq_embeddings == 0, max_batch, device,
                                       precision=encoder_precision)

    # ---- parameters: "encoder.*" / "quant_conv.*" belong to the encoder engine (ignored when there is none)
    def load_state_dict(self, sd, strict=True):
        dec = {k: v for k, v in sd.items() if not _is_encoder_key(k)}
        enc = {k: v for k, v in sd.items() if _is_encoder_key(k)}
        missing, unexpected = super().load_state_dict(dec, strict)
        if self._enc is not None and enc:     # a decoder-only dictionary leaves the encoder untouched
            m2, u2 = self._enc.load_state_dict(enc, strict)
            missing, unexpected = missing + m2, unexpected + u2
        return missing, unexpected

    def init_random(self, seed=0):
        super().init_random(seed)
        if self._enc is not None:
            self._enc.init_random(seed + 7)
        return self

    def enable_grad(self, enable: bool = True):
        """Gradient mode: decode() becomes differentiable w.r.t. the latent (native dgrad; batches <= max_batch).
        Costs workspace: every activation of a forward pass is kept until the backward pass.  With
        ``precision="fp32"`` the gradient is fp32-accurate too (split operands and gradients, fp32 element-wise and
        attention backward), and the decoded image is the one of forward-only mode bit for bit."""
        self._enable_grad(enable)
        self.forward_only = not enable
        return self

    _backward_fn = lib.b2e_vqdec_backward

    def _out_shape(self, B):
        return (B, self.config.out_channels, self.out_size, self.out_size)

    # ---- decode + latent gradient WITHOUT an autograd graph (analytic guidance: the caller supplies d(loss)/d(image))
    def _check_latent(self, latent, keep):
        cfg = self.config
        if latent.dim() != 4 or tuple(latent.shape[1:]) != (cfg.latent_channels, cfg.sample_size, cfg.sample_size):
            raise ValueError(f"VQModel.decode: expected (B,{cfg.latent_channels},{cfg.sample_size},{cfg.sample_size}), "
                             f"got {tuple(latent.shape)}")
        if keep and latent.shape[0] > self.max_batch:
            raise ValueError(f"VQModel.decode with gradient: batch {latent.shape[0]} > max_batch {self.max_batch}")

    def decode_keep(self, latent: torch.Tensor) -> torch.Tensor:
        """decode(latent).sample with the activations kept in the engine's workspace for ``latent_grad``."""
        if self.forward_only:
            raise _C.B2EError(f"{type(self).__name__}.decode_keep: call enable_grad() first")
        self._check_latent(latent, keep=True)
        return self._keep(latent.detach().to(torch.float32).contiguous())

    def latent_grad(self, d_image: torch.Tensor) -> torch.Tensor:
        """d(loss)/d(latent) for the last ``decode_keep`` given d(loss)/d(image) (native dgrad of the whole decoder)."""
        return self._keep_grad(d_image)

    def decode(self, latent: torch.Tensor, force_not_quantize: bool = False):
        if force_not_quantize:
            raise NotImplementedError("VQModel.decode(force_not_quantize=True) is not on the native engine")
        if not latent.is_cuda:
            raise _C.B2EError("VQModel.decode: latent must be a CUDA tensor (no CPU fallback)")
        grad = not self.forward_only and latent.requires_grad and torch.is_grad_enabled()
        self._check_latent(latent, keep=grad)
        if grad:
            zz = latent if (latent.dtype == torch.float32 and latent.is_contiguous()) else latent.to(torch.float32).contiguous()
            return SimpleNamespace(sample=self._keep_node(zz))
        # histories can be longer than max_batch
        return SimpleNamespace(sample=self._forward_sliced(latent.detach().to(torch.float32).contiguous()))

    def _encode_raw(self, x):
        if self._enc is None:
            raise NotImplementedError(f"{type(self).__name__}.encode: build the model with with_encoder=True")
        return self._enc(x)

    def encode(self, x):
        """``vqvae.encode(img).latents`` (pre-quantisation latents; the quantiser runs inside decode)."""
        return SimpleNamespace(latents=self._encode_raw(x))

    def __call__(self, *a, **k):
        raise TypeError("VQModel: call .decode(latent)")

    def profile(self, latent):
        z = latent.to(torch.float32).contiguous()
        return self._profile(z, None, torch.empty(self._out_shape(z.shape[0]), dtype=torch.float32, device=z.device))


# CompVis/stable-diffusion-v1-x `vae` decode path: 64x64x4 latent -> 512x512x3 image (x8), no quantiser
SD_VAE_CONFIG = dict(latent_channels=4, out_channels=3, block_out_channels=(128, 256, 512, 512), layers_per_block=2,
                     norm_num_groups=32, norm_eps=1e-6, sample_size=64)


class AutoencoderKL(VQModel):
    """Native decode path of ``diffusers.AutoencoderKL`` (``vae.decode(latent / 0.18215).sample``,
    src/diffusion_classes.py:93-99): post_quant_conv -> decoder, same engine as the VQ decoder without the quantiser.
    State-dict names as in diffusers (``post_quant_conv.*``, ``decoder.*``)."""

    def __init__(self, latent_channels=4, out_channels=3, block_out_channels=(128, 256, 512, 512), layers_per_block=2,
                 norm_num_groups=32, norm_eps=1e-6, sample_size=64, max_batch=8, device="cuda", with_encoder=False,
                 precision=None, encoder_precision=None):
        super().__init__(latent_channels=latent_channels, out_channels=out_channels, block_out_channels=block_out_channels,
                         layers_per_block=layers_per_block, norm_num_groups=norm_num_groups, norm_eps=norm_eps,
                         num_vq_embeddings=0, sample_size=sample_size, max_batch=max_batch, device=device,
                         with_encoder=with_encoder, precision=precision, encoder_precision=encoder_precision)

    def encode(self, x):
        """``vae.encode(img).latent_dist`` (the reference takes ``.mode()``, src/diffusion_classes.py:29)."""
        return SimpleNamespace(latent_dist=DiagonalGaussianDistribution(self._encode_raw(x)))
