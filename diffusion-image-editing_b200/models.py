"""Model factory (drop-in for src/models.py).

The reference downloads hub checkpoints; offline the factory builds the same architectures with
random-init weights (seeded) on the native sm_100a engine, and accepts a diffusers-layout
``state_dict`` so real checkpoints can be dropped in later."""
from types import SimpleNamespace
from typing import Optional

import torch

from b200edit import _C
from b200edit.scheduler import DDIMScheduler
from b200edit.unet import DDPM256_CONFIG, LDM_CELEBAHQ_CONFIG, UNet2DModel
from diffusion_classes import DDPM, LDM, SD  # noqa: F401
from utils import get_device


class NativePipeline(SimpleNamespace):
    """Duck-type of the diffusers pipeline object the path uses: .unet, .scheduler, .device."""

    def to(self, device):
        return self


def create_diffusion_model(name: str, sample_clipping: bool = True, *, max_batch: int = 8, seed: int = 0,
                           state_dict: Optional[dict] = None, unet_config: Optional[dict] = None, vqvae=None,
                           vq_config: Optional[dict] = None, vq_state_dict: Optional[dict] = None, guidance_module=None,
                           decoder_grad: bool = True, tokenizer=None, text_encoder=None, precision: Optional[str] = None,
                           with_encoder: bool = True, text_encoder_config: Optional[dict] = None,
                           text_encoder_state_dict: Optional[dict] = None, encoder_precision: Optional[str] = None):
    """``name``: "ddpm" (google/ddpm-celebahq-256 layout), "sd" (Stable Diffusion 1.x layout: native conditional UNet
    + native KL decoder with gradient; ``vqvae=`` substitutes the vae, ``tokenizer=`` / ``text_encoder=`` are the
    caller's CLIP modules) or "ldm" (CompVis/ldm-celebahq-256 layout: native UNet on
    the 64x64x3 latent + native VQ decoder (forward + latent gradient) and encoder; ``vqvae=`` substitutes the caller's VQ autoencoder module
    (encode().latents / decode().sample, as in the reference's pipeline object); ``guidance_module=`` is the
    differentiable decoder used when guidance runs through decode).  ``precision="fp32"`` selects the fp32-accurate
    (split-f16) noise predictor (all three families) and VQ / KL decoder (forward only: guidance through the decoder uses the fp16 engine).  ``with_encoder`` (default) also builds the native VQ / KL encoder behind
    ``LDM.encode`` / ``SD.encode``.  ``encoder_precision="fp32"`` selects the fp32-accurate native VQ / KL encoder and
    native CLIP text encoder (the inputs of a real-image or prompt-conditioned edit); it does not apply to a caller's
    ``vqvae=`` / ``text_encoder=`` and does not follow ``precision`` (``None``: the 16-bit type)."""
    if encoder_precision is not None:
        _C.resolve_precision(encoder_precision, "create_diffusion_model(encoder_precision)")   # refuse before building anything
    device = get_device()
    if name == "ddpm":
        unet = UNet2DModel(**(unet_config or DDPM256_CONFIG), max_batch=max_batch, device=device, precision=precision)
        if state_dict is not None:
            unet.load_state_dict(state_dict)
        else:
            unet.init_random(seed)
        scheduler = DDIMScheduler.from_preset("ddpm")
        scheduler.config.clip_sample = sample_clipping   # True for synthetic data, False for real images
        return DDPM(NativePipeline(unet=unet, scheduler=scheduler, device=device))
    if name == "ldm":
        from b200edit.vqmodel import LDM_VQ_CONFIG, VQModel
        unet = UNet2DModel(**(unet_config or LDM_CELEBAHQ_CONFIG), max_batch=max_batch, device=device, precision=precision)
        if state_dict is not None:
            unet.load_state_dict(state_dict)
        else:
            unet.init_random(seed)
        guidance_vqvae = None
        if vqvae is None:
            # native decoder: forward for the post-loop decoding of the sample / x0 history and, with
            # decoder_grad=True (default), the native dgrad for guidance THROUGH the decoder
            vqvae = VQModel(**(vq_config or LDM_VQ_CONFIG), max_batch=max_batch, device=device, with_encoder=with_encoder,
                            precision=precision, encoder_precision=encoder_precision)
            if vq_state_dict is not None:
                vqvae.load_state_dict(vq_state_dict)
            else:
                vqvae.init_random(seed + 1)
            # decoder weights for a gradient twin (random init: the decoder part of what init_random just loaded)
            vq_sd = vq_state_dict if vq_state_dict is not None else vqvae.random_state_dict(seed + 1)
            if decoder_grad and precision == "fp32":
                # the fp32-accurate (split-operand) decoder is forward-only: guidance THROUGH the decoder runs on a second,
                # f16-operand engine with the same weights (decoder gradient within 3e-3 relative RMS of fp32 autograd)
                guidance_vqvae = VQModel(**(vq_config or LDM_VQ_CONFIG), max_batch=max_batch, device=device, with_encoder=False,
                                         precision="fp16")
                guidance_vqvae.load_state_dict(vq_sd, strict=False)     # the encoder's entries are simply not used
                guidance_vqvae.enable_grad()
            elif decoder_grad:
                vqvae.enable_grad()
        elif isinstance(vqvae, torch.nn.Module) or not getattr(vqvae, "forward_only", False):
            guidance_vqvae = vqvae
        scheduler = DDIMScheduler.from_preset("ldm")
        scheduler.config.clip_sample = sample_clipping   # src/models.py:43 ("LDM was trained with this flag=False")
        return LDM(NativePipeline(unet=unet, scheduler=scheduler, vqvae=vqvae,
                                  guidance_vqvae=guidance_vqvae if guidance_module is None else guidance_module,
                                  device=device))
    if name == "sd":
        from b200edit.unet_cond import SD15_CONFIG, UNet2DConditionModel
        from b200edit.vqmodel import SD_VAE_CONFIG, AutoencoderKL
        # CFG doubles the latent batch: the UNet engine is sized for 2 * max_batch samples
        unet = UNet2DConditionModel(**(unet_config or SD15_CONFIG), max_batch=2 * max_batch, device=device, precision=precision)
        if state_dict is not None:
            unet.load_state_dict(state_dict)
        else:
            unet.init_random(seed)
        if vqvae is None:
            vae = AutoencoderKL(**(vq_config or SD_VAE_CONFIG), max_batch=max_batch, device=device, with_encoder=with_encoder,
                                precision=precision, encoder_precision=encoder_precision)
            if vq_state_dict is not None:
                vae.load_state_dict(vq_state_dict)
            else:
                vae.init_random(seed + 1)
            vq_sd = vq_state_dict if vq_state_dict is not None else vae.random_state_dict(seed + 1)
            guidance_vae = None
            if decoder_grad and precision == "fp32":      # see the "ldm" branch: f16-operand gradient twin
                guidance_vae = AutoencoderKL(**(vq_config or SD_VAE_CONFIG), max_batch=max_batch, device=device, with_encoder=False,
                                             precision="fp16")
                guidance_vae.load_state_dict(vq_sd, strict=False)
                guidance_vae.enable_grad()
            elif decoder_grad:
                vae.enable_grad()
        else:
            vae, guidance_vae = vqvae, None
        scheduler = DDIMScheduler.from_preset("sd")
        scheduler.config.clip_sample = sample_clipping
        # text side: the CLIP text encoder runs on the engine (b200edit.clip; transformers state_dict names) unless the
        # caller supplies a module; the tokenizer (BPE vocabulary files, unavailable offline) is always the caller's.
        # Prompts need both, precomputed text embeddings (2, 77, 768) need neither.
        if text_encoder is None:
            from b200edit.clip import SD15_CLIP_CONFIG, CLIPTextModel
            text_encoder = CLIPTextModel(**(text_encoder_config or SD15_CLIP_CONFIG), max_batch=2, device=device,
                                         precision=encoder_precision)
            if text_encoder_state_dict is not None:
                text_encoder.load_state_dict(text_encoder_state_dict)
            else:
                text_encoder.init_random(seed + 2)
        return SD(NativePipeline(unet=unet, scheduler=scheduler, vae=vae, guidance_vae=guidance_vae, tokenizer=tokenizer,
                                 text_encoder=text_encoder,
                                 device=device))
    raise ValueError(f"Unknown model name: {name}")


def get_pretrained_anyGAN(input_size: int = 256, max_batch: int = 1, state_dict_path: str = "../attribute_predictor.pt",
                          seed: int = 0, precision: Optional[str] = "fp32"):
    """The attribute predictor of ClassifierAttrFunc (src/models.py:69-77: ``models.resnet50()`` with an 80-way ``fc``
    loaded from ../attribute_predictor.pt) on the native engine: forward AND input gradient on the tcgen05 kernels, so
    classifier guidance needs no torch network.  ``input_size`` is the resolution of the decoded images it will see (256
    for DDPM / LDM, 512 for SD).  Offline (no checkpoint file) the weights are random-init (seeded).  ``precision``:
    "fp32" (default) runs the fp32-accurate forward, so the guidance gradient is routed through the fp32 network's
    ReLU / max-pool masks (input gradient within 1e-2 relative RMS of fp32 autograd); "fp16" is the f16-operand forward
    (3x fewer forward flops, gradient 0.15 relative RMS from fp32)."""
    import os
    from b200edit.resnet import resnet50_predictor
    sd = None
    if state_dict_path and os.path.exists(state_dict_path):
        sd = torch.load(state_dict_path, map_location="cpu")
        sd = sd.get("state_dict", sd)
    return resnet50_predictor(80, input_size, max_batch=max_batch, state_dict=sd, seed=seed, precision=precision)


def get_lpips(input_size: int = 256, max_batch: int = 1, state_dict: Optional[dict] = None, seed: int = 0,
              precision: Optional[str] = "fp32"):
    """The LPIPS (vgg) distance of ``use_lpips`` guidance and ``metrics.lpips`` (the reference's ``lpips.LPIPS(net='vgg')``)
    on the native engine: forward and input gradient on the tcgen05 kernels.  ``state_dict``: the full
    ``lpips.LPIPS(net='vgg').state_dict()``; without it the weights are seeded random (no pretrained VGG offline).
    ``precision`` "fp32" (default) runs the fp32-accurate forward because guidance differentiates the network (the
    ReLU / max-pool masks of the input gradient then agree with an fp32 evaluation); "fp16" is the 16-bit forward."""
    from b200edit.lpips import LPIPS
    net = LPIPS("vgg", input_size=input_size, max_batch=max_batch, device=get_device(), precision=precision)
    if state_dict is not None:
        net.load_state_dict(state_dict)
    else:
        net.init_random(seed)
    return net


class SegmentationModel:
    """Face parser front-end (src/models.py:80-118), same leading positional arguments as the reference:
    ``SegmentationModel(ckpt, n_classes, image_size)``.  The network is the native BiSeNet (b200edit.bisenet) for ANY
    square input resolution - mask creation feeds it 512x512, ``NetAttrFunc`` the decoded 256x256 image, both through
    this one object as in the reference - loaded from ``ckpt`` (the reference's Segmentation/res/cp/79999_iter.pth, a blob
    missing from the checkout) when the file exists, else seeded random-init weights.  ``net=`` (keyword-only)
    substitutes any callable mapping a (1,3,S,S) image to ([1,19,S,S] logits, ...).  ``max_batch`` (keyword-only) is the
    largest batch the default parser differentiates at once (``NetAttrFunc(per_sample=True)`` on a batch of images)."""

    def __init__(self, ckpt: str = "Segmentation/res/cp/79999_iter.pth", n_classes: int = 19, image_size: tuple = (512, 512),
                 *, net=None, seed: int = 0, precision: Optional[str] = None, max_batch: int = 1) -> None:
        self.device = get_device()
        if not (ckpt is None or isinstance(ckpt, (str, bytes)) or hasattr(ckpt, "__fspath__")):
            raise TypeError("SegmentationModel: the first argument is the checkpoint path (as in the reference); pass a "
                            "network with net=...")
        if net is None:
            import os
            from b200edit.bisenet import MultiResBiSeNet
            net = MultiResBiSeNet(n_classes, max_batch=max_batch, device=self.device, seed=seed, precision=precision)
            if ckpt and os.path.exists(ckpt):
                net.load_reference_state_dict(torch.load(ckpt, map_location="cpu"))
        self.net = net
        self.image_size = image_size
        self.mean = torch.tensor((0.485, 0.456, 0.406)).view(1, 3, 1, 1)
        self.std = torch.tensor((0.229, 0.224, 0.225)).view(1, 3, 1, 1)

    def process(self, image: torch.Tensor) -> torch.Tensor:
        x = torch.nn.functional.interpolate(image, size=self.image_size, mode="bilinear", antialias=True)
        return ((x - self.mean.to(x.device)) / self.std.to(x.device)).to(self.device)

    def __call__(self, image: torch.Tensor) -> torch.Tensor:
        """(1,3,H,W) -> (S,S) parsing map, as the reference.  (B,3,H,W) with B > 1 -> (B,S,S) int64: on the native parser
        the labels come from its fused upsample-and-argmax kernel, on a caller's ``net=`` from ``argmax(1)``."""
        x = self.process(image)
        if x.shape[0] > 1:
            from b200edit.bisenet import BiSeNet, MultiResBiSeNet
            if isinstance(self.net, (BiSeNet, MultiResBiSeNet)):
                return self.net.labels(x)
            return self.net(x)[0].argmax(1)
        out = self.net(x)[0]
        return out.squeeze(0).argmax(0)
