"""Segmentation-guided diffusion editing pipeline (drop-in for src/SegDiffEditPipeline.py).

The guided loop of ``edit_image`` runs one UNet forward (tcgen05 kernels) plus ONE fused CUDA kernel
per step (x0 prediction + clip + DDIM/DDPM update + sigma*z + analytic colour guidance) whenever the
strategy is a built-in colour loss on a pixel-space model; other strategies fall back to the
scheduler-step kernel followed by ``AttrFunc.apply``.  Per-step scalars are host-side and cached, so
the loop never synchronises with the device; images are converted to PIL once, after the loop."""
from dataclasses import dataclass
from typing import List, Optional

import torch
from PIL import Image

from attr_functions import AttrFunc
from b200edit import ops
from b200edit.outputs import BaseOutput
from constants import ATTRS
from ddim_inversion import ddim_inversion
from ddpm_inversion import check_batch, invert, reverse_step  # noqa: F401  (reverse_step re-exported like the reference)
from diffusion_classes import DDPM, LDM, SD
from diffusion_utils import diffusion_loop, get_noise_pred, get_variance_noise
from mask_creator import MaskCreator
from transforms import batch_to_pils, tensor_to_pil
from utils import apply_mask, generate_random_samples, get_device, process_lists_of_tensors


@dataclass
class EditorOutput(BaseOutput):
    imgs: Image.Image
    pred_original_samples: Optional[List[Image.Image]] = None
    model_outputs: Optional[List[torch.Tensor]] = None


class SegDiffEditPipeline:
    """Edits an image with a diffusion model, optionally restricted by a face-parsing mask:
    real images are inverted (DDIM or edit-friendly DDPM), noise maps can be resynthesised inside
    the mask, and an attribute function can steer every denoising step."""

    def __init__(self, diffusion_wrapper, segmentation_model=None):
        self.diffusion_wrapper = diffusion_wrapper
        self.segmentation_model = segmentation_model
        self.device = getattr(diffusion_wrapper, "device", None) or get_device()

    # ------------------------------------------------------------------ validation
    def check_classes(self, classes):
        for c in classes or ():
            assert 0 <= c < len(ATTRS)

    def check_inputs(self, attr_func, eta, mask, resynthesize, zs):
        if eta > 0 and zs is None:
            raise ValueError("eta > 0 and zs is empty")
        if zs is not None and eta == 0:
            raise ValueError("eta == 0 and zs is not empty")
        if attr_func is None and (mask is None or resynthesize is None):
            raise ValueError("attr_func is None and classes and mask is None implies no edit")

    def check_batch_shapes(self, xt, zs, xts, mask):
        """Batched edits (extension): 5-D xts (T+1,B,C,H,W) go with 5-D zs (T,B,C,H,W); a mask's batch is 1 or B."""
        if xts is not None and xts.dim() == 5:
            if zs is None or zs.dim() != 5 or tuple(zs.shape[1:]) != tuple(xts.shape[1:]):
                raise ValueError(f"xts of shape {tuple(xts.shape)} (T+1, B, C, H, W) needs zs of shape (T, B, C, H, W), got "
                                 f"{None if zs is None else tuple(zs.shape)}")
            B = xts.shape[1]
        else:
            B = xt.shape[0] if xt is not None and xt.dim() == 4 else 1
        if mask is not None and mask.dim() == 4 and mask.shape[0] not in (1, B):
            raise ValueError(f"the mask batch must be 1 or the image batch {B}, got a mask of shape {tuple(mask.shape)}")

    # ------------------------------------------------------------------ preparation
    def create_mask(self, classes, dilate_mask, segmentation, dim):
        return MaskCreator(dilate_mask=dilate_mask, resize_size=(dim, dim)).create_mask(segmentation, classes=classes)

    def prepare_for_edit(self, img: torch.Tensor, classes: Optional[List[int]] = None, dilate_mask: bool = False):
        """Returns (latent, mask, segmentation).  Call before edit_image.  A batch of B > 1 images gives (B, ...) latents,
        (B, S, S) parsing maps and (B, C, d, d) masks."""
        self.check_classes(classes)
        segmentation = mask = None
        if classes is not None:
            if self.segmentation_model is None:
                raise ValueError("classes given but the pipeline has no segmentation model")
            segmentation = self.segmentation_model(img)
            mask = self.create_mask(classes, dilate_mask, segmentation, self.diffusion_wrapper.data_dimensionality)
        return self.diffusion_wrapper.encode(img), mask, segmentation

    def edit_noise_map(self, noise_map: torch.Tensor, mask: torch.Tensor):
        """Fresh noise of the map's own shape ((B,C,H,W) or (T',B,C,H,W)) inside the mask."""
        n = noise_map.shape[:-3].numel()
        fresh = generate_random_samples(n, self.diffusion_wrapper.model.unet).to(noise_map.device)
        return apply_mask(mask, noise_map, fresh.reshape(noise_map.shape))

    def edit_noise_maps(self, xt, zs, mask, resynthesize):
        if mask is not None and resynthesize:
            xt = self.edit_noise_map(xt, mask)
            if zs is not None:
                zs = self.edit_noise_map(zs, mask)
        return xt, zs

    def prepare_text_emb(self, prompt):
        if prompt is None:
            return None
        return self.diffusion_wrapper.additional_prep(self.diffusion_wrapper.model, prompt)

    def postprocess(self, xt, pred_original_samples):
        decoded = self.diffusion_wrapper.decode(xt)
        img = tensor_to_pil(decoded) if decoded.shape[0] == 1 else batch_to_pils(decoded)
        return img, process_lists_of_tensors(self.diffusion_wrapper, pred_original_samples)

    def prepare_real_image_edit(self, img: torch.Tensor, eta: float = 0, inversion_method: str = "ddim",
                                classes: Optional[List[int]] = None, dilate_mask: bool = False,
                                prompt: Optional[str] = None, cfg_scale: Optional[float] = None,
                                prog_bar: bool = True):
        """Invert a real image: returns (xt, zs, xts, mask, segmentation).  A batch of B > 1 images is inverted in one
        pass (``ddpm_inversion.invert``): xt (B, ...), zs (T, B, ...), xts (T+1, B, ...)."""
        if inversion_method == "ddim" and eta > 0:
            raise ValueError("eta > 0 and inversion_method == 'ddim' is not possible")
        w = self.diffusion_wrapper
        if inversion_method == "ddpm" and img.dim() == 4:
            check_batch(w.model, img.shape[0], prompt is not None)     # before any network runs
        latent, mask, segmentation = self.prepare_for_edit(img, classes, dilate_mask)
        if type(w) in (DDPM, LDM):
            assert w.model.scheduler.config.clip_sample is False
        if inversion_method == "ddim":
            xt = ddim_inversion(model=w.model, x0=latent, prompt=prompt, cfg_scale=cfg_scale)
            zs = xts = None
        elif inversion_method == "ddpm":
            xt, zs, xts = invert(model=w.model, x0=latent, num_inference_steps=w.scheduler.num_inference_steps,
                                 eta=eta, prompt=prompt, cfg_scale=cfg_scale, prog_bar=prog_bar)
        else:
            raise ValueError(f"Unknown inversion method: {inversion_method}")
        if type(w) == SD and mask is not None:
            # one extra all-ones channel for the 4th latent channel (the reference hard-codes 32x32)
            ones = torch.ones((mask.shape[0], 1) + tuple(mask.shape[-2:]), device=xt.device)
            mask = torch.cat((mask, ones), dim=1)
        return xt, zs, xts, mask, segmentation

    # ------------------------------------------------------------------ the guided loop
    def edit_image(self, xt: torch.Tensor, eta: float = 0, model_outputs: Optional[List[torch.Tensor]] = None,
                   zs: Optional[torch.Tensor] = None, xts: Optional[torch.Tensor] = None,
                   mask: Optional[torch.Tensor] = None, attr_func: Optional[AttrFunc] = None,
                   prompt: Optional[str] = None, cfg_scale: Optional[float] = None, inversion_method: str = "ddim",
                   Tskip: Optional[int] = None, resynthesize: bool = False, *, prog_bar: bool = True,
                   output_type: str = "pil", x0_history_out: Optional[torch.Tensor] = None) -> EditorOutput:
        """Runs the (guided) reverse process from ``xt`` (or from ``xts[Tskip]`` with ``zs[Tskip:]``).

        output_type="pil" (reference behaviour): PIL image(s), PIL x0-prediction history, eps list.
        output_type="tensor" (extension): the final sample tensor and the x0 history as tensors.
        x0_history_out (extension, with output_type="tensor"): a pinned host tensor (steps, B, C, H, W); every step's x0
        prediction is copied into it on a side stream while the next step computes (the device->host traffic of the
        history - 6.6 MB per step at batch 8 - leaves the critical path); the returned history are its slices.  The call
        blocks the host until the last of those copies has landed (the final decode has to be consumed anyway), so the
        slices are safe to read as soon as it returns."""
        self.check_inputs(attr_func=attr_func, eta=eta, mask=mask, resynthesize=resynthesize, zs=zs)
        self.check_batch_shapes(xt, zs, xts, mask)
        xt, zs = self.edit_noise_maps(xt, zs, mask, resynthesize)
        text_emb = self.prepare_text_emb(prompt)
        w = self.diffusion_wrapper
        sch = w.model.scheduler
        eps_hist, x0_hist = [], []
        if xts is not None:
            xt = xts[Tskip] if xts.dim() == 5 else xts[Tskip].unsqueeze(0)
            zs = zs[Tskip:]
        mode = "ddpm" if (inversion_method == "ddpm" and Tskip is not None) else "ddim"
        clip = bool(sch.config.clip_sample) if mode == "ddim" else False
        akw = None
        if attr_func is not None:
            attr_func.kwargs["mask"] = mask if (attr_func.kwargs.get("use_mask", False) and mask is not None) else None
            akw = attr_func.kwargs
        copy_stream = None
        if x0_history_out is not None:
            if output_type != "tensor" or x0_history_out.is_cuda:
                raise ValueError("x0_history_out needs output_type='tensor' and a host tensor")
            n_steps = zs.shape[0] if zs is not None else len(sch.timesteps)
            want = (xt.shape[0],) + tuple(xt.shape[1:])
            if (x0_history_out.dtype != torch.float32 or x0_history_out.dim() != 5 or x0_history_out.shape[0] < n_steps
                    or tuple(x0_history_out.shape[1:]) != want):
                raise ValueError(f"x0_history_out must be a float32 host tensor of shape (>= {n_steps}, {', '.join(map(str, want))}); "
                                 f"got {tuple(x0_history_out.shape)} {x0_history_out.dtype}")
            copy_stream = getattr(self, "_copy_stream", None)
            if copy_stream is None:
                copy_stream = self._copy_stream = torch.cuda.Stream(device=xt.device)
        for step_idx, timestep in diffusion_loop(w.model, zs, prog_bar=prog_bar):
            t = int(timestep)
            eps = get_noise_pred(w.model, xt, timestep, text_emb, cfg_scale)
            z = get_variance_noise(zs, step_idx, eta)
            c = sch.coeffs(t, eta, mode)
            fk = None
            guided = attr_func is not None and attr_func.in_window(step_idx)
            if guided:
                fk = attr_func.fused_kwargs(xt, w, **akw)
            if fk is not None and fk.pop("l2reg", False):
                xt, x0_pred = ops.guided_step_l2reg(xt, eps, c, clip=clip, clip_range=sch.config.clip_sample_range,
                                                    noise=z, **fk)
            elif fk is not None:
                xt, x0_pred = ops.guided_step(xt, eps, c, clip=clip, clip_range=sch.config.clip_sample_range,
                                              noise=z, **fk)
            else:
                # scheduler / reverse step (the reference leaves x0 unbound on its ddpm branch; it is
                # produced by the same kernel here), then the generic autograd guidance if any
                xt, x0_pred = ops.guided_step(xt, eps, c, clip=clip, clip_range=sch.config.clip_sample_range, noise=z)
                if guided:
                    xt, _ = attr_func.apply(xt=xt, zt=z, model_output=eps, timestep=timestep, step_idx=step_idx,
                                            model=w, **akw)
            eps_hist.append(eps)
            if copy_stream is not None:
                # stream the x0 prediction to the host behind the next step's UNet forward
                done = torch.cuda.Event()
                done.record()
                copy_stream.wait_event(done)
                with torch.cuda.stream(copy_stream):
                    x0_history_out[len(x0_hist)].copy_(x0_pred, non_blocking=True)
                x0_pred.record_stream(copy_stream)
                x0_hist.append(x0_history_out[len(x0_hist)])
            else:
                x0_hist.append(x0_pred)
        if copy_stream is not None:
            torch.cuda.current_stream().wait_stream(copy_stream)   # device order: the history precedes later work of the caller
            copy_stream.synchronize()                              # host order: the returned slices hold their final contents
        if output_type == "tensor":
            return EditorOutput(w.decode(xt), x0_hist, eps_hist)
        img, x0_imgs = self.postprocess(xt, x0_hist)
        return EditorOutput(img, x0_imgs, eps_hist)
