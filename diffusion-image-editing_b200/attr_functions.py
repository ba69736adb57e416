"""Guidance ("attribute function") strategies (drop-in for src/attr_functions.py).

``AttrFunc.apply`` nudges the post-step sample down the gradient of a loss evaluated on the
predicted clean image:  x <- x + (-d(loss_scale*loss)/dx) * alphas_cumprod[t]**2.

* Built-in colour strategies with an identity decoder (pixel-space DDPM) use the ANALYTIC gradient
  inside one fused CUDA kernel - no autograd graph, no reduction (the loss value is never needed
  for the update); masked-gradient and masked + L2-regularised variants included.
* The same colour strategies on a latent model (LDM / SD) whose decoder runs on the engine: the loss gradient w.r.t. the
  DECODED image is closed-form too, so the nudge is x0' kernel -> native decoder forward -> analytic d(loss)/d(image) kernel ->
  native decoder backward -> update kernel, again without autograd (``_apply_native_decoder``).
* Any other strategy (user subclasses, network losses) evaluates ``loss`` with torch autograd on the device - exactly the
  reference's procedure - and the resulting gradient is applied by a CUDA kernel.  That is the extension contract of the
  reference: subclass, implement ``loss``, register.
* The network strategies (``NetAttrFunc`` / ``ClassifierAttrFunc``) with ``per_sample=True`` on a native parser / predictor
  (and an identity or native decoder) run kernel to kernel as well: x0' kernel -> (decoder forward) -> network forward ->
  batched loss head (value and gradient of every image) -> network input gradient -> (decoder backward) -> update kernel
  (``_apply_native_network``).
* ``mask_pred_original_sample=True, use_lpips=True`` needs the distance network as ``lpips_model=`` (``models.get_lpips``,
  the native LPIPS-vgg, or any callable ``(in0, in1) -> (B, 1, 1, 1)``): the loss is ``loss(mask * x0') +
  lambda_ * LPIPS(1 - mask * x0', x_0)``, differentiated by autograd through the native LPIPS node.  Without
  ``lpips_model`` ``use_lpips`` raises, as it must without VGG weights.
"""
from abc import ABC, abstractmethod

import torch

from b200edit import ops
from b200edit._C import B2EError


def l2_norm(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """sqrt(sum((x - y)^2)).  Differentiable (torch) when a gradient is required, else one reduction kernel."""
    if x.requires_grad or y.requires_grad or not x.is_cuda:
        return torch.sqrt(torch.sum((x - y) ** 2))
    return ops.l2_distance(x, y)


def apply_lpips(xt, x0, loss_fn_vgg):
    return loss_fn_vgg(xt, x0)


def single_color_loss(images: torch.Tensor, idx: int, target: float) -> torch.Tensor:
    """mean |images[:, idx] - target| over batch and pixels."""
    if images.requires_grad or not images.is_cuda:
        return torch.abs(images[:, idx, :, :] - target).mean()
    t = [None] * images.shape[1]
    t[idx] = target
    return ops.channel_l1(images, t)[idx]


def color_loss(images: torch.Tensor, r_target: float, g_target: float, b_target: float) -> torch.Tensor:
    """Target-weighted sum of the per-channel mean absolute errors (the weights ARE the targets)."""
    if images.requires_grad or not images.is_cuda:
        return (single_color_loss(images, 0, r_target) * r_target + single_color_loss(images, 1, g_target) * g_target
                + single_color_loss(images, 2, b_target) * b_target)
    e = ops.channel_l1(images, [r_target, g_target, b_target])
    return e[0] * r_target + e[1] * g_target + e[2] * b_target


def _identity_decoder(model) -> bool:
    return bool(getattr(model, "decode_is_identity", False))


def _native_decoder(model, B):
    """The decoder of a nudge of B samples without autograd, as (decoder, chain): (None, 1.0) for an identity decoder;
    a latent model's native decoder in gradient mode and chain = d(decoder input) / d(x0 prediction); None when the
    model's decoder is not native or B exceeds its max_batch."""
    if _identity_decoder(model):
        return None, 1.0
    nd = getattr(model, "native_decoder", None)
    nd = nd() if callable(nd) else None
    if nd is None or B > nd[0].max_batch:
        return None
    return nd


def _decode_x0(xt, model_output, coeffs, dec, chain):
    """x0' = (x - sqrt(1-a) eps) / sqrt(a), then the wrapper's decode scaling (SD: 1 / 0.18215 * latent) as its own rounding
    step - the reference's op order, so the decoder sees bit-identical input on both paths - and the decoder forward,
    kept for the backward of ``_guide``."""
    lat = ops.pred_x0(xt, model_output, coeffs.sqrt_a_t, coeffs.sqrt_b_t)
    if dec is None:
        return lat
    if chain != 1.0:
        lat = ops.axpby(lat, lat, chain, 0.0)
    return dec.decode_keep(lat)


def _guide(xt, d_img, dec, chain, coeffs, gmask):
    """The nudged sample from d(loss)/d(image) of ``_decode_x0``'s image: decoder backward, then the update kernel."""
    d_lat = d_img if dec is None else dec.latent_grad(d_img)
    return ops.apply_latent_guidance(xt, d_lat, chain, coeffs.sqrt_a_t, coeffs.a_t_sq, mask=gmask)


class AttrFunc(ABC):
    """Base class of the guidance strategies.  kwargs understood by ``apply`` (also stored at
    construction and splatted back by the pipeline): use_mask, mask, mask_attr_grad,
    mask_pred_original_sample, use_l2, use_lpips, lambda_, x_0.  ``per_sample=True`` (extension) makes every image of
    a batch its own problem: the colour losses average per image instead of over the whole batch, the network losses
    are sum_b L_b with L_b the reference's loss on image b alone (the reference's heads read batch element 0 only)."""

    def __init__(self, loss_scale: float = 1, t1: int = 0, t2: int = 50, nudge_xt=True, nudge_zt=False,
                 per_sample: bool = False, **kwargs) -> None:
        lpips_model = kwargs.pop("lpips_model", None)
        self.kwargs = kwargs
        self.loss_scale = loss_scale
        self.t1, self.t2 = t1, t2
        self.nudge_xt, self.nudge_zt = nudge_xt, nudge_zt
        self.per_sample = per_sample
        if kwargs.get("use_lpips", False):
            if lpips_model is None:
                raise NotImplementedError("LPIPS regularisation needs the lpips package and VGG weights, "
                                          "neither of which is available offline; pass lpips_model= "
                                          "(models.get_lpips) or use use_l2=True")
            self.metric = lpips_model
        elif kwargs.get("use_l2", False):
            self.metric = l2_norm

    @property
    def name(self) -> str:
        return self.__class__.__name__

    @abstractmethod
    def loss(self, pred_original_sample: torch.Tensor, **kwargs) -> torch.Tensor:
        raise NotImplementedError

    # ---- fused-kernel description of the loss; None -> generic autograd path
    def colour_spec(self):
        return None

    # ---- native network strategies (per_sample): the engine that evaluates the loss network on (B, 3, size, size)
    # images with forward_keep / input_grad, or None; and the batched head: d(loss_scale * sum_b L_b) / d(logits)
    def native_network(self, size: int):
        return None

    def native_head_grad(self, logits):
        raise NotImplementedError

    # ---- generic (autograd) pieces, same structure as the reference
    def calculate_loss(self, pred_original_sample: torch.Tensor, **kwargs) -> torch.Tensor:
        if kwargs.get("mask_pred_original_sample", False):
            lambda_, mask, x_0 = kwargs.get("lambda_"), kwargs.get("mask"), kwargs.get("x_0")
            if kwargs.get("use_lpips", False):
                return self.loss(mask * pred_original_sample) + lambda_ * apply_lpips(
                    1 - mask * pred_original_sample, x_0, self._lpips_model())
            if kwargs.get("use_l2", False):
                return self.loss(mask * pred_original_sample) + lambda_ * l2_norm(
                    1 - mask * pred_original_sample, x_0)
            raise ValueError("No metric specified")
        return self.loss(pred_original_sample, **kwargs)

    def _has_lpips(self) -> bool:
        m = getattr(self, "metric", None)
        return m is not None and m is not l2_norm

    def _lpips_model(self):
        if not self._has_lpips():
            raise NotImplementedError("LPIPS is unavailable offline without lpips_model= (models.get_lpips)")
        return self.metric

    def edit_attr_grad(self, attr_grad, **kwargs):
        if kwargs.get("mask_attr_grad", False):
            if kwargs.get("mask", False) is None:
                raise ValueError("No mask specified")
            attr_grad = kwargs.get("mask") * attr_grad
        return attr_grad

    def get_attr_grad(self, xt, pred_original_sample, loss_scale, **kwargs):
        attr_loss = self.calculate_loss(pred_original_sample, **kwargs) * loss_scale
        if self.per_sample and self.colour_spec() is not None:
            # the colour losses average over the batch as well; per_sample (extension) makes every image its own problem:
            # the sum of the per-image means = batch size x the batch mean
            attr_loss = attr_loss * pred_original_sample.shape[0]
        attr_grad = -torch.autograd.grad(attr_loss, xt)[0]
        return self.edit_attr_grad(attr_grad, **kwargs)

    def _apply_autograd(self, xt, zt, model_output, coeffs, model, **kwargs):
        with torch.enable_grad():
            x = xt.detach().requires_grad_(True)
            pred = (x - coeffs.sqrt_b_t * model_output) / coeffs.sqrt_a_t
            pred = model.decode(pred, no_grad=False)
            g = self.get_attr_grad(x, pred, self.loss_scale, **kwargs)
        g = g.detach().contiguous()
        if self.nudge_zt and zt is not None:
            zt = ops.apply_guidance_grad(zt.detach(), g.expand_as(zt) if g.shape != zt.shape else g, coeffs.a_t_sq)
        if self.nudge_xt:
            xt = ops.apply_guidance_grad(xt.detach(), g, coeffs.a_t_sq)
        return xt, zt

    def fused_kwargs(self, xt, model, **kwargs):
        """Arguments for ops.guided_step describing this strategy, or None if it cannot be fused."""
        spec = self.colour_spec()
        if spec is None or not _identity_decoder(model) or self.nudge_zt or not self.nudge_xt:
            return None
        if xt.shape[1] > 4 or xt.shape[1] < len(spec[0]):
            return None
        targets, weights = spec
        mask = kwargs.get("mask")
        if kwargs.get("mask_attr_grad", False) and mask is None:
            raise ValueError("No mask specified")
        fk = dict(targets=targets, weights=weights, loss_scale=self.loss_scale,
                  mask=mask if (kwargs.get("mask_attr_grad", False) or kwargs.get("mask_pred_original_sample", False)) else None,
                  mask_grad=bool(kwargs.get("mask_attr_grad", False)),
                  n_mean=(xt.shape[-1] * xt.shape[-2]) if self.per_sample else None)
        if kwargs.get("mask_pred_original_sample", False):
            if kwargs.get("use_lpips", False) and self._has_lpips():
                return None             # LPIPS regulariser: not one of the fused kernels
            if not kwargs.get("use_l2", False):
                if kwargs.get("use_lpips", False):
                    raise NotImplementedError("LPIPS is unavailable offline")
                raise ValueError("No metric specified")
            if mask is None or kwargs.get("x_0") is None or kwargs.get("lambda_") is None:
                raise ValueError("mask_pred_original_sample needs mask, x_0 and lambda_")
            fk.update(l2reg=True, x_ref=kwargs["x_0"], lambda_=kwargs["lambda_"])
        return fk

    def _apply_native_decoder(self, xt, model_output, coeffs, model, **kwargs):
        """Built-in colour strategies on a latent model whose decoder runs on the engine in gradient mode: the whole nudge is
        native CUDA with the ANALYTIC loss gradient - x0' prediction kernel -> decoder forward -> closed-form d(loss)/d(image)
        kernel -> decoder backward (dgrad twins) -> fused update kernel.  No autograd graph, no torch arithmetic.
        Returns None when the strategy / model does not qualify (the caller falls back to autograd, as the reference)."""
        spec = self.colour_spec()
        nd = _native_decoder(model, xt.shape[0])
        if spec is None or nd is None or nd[0] is None or self.nudge_zt or not self.nudge_xt:
            return None
        dec, chain = nd
        targets, weights = spec
        mask = kwargs.get("mask")
        mask_pred = bool(kwargs.get("mask_pred_original_sample", False))
        if kwargs.get("mask_attr_grad", False) and mask is None:
            raise ValueError("No mask specified")
        out_size = getattr(dec, "out_size", None)
        if mask_pred:
            if kwargs.get("use_lpips", False) or not kwargs.get("use_l2", False):
                return None            # the generic path raises the reference's errors
            x_0, lam = kwargs.get("x_0"), kwargs.get("lambda_")
            if mask is None or x_0 is None or lam is None or mask.shape[-1] != out_size or x_0.shape[-1] != out_size:
                return None            # shapes that do not broadcast against the decoded image: let torch report it
        gmask = mask if kwargs.get("mask_attr_grad", False) else None
        if gmask is not None and gmask.shape[-1] != xt.shape[-1]:
            return None                # a mask that does not match the latent: the generic path reports it
        img = _decode_x0(xt, model_output, coeffs, dec, chain)
        n_mean = img.shape[-1] * img.shape[-2] * (1 if self.per_sample else img.shape[0])
        d_img = ops.color_loss_grad(img, targets, weights, self.loss_scale, n_mean,
                                    mask=mask if mask_pred else None, x_ref=kwargs.get("x_0") if mask_pred else None,
                                    lambda_=kwargs.get("lambda_") if mask_pred else None)
        return _guide(xt, d_img, dec, chain, coeffs, gmask)

    def _apply_native_lpips(self, xt, model_output, coeffs, model, **kwargs):
        """Built-in colour strategies with the LPIPS regulariser (mask_pred_original_sample + use_lpips) on the native
        LPIPS network: x0' kernel (-> native decoder forward) -> LPIPS forward on 1 - mask * img (formed by its input
        packer) and backward -> one kernel for mask * d colour(mask * img) + lambda_ * d LPIPS -> (native decoder backward)
        -> update kernel.  No autograd.  With B > 1 images the regulariser is lambda_ * sum_b LPIPS_b (the reference's
        autograd call accepts only one image, its loss being (B, 1, 1, 1)).  Returns None when the strategy / model / shapes
        do not qualify (autograd path)."""
        from b200edit.lpips import LPIPS
        spec, lp = self.colour_spec(), getattr(self, "metric", None)
        if (spec is None or not isinstance(lp, LPIPS) or self.nudge_zt or not self.nudge_xt or self.per_sample
                or not kwargs.get("mask_pred_original_sample", False) or not kwargs.get("use_lpips", False)):
            return None
        mask, x_0, lam = kwargs.get("mask"), kwargs.get("x_0"), kwargs.get("lambda_")
        if kwargs.get("mask_attr_grad", False) and mask is None:
            raise ValueError("No mask specified")
        if mask is None or x_0 is None or lam is None or not torch.is_tensor(mask) or not torch.is_tensor(x_0):
            return None
        nd = _native_decoder(model, xt.shape[0])
        if nd is None:
            return None
        dec, chain = nd
        S = lp.config.input_size
        B = xt.shape[0]
        if (B > lp.max_batch or mask.dim() != 4 or mask.shape[0] not in (1, B) or mask.shape[1] not in (1, 3)
                or tuple(mask.shape[2:]) != (S, S) or x_0.dim() != 4 or tuple(x_0.shape[1:]) != (3, S, S)
                or x_0.shape[0] not in (1, B)):
            return None
        gmask = mask if kwargs.get("mask_attr_grad", False) else None
        if gmask is not None and tuple(gmask.shape[1:]) != tuple(xt.shape[1:]):
            return None                # a mask that does not match the sample: the generic path reports it
        targets, weights = spec
        img = _decode_x0(xt, model_output, coeffs, dec, chain)
        if tuple(img.shape[1:]) != (3, S, S):
            return None
        with torch.no_grad():
            lp(img, x_0, mask=mask)
            d_lp = lp.input_grad(torch.ones(B, dtype=torch.float32, device=img.device))
        d_img = ops.lpips_guidance_grad(img, mask, d_lp, targets, weights, self.loss_scale,
                                        img.shape[-1] * img.shape[-2] * B, lam)
        return _guide(xt, d_img, dec, chain, coeffs, gmask)

    def _apply_native_network(self, xt, model_output, coeffs, model, **kwargs):
        """Network strategies with per_sample=True on a native network: x0' kernel (-> chain scaling, native decoder
        forward) -> network forward_keep -> batched loss head (every image's gradient, scaled by loss_scale) -> network
        input_grad (-> native decoder backward) -> update kernel.  No autograd graph, no torch arithmetic.  Image b's nudge
        is the batch-1 nudge of image b.  Returns None when the strategy / model / shapes do not qualify (autograd path)."""
        if (not self.per_sample or self.nudge_zt or not self.nudge_xt
                or kwargs.get("mask_pred_original_sample", False)):
            return None
        mask = kwargs.get("mask")
        if kwargs.get("mask_attr_grad", False) and mask is None:
            raise ValueError("No mask specified")
        B = xt.shape[0]
        nd = _native_decoder(model, B)
        if nd is None:
            return None
        dec, chain = nd
        size = xt.shape[-1] if dec is None else getattr(dec, "out_size", None)
        if size is None:
            return None
        gmask = mask if kwargs.get("mask_attr_grad", False) else None
        if gmask is not None and (not torch.is_tensor(gmask) or gmask.dim() != 4 or gmask.shape[0] not in (1, B)
                                  or gmask.shape[1] not in (1, xt.shape[1]) or gmask.shape[2:] != xt.shape[2:]):
            return None                # a mask that does not match the sample: the generic path reports it
        net = self.native_network(int(size))
        if net is None or B > net.max_batch:
            return None
        img = _decode_x0(xt, model_output, coeffs, dec, chain)
        d_img = net.input_grad(self.native_head_grad(net.forward_keep(img)))
        return _guide(xt, d_img, dec, chain, coeffs, gmask)

    def in_window(self, step_idx: int) -> bool:
        return self.t1 <= step_idx < self.t2

    def apply(self, xt, zt, model_output, timestep, step_idx, model, **kwargs):
        """Returns (xt, zt) with xt nudged (and zt if nudge_zt).  ``model`` is the diffusion wrapper
        (needs .scheduler and .decode)."""
        if not self.in_window(step_idx):
            return xt, zt
        coeffs = model.scheduler.coeffs(int(timestep), 0.0, "ddim")
        fk = self.fused_kwargs(xt, model, **kwargs)
        if fk is None:
            out = self._apply_native_network(xt, model_output, coeffs, model, **kwargs)
            if out is not None:
                return out, zt
            out = self._apply_native_lpips(xt, model_output, coeffs, model, **kwargs)
            if out is not None:
                return out, zt
            out = self._apply_native_decoder(xt, model_output, coeffs, model, **kwargs)
            if out is not None:
                return out, zt
            return self._apply_autograd(xt, zt, model_output, coeffs, model, **kwargs)
        if fk.pop("l2reg", False):
            out, _ = ops.guided_step_l2reg(xt, model_output, coeffs, x_ref=fk["x_ref"], mask=fk["mask"],
                                           lambda_=fk["lambda_"], targets=fk["targets"], weights=fk["weights"],
                                           loss_scale=fk["loss_scale"], mask_grad=fk["mask_grad"],
                                           n_mean=fk["n_mean"], no_step=True)
        else:
            out, _ = ops.guided_step(xt, model_output, coeffs, want_x0=False, no_step=True, **fk)
        return out, zt


class SingleColorAttrFunc(AttrFunc):
    """Pull one colour channel towards a target value."""

    def __init__(self, target: float, color_idx: int, **kwargs) -> None:
        super().__init__(**kwargs)
        self.target, self.color_idx = target, color_idx

    def loss(self, p_t: torch.Tensor, **kwargs) -> torch.Tensor:
        return single_color_loss(p_t, self.color_idx, self.target)

    def colour_spec(self):
        t = [None, None, None]
        if not 0 <= self.color_idx < 3:
            return None
        t[self.color_idx] = self.target
        return t, None


class MultiColorAttrFunc(AttrFunc):
    """Pull all three colour channels towards (r, g, b); each channel's error is weighted by its target."""

    def __init__(self, r_target: float, g_target: float, b_target: float, **kwargs) -> None:
        super().__init__(**kwargs)
        self.r_target, self.g_target, self.b_target = r_target, g_target, b_target

    def loss(self, p_t: torch.Tensor, **kwargs) -> torch.Tensor:
        # the reference's loss() takes no **kwargs and therefore raises TypeError whenever the
        # pipeline passes its kwargs (always); accepting them keeps the math and makes it usable
        return color_loss(p_t, r_target=self.r_target, g_target=self.g_target, b_target=self.b_target)

    def colour_spec(self):
        t = [self.r_target, self.g_target, self.b_target]
        return t, t


class NetAttrFunc(AttrFunc):
    """Segmentation-area guidance: softmax over the parser's classes, mean area of the selected
    classes (area normalised by the literal 256*256 of the reference)."""

    def __init__(self, segmentation_model, idx_for_class: list, **kwargs) -> None:
        super().__init__(**kwargs)
        self.segmentation_model = segmentation_model
        self.idx_for_class = idx_for_class
        # the native face parser differentiates through its own dgrad kernels once gradient mode is on
        net = getattr(segmentation_model, "net", None)
        if hasattr(net, "enable_grad") and not getattr(net, "differentiable", True):
            net.enable_grad()

    def _head_ids(self):
        """The class ids when the fused head can evaluate the loss (a list of distinct ids), else None."""
        if not isinstance(self.idx_for_class, (list, tuple)):
            return None
        ids = [int(c) for c in self.idx_for_class]
        return ids if len(set(ids)) == len(ids) else None

    def loss(self, img, **kwargs):
        out = self.segmentation_model.net(img)[0]
        ids = self._head_ids()
        if self.per_sample:
            # sum_b of the reference's loss on image b alone
            if ids is not None and out.is_cuda and out.dtype == torch.float32 and out.dim() == 4 and out.shape[1] <= 32:
                return ops.seg_area_loss(out, ids, per_sample=True)
            area = out.softmax(dim=1).sum(dim=(2, 3)) / (256 * 256)
            return area[:, self.idx_for_class].sum()
        if (ids is not None and out.is_cuda and out.dtype == torch.float32 and out.dim() == 4 and out.shape[0] == 1
                and out.shape[1] <= 32):
            # fused head: softmax + selected-class area and its analytic gradient in one kernel; the parser
            # itself (the user's torch module) is differentiated by autograd as in the reference
            return ops.seg_area_loss(out, ids)
        out = out.squeeze(0).softmax(dim=0)
        out = out.sum(dim=(1, 2)) / (256 * 256)
        return out[self.idx_for_class].sum()

    def native_network(self, size):
        from b200edit.bisenet import BiSeNet, MultiResBiSeNet
        net = getattr(self.segmentation_model, "net", None)
        ids = self._head_ids()
        if ids is None:
            return None
        if isinstance(net, MultiResBiSeNet):
            if size % 32 or size < 64 or net.n_classes > 32:
                return None
            net = net.engine(size, grad=True)
        if (not isinstance(net, BiSeNet) or not net.differentiable or net.config.input_size != size
                or net.config.n_classes > 32):
            return None
        return net

    def native_head_grad(self, logits):
        _, grad = ops.seg_area_head(logits, self._head_ids(), per_sample=True, grad_scale=self.loss_scale)
        return grad


class ClassifierAttrFunc(AttrFunc):
    """Classifier guidance on an 80-logit (40 attributes x 2) predictor; uses batch element 0 (per_sample: every image)."""

    def __init__(self, predictor, idx_for_class, idx_of_interest=0, regularize_idx_idx_score=(None, None, None),
                 **kwargs) -> None:
        super().__init__(**kwargs)
        self.predictor = predictor
        self.idx_for_class, self.idx_of_interest = idx_for_class, idx_of_interest
        self.regularize_idx_idx_score = regularize_idx_idx_score

    def _fused_head(self):
        return isinstance(self.idx_for_class, int) and self.idx_of_interest in (0, 1)

    def loss(self, xt, **kwargs):
        logits = self.predictor(xt)
        r_idx, r_pred, r_score = self.regularize_idx_idx_score
        if self.per_sample:
            # sum_b of the reference's loss on image b alone (its first 80 logits)
            if (self._fused_head() and logits.is_cuda and logits.dtype == torch.float32 and logits.dim() == 2
                    and logits.shape[1] == 80):
                return ops.classifier_logit_loss(logits, self.idx_for_class, self.idx_of_interest,
                                                 self.regularize_idx_idx_score, per_sample=True)
            attr = logits.reshape(logits.shape[0], -1)[:, :80].reshape(-1, 40, 2)
            value = attr[:, self.idx_for_class, self.idx_of_interest]
            if r_idx is not None:
                value = value + (attr[:, r_idx, r_pred] + r_score[r_pred]) ** 2
            return value.sum()
        if (logits.is_cuda and logits.dtype == torch.float32 and logits.numel() % 80 == 0 and self._fused_head()):
            return ops.classifier_logit_loss(logits, self.idx_for_class, self.idx_of_interest,
                                             self.regularize_idx_idx_score)
        attr = logits.view(-1, 40, 2)
        value = attr[0][self.idx_for_class][self.idx_of_interest]
        if r_idx is not None:
            value = value + (attr[0][r_idx][r_pred] + r_score[r_pred]) ** 2
        return value

    def native_network(self, size):
        from b200edit.resnet import ResNet
        net = self.predictor
        cfg = getattr(net, "config", None)
        if (not self._fused_head() or not isinstance(net, ResNet) or cfg.num_classes != 80 or cfg.in_channels != 3
                or cfg.input_size != size):
            return None
        return net

    def native_head_grad(self, logits):
        _, grad = ops.classifier_head(logits, self.idx_for_class, self.idx_of_interest, self.regularize_idx_idx_score,
                                      per_sample=True, grad_scale=self.loss_scale)
        return grad


class AnyGANAttrFunc(ClassifierAttrFunc):
    """The reference's registry and metrics import this name, which its attr_functions never
    defines (ImportError); it is the classifier strategy fed by the AnyCost-GAN attribute predictor."""

__all__ = ["AttrFunc", "SingleColorAttrFunc", "MultiColorAttrFunc", "NetAttrFunc", "ClassifierAttrFunc",
           "AnyGANAttrFunc", "l2_norm", "single_color_loss", "color_loss", "apply_lpips", "B2EError"]
