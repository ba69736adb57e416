"""Tensor-level wrappers over the C ABI.  Inputs are CUDA fp32 contiguous torch tensors; outputs
are freshly allocated with torch (functional semantics, like the reference).  All launches go to
torch's current stream; nothing here synchronises with the host."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _C
from ._C import GuidedStepParams, L2RegParams, StepCoeffs, check, lib


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise _C.B2EError(f"{name}: tensor is on {t.device}; the b200edit operators are CUDA-only "
                          "(no CPU fallback)")
    if t.dtype != torch.float32:
        raise _C.B2EError(f"{name}: expected float32, got {t.dtype}")
    _C.require_device()
    return t.contiguous()


# ----------------------------------------------------------------------------- coefficients
def step_coeffs(alphas_cumprod: torch.Tensor, final_alpha_cumprod, t: int, t_prev: int,
                eta: float = 0.0, mode: str = "ddim") -> StepCoeffs:
    """Per-step scalars, formed exactly like the reference forms them: as fp32 0-d CPU tensors
    with torch's own scalar kernels and the reference's op order (src/diffusion_utils.py:6-31,
    DDIMScheduler.step, src/ddpm_inversion.py:203-229).  torch's CPU ``x ** 0.5`` is not always
    the correctly rounded square root, so the host layer deliberately uses torch here rather
    than C ``sqrtf`` (b2e_step_coeffs_compute is the torch-free variant, within 1 ulp)."""
    ac = alphas_cumprod
    a_t = ac[t]
    a_p = ac[t_prev] if t_prev >= 0 else torch.as_tensor(final_alpha_cumprod, dtype=torch.float32)
    b_t = 1 - a_t
    var = ((1 - a_p) / b_t) * (1 - a_t / a_p)
    sigma = eta * var ** 0.5
    if mode == "ddim":
        dirc = (1 - a_p - sigma ** 2) ** 0.5
    else:
        dirc = (1 - a_p - eta * var) ** 0.5
    out = StepCoeffs()
    out.sqrt_a_t = float(a_t ** 0.5)
    out.sqrt_b_t = float(b_t ** 0.5)
    out.sqrt_a_prev = float(a_p ** 0.5)
    out.dir_coef = float(dirc)
    out.sigma = float(sigma)
    out.a_t_sq = float(a_t ** 2)
    out.variance = float(var)
    out.a_t = float(a_t)
    out.a_prev = float(a_p)
    return out


def step_coeffs_c(alphas_cumprod: torch.Tensor, final_alpha_cumprod: float, t: int, t_prev: int,
                  eta: float = 0.0, mode: str = "ddim") -> StepCoeffs:
    """Torch-free coefficients from the C ABI (IEEE sqrtf)."""
    ac = alphas_cumprod
    if ac.device.type != "cpu" or ac.dtype != torch.float32 or not ac.is_contiguous():
        ac = ac.detach().to("cpu", torch.float32).contiguous()
    out = StepCoeffs()
    check(lib.b2e_step_coeffs_compute(C.c_void_p(ac.data_ptr()), ac.numel(), float(final_alpha_cumprod),
                                      int(t), int(t_prev), float(eta), 0 if mode == "ddim" else 1,
                                      C.byref(out)), "step_coeffs")
    return out


# ----------------------------------------------------------------------------- fused step
def _fill_params(p: GuidedStepParams, c: StepCoeffs, B, Cc, HW, clip, clip_range, z, mask,
                 targets, weights, loss_scale, mask_grad, n_mean):
    p.c = c
    p.clip = int(bool(clip))
    p.clip_range = float(clip_range)
    p.has_noise = int(z is not None)
    p.noise_batched = int(z is not None and z.dim() == 4 and z.shape[0] == B and B > 1)
    p.guide = int(targets is not None)
    n = float(B * HW) if n_mean is None else float(n_mean)
    if targets is not None:
        for i in range(Cc):
            tgt = targets[i] if i < len(targets) else None
            p.has_target[i] = int(tgt is not None)
            if tgt is not None:
                p.target[i] = float(tgt)
                w = 1.0 if weights is None else float(weights[i])
                # k_c = loss_scale (* w_c) / N in fp32, the order of the autograd chain
                k = torch.tensor(float(loss_scale), dtype=torch.float32)
                if w != 1.0:
                    k = k * torch.tensor(w, dtype=torch.float32)
                p.coef[i] = float(k / n)
    p.mask_grad = int(bool(mask_grad) and mask is not None)
    p.mask_batched = int(mask is not None and mask.shape[0] == B and B > 1)


def guided_step(x_t: torch.Tensor, eps: torch.Tensor, c: StepCoeffs, *, clip=False, clip_range=1.0,
                noise: Optional[torch.Tensor] = None, targets: Optional[Sequence] = None,
                weights: Optional[Sequence] = None, loss_scale: float = 1.0,
                mask: Optional[torch.Tensor] = None, mask_grad=False, n_mean=None, want_x0=True,
                no_step=False):
    """Fused x0-prediction + scheduler update (+ sigma*z) + colour guidance.
    Returns (x_prev, x0_pred)."""
    x_t, eps = _f32(x_t, "x_t"), _f32(eps, "eps")
    if x_t.shape != eps.shape or x_t.dim() != 4:
        raise ValueError(f"x_t {tuple(x_t.shape)} and eps {tuple(eps.shape)} must be equal 4-D shapes")
    B, Cc, H, W = x_t.shape
    if noise is not None:
        noise = _f32(noise, "variance_noise")
        if noise.numel() not in (Cc * H * W, B * Cc * H * W):
            raise ValueError(f"variance_noise shape {tuple(noise.shape)} does not broadcast to {tuple(x_t.shape)}")
    if mask is not None:
        mask = _f32(mask, "mask")
        if mask.numel() == H * W or (mask.dim() == 4 and mask.shape[1] == 1):
            mask = mask.expand(mask.shape[0] if mask.dim() == 4 else 1, Cc, H, W).contiguous()
        if mask.numel() not in (Cc * H * W, B * Cc * H * W):
            raise ValueError(f"mask shape {tuple(mask.shape)} does not broadcast to {tuple(x_t.shape)}")
        mask = mask.reshape(-1, Cc, H, W)
    p = GuidedStepParams()
    _fill_params(p, c, B, Cc, H * W, clip, clip_range, noise, mask, targets, weights, loss_scale,
                 mask_grad, n_mean)
    p.no_step = int(bool(no_step))
    x_prev = torch.empty_like(x_t)
    x0 = torch.empty_like(x_t) if want_x0 else None
    check(lib.b2e_guided_step_f32(_p(x_t), _p(eps), _p(noise), _p(mask), _p(x_prev), _p(x0), B, Cc,
                                  H * W, C.byref(p), _stream()), "guided_step")
    return x_prev, x0


def guided_step_l2reg(x_t, eps, c: StepCoeffs, *, x_ref, mask, lambda_, targets, weights=None,
                      loss_scale=1.0, clip=False, clip_range=1.0, noise=None, mask_grad=False,
                      guide=True, n_mean=None, no_step=False):
    """Masked + L2-regularised colour guidance (two-pass).  Returns (x_prev, x0_pred)."""
    x_t, eps, x_ref, mask = _f32(x_t, "x_t"), _f32(eps, "eps"), _f32(x_ref, "x_0"), _f32(mask, "mask")
    B, Cc, H, W = x_t.shape
    if noise is not None:
        noise = _f32(noise, "variance_noise")
    mask = mask.reshape(-1, Cc, H, W)
    if x_ref.shape != x_t.shape:
        x_ref = x_ref.expand_as(x_t).contiguous()
    p = L2RegParams()
    _fill_params(p.base, c, B, Cc, H * W, clip, clip_range, noise, mask, targets, weights, loss_scale,
                 mask_grad, n_mean)
    p.base.guide = int(bool(guide))
    p.base.no_step = int(bool(no_step))
    p.base.mask_batched = int(mask.shape[0] == B and B > 1)
    p.lambda_ = float(lambda_)
    p.loss_scale = float(loss_scale)
    ws_bytes = lib.b2e_l2reg_workspace_bytes(B, Cc, H * W)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x_t.device)
    x_prev, x0 = torch.empty_like(x_t), torch.empty_like(x_t)
    check(lib.b2e_guided_step_l2reg_f32(_p(x_t), _p(eps), _p(noise), _p(mask), _p(x_ref), _p(x_prev),
                                        _p(x0), B, Cc, H * W, C.byref(p), _p(ws), ws_bytes, _stream()),
          "guided_step_l2reg")
    return x_prev, x0


def apply_guidance_grad(x, neg_grad, a_t_sq: float, mask=None):
    x, neg_grad = _f32(x, "x").clone(), _f32(neg_grad, "grad")
    B = x.shape[0]
    chw = x.numel() // B
    mb = 0
    if mask is not None:
        mask = _f32(mask, "mask").expand(-1, *x.shape[1:]).contiguous() if mask.dim() == 4 else _f32(mask, "mask")
        mb = int(mask.numel() == x.numel() and B > 1)
    check(lib.b2e_apply_guidance_grad_f32(_p(x), _p(neg_grad), _p(mask), B, chw, mb, float(a_t_sq),
                                          _stream()), "apply_guidance_grad")
    return x


def _color_grad_params(targets, weights, loss_scale, n_mean, Cc):
    p = _C.ColorGradParams()
    for c in range(4):
        t = targets[c] if c < len(targets) else None
        w = 1.0 if weights is None else (weights[c] if c < len(weights) and weights[c] is not None else 0.0)
        p.has_target[c] = int(t is not None and c < Cc)
        p.target[c] = float(t) if t is not None else 0.0
        p.k[c] = float(torch.tensor(float(loss_scale), dtype=torch.float32) * torch.tensor(float(w), dtype=torch.float32)
                       / torch.tensor(float(n_mean), dtype=torch.float32)) if t is not None else 0.0
    return p


def lpips_guidance_grad(img, mask, d_lpips, targets, weights, loss_scale, n_mean, lambda_):
    """d(loss_scale * (colour loss(mask * img) + lambda_ * LPIPS(1 - mask * img, x_0))) / d(img) in one kernel, given
    d_lpips = d(LPIPS) / d(img) from the native LPIPS backward (its -mask chain included).  mask (1 | B, C, H, W)."""
    img, d_lpips = _f32(img, "decoded image"), _f32(d_lpips, "d_lpips")
    B, Cc, H, W = img.shape
    mask = _f32(mask, "mask")
    if mask.shape[1:] != img.shape[1:]:
        mask = mask.expand(mask.shape[0], Cc, H, W).contiguous()
    p = _color_grad_params(targets, weights, loss_scale, n_mean, Cc)
    p.lam_scale = float(loss_scale) * float(lambda_)
    p.mask_batched = int(mask.shape[0] == B and B > 1)
    out = torch.empty_like(img)
    check(lib.b2e_lpips_guidance_grad_f32(_p(img), _p(mask), _p(d_lpips), _p(out), B, Cc, H * W, C.byref(p), _stream()),
          "lpips_guidance_grad")
    return out


def color_loss_grad(img, targets, weights, loss_scale, n_mean, mask=None, x_ref=None, lambda_=None):
    """d(loss_scale * colour loss)/d(decoded image) in closed form (guidance through a latent decoder; the result feeds the
    decoder's native backward pass).  targets / weights as in guided_step; n_mean = elements the loss mean runs over.
    mask + x_ref + lambda_: the masked-prediction + L2-regularised variant (mask_pred_original_sample, use_l2)."""
    img = _f32(img, "decoded image")
    B, Cc, H, W = img.shape
    p = _color_grad_params(targets, weights, loss_scale, n_mean, Cc)
    ws = None
    ws_bytes = 0
    if x_ref is not None:
        if mask is None or lambda_ is None:
            raise ValueError("color_loss_grad: the L2-regularised variant needs mask, x_0 and lambda_")
        mask = _f32(mask, "mask").expand(-1, Cc, H, W).contiguous() if mask.shape[1:] != img.shape[1:] else _f32(mask, "mask")
        x_ref = _f32(x_ref, "x_0")
        if x_ref.shape != img.shape:
            x_ref = x_ref.expand_as(img).contiguous()
        p.use_mask_pred = 1
        p.mask_batched = int(mask.shape[0] == B and B > 1)
        p.lam_scale = float(loss_scale) * float(lambda_)
        ws_bytes = lib.b2e_color_loss_grad_workspace_bytes()
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=img.device)
    out = torch.empty_like(img)
    check(lib.b2e_color_loss_grad_f32(_p(img), _p(mask) if x_ref is not None else None, _p(x_ref), _p(out), B, Cc, H * W,
                                      C.byref(p), _p(ws), ws_bytes, _stream()), "color_loss_grad")
    return out


def apply_latent_guidance(x, d_latent, chain: float, sqrt_a_t: float, a_t_sq: float, mask=None):
    """x + (mask *) (-(d_latent * chain) / sqrt_a_t) * a_t_sq  (new tensor): the nudge of AttrFunc.apply once the decoder's
    backward pass has produced d_latent = dL/d(decoder input)."""
    x, d_latent = _f32(x, "x").clone(), _f32(d_latent, "d_latent")
    B = x.shape[0]
    chw = x.numel() // B
    mb = 0
    if mask is not None:
        mask = _f32(mask, "mask").expand(-1, *x.shape[1:]).contiguous() if mask.dim() == 4 else _f32(mask, "mask")
        mb = int(mask.numel() == x.numel() and B > 1)
    check(lib.b2e_apply_latent_guidance_f32(_p(x), _p(d_latent), _p(mask), B, chw, mb, float(chain), float(sqrt_a_t),
                                            float(a_t_sq), _stream()), "apply_latent_guidance")
    return x


# ----------------------------------------------------------------------------- single ops
def pred_x0(x_t, eps, sqrt_a_t: float, sqrt_b_t: float):
    x_t, eps = _f32(x_t, "sample"), _f32(eps, "model_output")
    out = torch.empty_like(x_t)
    check(lib.b2e_pred_x0_f32(_p(x_t), _p(eps), _p(out), x_t.numel(), sqrt_a_t, sqrt_b_t, _stream()), "pred_x0")
    return out


def renoise(x, eps, c_a: float, c_b: float, c_out_x0: float, c_out_e: float):
    x, eps = _f32(x, "sample"), _f32(eps, "model_output")
    out = torch.empty_like(x)
    check(lib.b2e_renoise_f32(_p(x), _p(eps), _p(out), x.numel(), c_a, c_b, c_out_x0, c_out_e, _stream()),
          "renoise")
    return out


def axpby(x, y, a: float, b: float):
    """out = a*x + b*y (two rounded products, one rounded sum)."""
    x, y = _f32(x, "x"), _f32(y, "y")
    if x.shape != y.shape:
        y = y.expand_as(x).contiguous()
    out = torch.empty_like(x)
    check(lib.b2e_axpby_f32(_p(x), _p(y), _p(out), x.numel(), float(a), float(b), _stream()), "axpby")
    return out


def _loss_ws(device):
    n = lib.b2e_loss_workspace_bytes()
    return torch.empty(n, dtype=torch.uint8, device=device), n


def l2_distance(x, y):
    """sqrt(sum((x-y)^2)) as a 0-d CUDA tensor (src/attr_functions.py:11-13)."""
    x, y = _f32(x, "x"), _f32(y, "y")
    if x.shape != y.shape:
        y = y.expand_as(x).contiguous()
    ws, n = _loss_ws(x.device)
    out = torch.empty(1, dtype=torch.float32, device=x.device)
    check(lib.b2e_l2_distance_f32(_p(x), _p(y), x.numel(), _p(out), _p(ws), n, _stream()), "l2_distance")
    return out[0]


def channel_l1(img, targets):
    """Per-channel mean |img[:,c] - targets[c]| over (B,H,W) -> fp32 CUDA tensor [C]."""
    img = _f32(img, "images")
    B, Cc, H, W = img.shape
    tg = (C.c_float * 4)(*([float(t if t is not None else 0.0) for t in targets] + [0.0] * (4 - len(targets))))
    ws, n = _loss_ws(img.device)
    out = torch.empty(4, dtype=torch.float32, device=img.device)
    check(lib.b2e_channel_l1_f32(_p(img), B, Cc, H * W, tg, _p(out), _p(ws), n, _stream()), "channel_l1")
    return out[:Cc]


def seg_area_head(logits, classes, area_divisor=256.0 * 256.0, want_grad=True, per_sample=False, grad_scale=1.0):
    """NetAttrFunc.loss head (src/attr_functions.py:213-219) on the parser logits of ONE image, (C,H,W) or
    (1,C,H,W): returns (loss 0-d tensor, dL/dlogits with the shape of ``logits`` or None).
    ``per_sample=True``: logits (B,C,H,W), the head of every image on its own -> (loss (B,), dL_b/dlogits_b * grad_scale);
    image b's values are bit-identical to a B = 1 call on image b."""
    lg = _f32(logits, "logits")
    ids = [int(c) for c in classes]
    arr = (C.c_int32 * max(1, len(ids)))(*ids)
    if per_sample:
        if lg.dim() != 4:
            raise ValueError(f"seg_area_head(per_sample=True): expected (B,C,H,W) logits, got {tuple(lg.shape)}")
        B, Cc, H, W = lg.shape
        n = lib.b2e_seg_area_head_batched_workspace_bytes(B)
        ws = torch.empty(n, dtype=torch.uint8, device=lg.device)
        loss = torch.empty(B, dtype=torch.float32, device=lg.device)
        grad = torch.empty_like(lg) if want_grad else None
        check(lib.b2e_seg_area_head_batched_f32(_p(lg), B, Cc, H * W, arr, len(ids), float(area_divisor), float(grad_scale),
                                                _p(loss), _p(grad), _p(ws), n, _stream()), "seg_area_head")
        return loss, grad
    if lg.dim() == 4:
        if lg.shape[0] != 1:
            raise ValueError("seg_area_head: the reference head squeezes batch dimension 0 (batch 1 only)")
        core = lg[0]
    else:
        core = lg
    Cc, H, W = core.shape
    n = lib.b2e_seg_area_head_workspace_bytes()
    ws = torch.empty(n, dtype=torch.uint8, device=lg.device)
    loss = torch.empty(1, dtype=torch.float32, device=lg.device)
    grad = torch.empty_like(lg) if want_grad else None
    check(lib.b2e_seg_area_head_f32(_p(core), Cc, H * W, arr, len(ids), float(area_divisor), _p(loss), _p(grad),
                                    _p(ws), n, _stream()), "seg_area_head")
    return loss[0], grad


def _classifier_reg(reg):
    r_idx, r_pred, r_score = reg
    if r_idx is None:
        return -1, 0, 0.0
    return int(r_idx), int(r_pred), float(r_score[int(r_pred)])


def classifier_head(logits, idx_for_class: int, idx_of_interest: int = 0, reg=(None, None, None), want_grad=True,
                    per_sample=False, grad_scale=1.0):
    """ClassifierAttrFunc.loss head (src/attr_functions.py:237-257) on (B,80) logits: (loss 0-d, dL/dlogits).
    ``per_sample=True``: the head of every row on its own -> (loss (B,), dL_b/dlogits_b * grad_scale)."""
    lg = _f32(logits, "logits")
    ri, rp, rs = _classifier_reg(reg)
    if per_sample:
        if lg.dim() != 2 or lg.shape[1] != 80:
            raise ValueError(f"classifier_head(per_sample=True): expected (B,80) logits, got {tuple(lg.shape)}")
        B = lg.shape[0]
        loss = torch.empty(B, dtype=torch.float32, device=lg.device)
        grad = torch.empty_like(lg) if want_grad else None
        check(lib.b2e_classifier_head_batched_f32(_p(lg), B, int(idx_for_class), int(idx_of_interest), ri, rp, rs,
                                                  float(grad_scale), _p(loss), _p(grad), _stream()), "classifier_head")
        return loss, grad
    loss = torch.empty(1, dtype=torch.float32, device=lg.device)
    grad = torch.empty_like(lg) if want_grad else None
    check(lib.b2e_classifier_head_f32(_p(lg), lg.numel(), int(idx_for_class), int(idx_of_interest), ri, rp, rs,
                                      _p(loss), _p(grad), _stream()), "classifier_head")
    return loss[0], grad


class _SegAreaHeadFn(torch.autograd.Function):
    """loss = head(logits) with the analytic gradient from the same kernel launch (the network below it is the
    user's torch module and is differentiated by autograd, exactly as in the reference).  per_sample: sum_b L_b."""

    @staticmethod
    def forward(ctx, logits, classes, area_divisor, per_sample=False):
        loss, grad = seg_area_head(logits.detach(), classes, area_divisor, want_grad=True, per_sample=per_sample)
        ctx.save_for_backward(grad)
        return loss.sum() if per_sample else loss

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return grad * g, None, None, None


class _ClassifierHeadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, idx_for_class, idx_of_interest, reg, per_sample=False):
        loss, grad = classifier_head(logits.detach(), idx_for_class, idx_of_interest, reg, want_grad=True,
                                     per_sample=per_sample)
        ctx.save_for_backward(grad)
        return loss.sum() if per_sample else loss

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return grad * g, None, None, None, None


def seg_area_loss(logits, classes, area_divisor=256.0 * 256.0, per_sample=False):
    """Differentiable NetAttrFunc head (fused value + analytic gradient); per_sample: sum_b of each image's head."""
    return _SegAreaHeadFn.apply(logits, tuple(int(c) for c in classes), float(area_divisor), bool(per_sample))


def classifier_logit_loss(logits, idx_for_class, idx_of_interest=0, reg=(None, None, None), per_sample=False):
    """Differentiable ClassifierAttrFunc head (fused value + analytic gradient); per_sample: sum_b of each row's head."""
    return _ClassifierHeadFn.apply(logits, int(idx_for_class), int(idx_of_interest), reg, bool(per_sample))


def cfg_combine(e_first, e_second, scale: float):
    e_first, e_second = _f32(e_first, "eps_first"), _f32(e_second, "eps_second")
    out = torch.empty_like(e_first)
    check(lib.b2e_cfg_combine_f32(_p(e_first), _p(e_second), _p(out), out.numel(), float(scale), _stream()),
          "cfg_combine")
    return out


def apply_mask(mask, zo, zv):
    mask, zo, zv = _f32(mask, "mask"), _f32(zo, "zo"), _f32(zv, "zv")
    if zo.shape != zv.shape:
        raise ValueError("apply_mask: zo and zv must have the same shape")
    rows, chw = zo.shape[0], zo[0].numel()
    if mask.numel() == zo.numel() and mask.numel() != chw:
        rows, chw = 1, zo.numel()                 # one mask per image of a (B,C,H,W) batch
    elif mask.numel() != chw:
        mask = mask.expand(1, *zo.shape[1:]).contiguous()
    out = torch.empty_like(zo)
    check(lib.b2e_apply_mask_f32(_p(mask), _p(zo), _p(zv), _p(out), rows, chw, _stream()), "apply_mask")
    return out


def to_uint8(x):
    """(B,C,H,W) fp32 in [-1,1] -> (B,H,W,C) uint8 with the reference's tensor_to_pil numerics."""
    x = _f32(x, "image")
    B, Cc, H, W = x.shape
    out = torch.empty((B, H, W, Cc), dtype=torch.uint8, device=x.device)
    check(lib.b2e_to_uint8_f32(_p(x), _p(out), B, Cc, H * W, _stream()), "to_uint8")
    return out


def sample_xts(x0, noise, sa, sb):
    """x0 (1,C,H,W) or (C,H,W); noise (T,C,H,W); sa/sb fp32 device [T] -> xts (T+1,C,H,W)."""
    x0, noise, sa, sb = _f32(x0, "x0"), _f32(noise, "noise"), _f32(sa, "sa"), _f32(sb, "sb")
    T = noise.shape[0]
    chw = noise[0].numel()
    xts = torch.empty((T + 1,) + tuple(noise.shape[1:]), dtype=torch.float32, device=x0.device)
    check(lib.b2e_sample_xts_f32(_p(x0), _p(noise), _p(sa), _p(sb), _p(xts), T, chw, _stream()), "sample_xts")
    return xts


def extract_noise(x_t, eps, x_tm1: torch.Tensor, z_out: torch.Tensor, c: StepCoeffs):
    """In place: z_out <- (x_tm1 - mu)/sigma ; x_tm1 <- mu + sigma*z."""
    x_t, eps = _f32(x_t, "x_t"), _f32(eps, "eps")
    if not (x_tm1.is_contiguous() and z_out.is_contiguous()):
        raise ValueError("extract_noise: x_tm1 and z_out must be contiguous views")
    check(lib.b2e_extract_noise_f32(_p(x_t), _p(eps), _p(x_tm1), _p(z_out), x_t.numel(), C.byref(c), _stream()),
          "extract_noise")


# ----------------------------------------------------------------------------- masks
def mask_from_seg(seg: torch.Tensor, classes: Sequence[int], dilate: bool, size, channels=3, ksize=7,
                  antialias=True):
    """(H,W) parsing map -> (1,channels,oh,ow) mask; an (N,H,W) stack of N > 1 maps -> (N,channels,oh,ow) in one call,
    map n bit-identical to the single-map result."""
    if not seg.is_cuda:
        raise _C.B2EError("mask_from_seg: segmentation must be a CUDA tensor (no CPU fallback)")
    _C.require_device()
    seg = seg.to(torch.int64).contiguous()
    H, W = seg.shape[-2:]
    oh, ow = int(size[0]), int(size[1])
    cls = (C.c_int32 * max(1, len(classes)))(*[int(c) for c in classes])
    if seg.dim() == 3 and seg.shape[0] > 1:
        N = seg.shape[0]
        nbytes = lib.b2e_mask_batched_workspace_bytes(N, H, W, oh, ow)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=seg.device)
        out = torch.empty((N, channels, oh, ow), dtype=torch.float32, device=seg.device)
        check(lib.b2e_mask_from_seg_batched(_p(seg), N, H, W, cls, len(classes), int(bool(dilate)), ksize, oh, ow, channels,
                                            int(bool(antialias)), _p(out), _p(ws), nbytes, _stream()), "mask_from_seg")
        return out
    nbytes = lib.b2e_mask_workspace_bytes(H, W, oh, ow)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=seg.device)
    out = torch.empty((1, channels, oh, ow), dtype=torch.float32, device=seg.device)
    check(lib.b2e_mask_from_seg(_p(seg), H, W, cls, len(classes), int(bool(dilate)), ksize, oh, ow, channels,
                                int(bool(antialias)), _p(out), _p(ws), nbytes, _stream()), "mask_from_seg")
    return out


def resize_bilinear_aa(x: torch.Tensor, size):
    x = _f32(x, "image")
    H, W = x.shape[-2:]
    lead = x.shape[:-2]
    oh, ow = int(size[0]), int(size[1])
    nbytes = lib.b2e_mask_workspace_bytes(H, W, oh, ow)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    planes = x.reshape(-1, H, W)
    out = torch.empty((planes.shape[0], oh, ow), dtype=torch.float32, device=x.device)
    for i in range(planes.shape[0]):
        check(lib.b2e_resize_bilinear_aa_f32(_p(planes[i]), H, W, _p(out[i]), oh, ow, _p(ws), nbytes, _stream()),
              "resize_bilinear_aa")
    return out.reshape(*lead, oh, ow)


def bilinear_argmax(x_nhwc: torch.Tensor, K: int, S: int, planes: int = 1) -> torch.Tensor:
    """Test hook for the face parser's label kernel: x (N,Hi,Wi,planes*P) in the engine's 16-bit type (``act_dtype()``)
    -> (N,S,S) int64, the argmax over the first K channels of the align_corners bilinear upsampling to S x S."""
    _C.require_device()
    if not x_nhwc.is_cuda or x_nhwc.dtype != act_dtype() or x_nhwc.dim() != 4 or x_nhwc.shape[-1] % planes:
        raise ValueError(f"bilinear_argmax: x must be a CUDA {act_dtype()} (N,Hi,Wi,planes*P) tensor")
    N, Hi, Wi, PP = x_nhwc.shape
    out = torch.empty((N, S, S), dtype=torch.int64, device=x_nhwc.device)
    check(lib.b2e_bilinear_ac_argmax_f16(_p(x_nhwc.contiguous()), _p(out), N, Hi, Wi, PP // planes, K, S, planes, _stream()),
          "bilinear_argmax")
    return out


def morphology2d(x, weight, op: str, soft_max=False, beta=20.0):
    x, weight = _f32(x, "x"), _f32(weight, "weight")
    B, Cin, H, W = x.shape
    Cout, Cin2, k, k2 = weight.shape
    if Cin2 != Cin or k != k2:
        raise ValueError("morphology2d: weight shape does not match input")
    out = torch.empty((B, Cout, H, W), dtype=torch.float32, device=x.device)
    check(lib.b2e_morphology2d_f32(_p(x), _p(weight), _p(out), B, Cin, Cout, H, W, k,
                                   0 if op == "dilation2d" else 1, int(bool(soft_max)), float(beta), _stream()),
          "morphology2d")
    return out


def act_dtype():
    """torch dtype of the engine's 16-bit activations / tensor-core operands (fp16 unless built with -DB2E_ACT_BF16)."""
    return torch.bfloat16 if lib.b2e_act_dtype() == 1 else torch.float16


def upsample_conv3x3_nhwc_f16(x, w, bias):
    """Test hook: conv3x3(nearest-upsample x2 (x)) + bias as four 2x2 sub-pixel phase convolutions (16-bit NHWC)."""
    _C.require_device()
    N, H, W, Cin = x.shape
    Cout = w.shape[0]
    if x.dtype != act_dtype() or tuple(w.shape[1:]) != (Cin, 3, 3):
        raise ValueError(f"upsample_conv3x3_nhwc_f16: x must be {act_dtype()} (N,H,W,Cin), w (Cout,Cin,3,3)")
    out = torch.empty((N, 2 * H, 2 * W, Cout), dtype=act_dtype(), device=x.device)
    check(lib.b2e_upsample_conv3x3_nhwc_f16(_p(x.contiguous()), _p(w.contiguous().float()),
                                            _p(bias.contiguous().float()) if bias is not None else None, _p(out), N, H, W,
                                            Cin, Cout, _stream()), "upsample_conv3x3_nhwc_f16")
    return out


ATTENTION_PATHS = {"fused": 0, "materialised": 1, "single_head": 2, "cuda_core": 3, "fp32_split": 4, "fp32_tiled": 5,
                   "fp32_tiled_causal": 6}


def split_planes(x: torch.Tensor) -> torch.Tensor:
    """fp32 (..., P) -> the fp32-accurate mode's split tensor (..., 3P): [hi | lo | hi] planes, hi = 16-bit(x),
    lo = 16-bit(x - hi)."""
    hi = x.to(act_dtype())
    lo = (x - hi.float()).to(act_dtype())
    return torch.cat([hi, lo, hi], dim=-1).contiguous()


def merge_planes(x: torch.Tensor) -> torch.Tensor:
    """Split tensor (..., 3P) -> fp32 hi + lo (..., P)."""
    P = x.shape[-1] // 3
    return x[..., :P].float() + x[..., P:2 * P].float()


def attention_f16(q, kv, *, hw, heads, head_dim, k_col, v_col, out_pitch, q_col=0, valid_k=None, causal=False,
                  path="fused", softmax_warps=8, out=None):
    """Test hook for the attention paths (include/b200edit.h, b2e_attention_f16): softmax(Q K^T / sqrt(head_dim)) V over
    channel windows, keys >= valid_k (default: all) masked, through the engine's own launch sequence of `path`
    (one of ATTENTION_PATHS; "fp32_tiled_causal" is the causal instantiation of "fp32_tiled" and needs causal=True).

    q (B, H*W, q_pitch) and kv (B, Tk, kv_pitch) are token-major tensors in `act_dtype()`; the "fp32_*" paths take fp32
    tensors and split them into [hi | lo | hi] planes here (q is kv: one packed tensor).  Returns `out` (B, H*W, out_pitch)
    in `act_dtype()`, or the split output (B, H*W, 3 * out_pitch) of the fp32 paths (``merge_planes`` gives hi + lo)."""
    _C.require_device()
    if path not in ATTENTION_PATHS:
        raise ValueError(f"attention_f16: path must be one of {sorted(ATTENTION_PATHS)}")
    planes = 3 if path.startswith("fp32") else 1
    want = torch.float32 if planes == 3 else act_dtype()
    if (q.dtype != want or kv.dtype != want or q.dim() != 3 or kv.dim() != 3 or not q.is_cuda or not kv.is_cuda
            or q.shape[1] != hw[0] * hw[1] or q.shape[0] != kv.shape[0]):
        raise ValueError(f"attention_f16: q (B, H*W, pitch), kv (B, Tk, pitch) must be CUDA {want} tensors for path {path}")
    packed = q is kv
    if planes == 3:
        q = split_planes(q)
        kv = q if packed else split_planes(kv)
    else:
        q = q.contiguous()
        kv = q if packed else kv.contiguous()
    B, Tq, qpp = q.shape
    Tk, kvpp = kv.shape[1], kv.shape[2]
    H, W = hw
    if out is None:
        out = torch.empty((B, Tq, planes * out_pitch), dtype=act_dtype(), device=q.device)
    if out.shape != (B, Tq, planes * out_pitch) or out.dtype != act_dtype() or not out.is_contiguous():
        raise ValueError("attention_f16: out must be a contiguous (B, H*W, planes * out_pitch) tensor")
    check(lib.b2e_attention_f16(_p(q), qpp // planes, q_col, _p(kv), kvpp // planes, k_col, v_col, _p(out), out_pitch,
                                B, H, W, Tk, Tk if valid_k is None else valid_k, heads, head_dim, int(bool(causal)),
                                ATTENTION_PATHS[path], softmax_warps, _stream()), "attention_f16")
    return out


def conv2d_nhwc_f16(x, w, bias, stride=1, residual=None):
    """Test hook for the tcgen05 implicit-GEMM convolution (optionally + residual; 16-bit NHWC, `act_dtype()`)."""
    _C.require_device()
    N, H, W, Cin = x.shape
    Cout, _, k, _ = w.shape
    if x.dtype != act_dtype() or (residual is not None and residual.dtype != act_dtype()):
        raise ValueError(f"conv2d_nhwc_f16: operands must be {act_dtype()}")
    out = torch.empty((N, H // stride, W // stride, Cout), dtype=act_dtype(), device=x.device)
    check(lib.b2e_conv2d_nhwc_f16(_p(x.contiguous()), _p(w.contiguous().float()),
                                   _p(bias.contiguous().float()) if bias is not None else None,
                                   _p(residual.contiguous()) if residual is not None else None, _p(out), N, H, W,
                                   Cin, Cout, k, stride, _stream()), "conv2d_nhwc_f16")
    return out
