"""Edit-friendly DDPM inversion and regeneration (drop-in for src/ddpm_inversion.py; algorithm of
Huberman-Spiegelglas et al., arXiv:2304.06140).  Index conventions: xts[idx] is the sample at
scheduler.timesteps[idx] (idx 0 = noisiest), xts[T] = x0; zs[idx] is the noise injected when
stepping from timesteps[idx] to the next cleaner level; zs[T-1] = 0.

Batches (extension): an x0 of B > 1 images (B,C,H,W) is inverted in one pass, every step one batch-B forward of the
noise predictor; xts is then (T+1,B,C,H,W) and zs (T,B,C,H,W), image b's slice equal to inverting image b alone with
the same noise.  One prompt is shared by the batch."""
from typing import Optional

import torch
from tqdm import tqdm

from b200edit import ops
from diffusion_utils import (calculate_variance, compute_alpha_products, compute_predicted_original_sample,
                             encode_text, get_noise_pred, get_previous_timestep, get_variance_noise)

__all__ = ["mu_tilde", "sample_xts_from_x0", "forward_step", "inversion_forward_process", "invert",
           "reverse_step", "inversion_reverse_process", "sample", "calculate_variance", "get_variance_noise"]


def mu_tilde(model, xt, x0, timestep):
    """Posterior mean mu~(x_t, x_0), DDPM eq. 7 (src/ddpm_inversion.py:16-28)."""
    prev_t = get_previous_timestep(model, int(timestep))
    a_t, a_prev = compute_alpha_products(model, int(timestep), prev_t)
    a_bar = model.scheduler.alphas_cumprod[int(timestep)]
    c0 = (a_prev ** 0.5 * (1 - a_t)) / (1 - a_bar)
    ct = (a_t ** 0.5 * (1 - a_prev)) / (1 - a_bar)
    return ops.axpby(x0, xt, float(c0), float(ct))


def _is_batch(x0) -> bool:
    return x0.dim() == 4 and x0.shape[0] > 1


def check_batch(model, B: int, cfg: bool):
    """A batch of B > 1 images runs as one forward of the noise predictor (2B samples with classifier-free guidance): it
    must fit the predictor's ``max_batch``."""
    mb = getattr(model.unet, "max_batch", None)
    need = 2 * B if cfg else B
    if B > 1 and mb is not None and need > mb:
        raise ValueError(f"a batch of {B} images needs {need} samples per noise-predictor call"
                         f"{' (classifier-free guidance doubles it)' if cfg else ''}, above the predictor's max_batch {mb}")


def sample_xts_from_x0(model, x0, num_inference_steps=50, noise: Optional[torch.Tensor] = None):
    """Independent forward-noised copies x_t = sqrt(a_t) x0 + sqrt(1-a_t) n_t for every inference
    timestep, plus x0 itself: (T+1,C,H,W) (src/ddpm_inversion.py:31-55).  ``noise`` (T,C,H,W) may be
    injected (noise[idx] belongs to timesteps[idx]); otherwise it is drawn like the reference draws
    it: one randn_like(x0) per timestep, ascending t, on x0's device generator.  x0 (B,C,H,W) with B > 1:
    (T+1,B,C,H,W), ``noise`` (T,B,C,H,W), each timestep's draw one randn_like over the batch."""
    sch = model.scheduler
    ts = sch.timesteps
    T = len(ts)
    batched = _is_batch(x0)
    if not batched:
        x0 = x0.reshape(1, *x0.shape[-3:])
    elif noise is not None and tuple(noise.shape) != (T,) + tuple(x0.shape):
        raise ValueError(f"noise must be (T, B, C, H, W) = {(T,) + tuple(x0.shape)} for x0 {tuple(x0.shape)}, "
                         f"got {tuple(noise.shape)}")
    if noise is None:
        draws = [None] * T
        for idx in reversed(range(T)):
            draws[idx] = torch.randn_like(x0) if batched else torch.randn_like(x0)[0]
        noise = torch.stack(draws)
    ac = sch.alphas_cumprod
    sa = (ac[ts] ** 0.5).to(x0.device)
    sb = ((1 - ac) ** 0.5)[ts].to(x0.device)
    return ops.sample_xts(x0, noise, sa, sb)


def forward_step(model, model_output, timestep, sample):
    """eta = 0 inversion step: x0-prediction re-noised to t + stride (src/ddpm_inversion.py:58-77)."""
    sch = model.scheduler
    t = int(timestep)
    n = sch.config.num_train_timesteps
    t_next = min(n - 2, t + n // sch.num_inference_steps)
    a_t, a_n = sch.alphas_cumprod[t], sch.alphas_cumprod[t_next]
    return ops.renoise(sample, model_output, float(a_t ** 0.5), float((1 - a_t) ** 0.5), float(a_n ** 0.5),
                       float((1 - a_n) ** 0.5))


def inversion_forward_process(model, x0, etas=None, num_inference_steps=50, prompt: Optional[str] = None,
                              cfg_scale: float = 3.5, prog_bar=False, noise: Optional[torch.Tensor] = None):
    if _is_batch(x0):
        check_batch(model, x0.shape[0], prompt is not None)
    context = None
    if prompt is not None:
        context = torch.cat([encode_text(model, prompt), encode_text(model, "")])
    sch = model.scheduler
    sch.set_timesteps(num_inference_steps)
    ts = [int(t) for t in sch.timesteps]
    T = len(ts)
    eta_is_zero = etas is None or (type(etas) in [int, float] and etas == 0)
    if not eta_is_zero:
        if type(etas) in [int, float]:
            etas = [etas] * T
        xts = sample_xts_from_x0(model, x0, num_inference_steps=num_inference_steps, noise=noise)
        zs = torch.zeros((T,) + tuple(xts.shape[1:]), device=xts.device, dtype=torch.float32)
    else:
        xts, zs = None, None
    xt = x0
    order = list(reversed(range(T)))
    for idx in (tqdm(order) if prog_bar else order):
        t = ts[idx]
        if not eta_is_zero:
            xt = xts[idx] if xts.dim() == 5 else xts[idx][None]
        eps = get_noise_pred(model, xt, torch.tensor(t), context, cfg_scale)
        if eta_is_zero:
            xt = forward_step(model, eps, t, xt)
        else:
            # z_t = (x_{t-1} - mu_t)/(eta sqrt(var)); x_{t-1} <- mu_t + eta sqrt(var) z_t  (one kernel, in place)
            ops.extract_noise(xt, eps, xts[idx + 1], zs[idx], sch.coeffs(t, etas[idx], "ddpm"))
    if zs is not None:
        zs[-1].zero_()
    return xt, zs, xts


def invert(model, x0, num_inference_steps=50, eta=1, prompt: Optional[str] = None, cfg_scale: float = 3.5,
           prog_bar=True, noise: Optional[torch.Tensor] = None):
    """Returns (x_T, zs, xts) - Algorithm 1 of arXiv:2304.06140.  x0 (B,C,H,W), B > 1: x_T (B,C,H,W), zs (T,B,C,H,W),
    xts (T+1,B,C,H,W); ``noise`` (T,B,C,H,W)."""
    return inversion_forward_process(model, x0, num_inference_steps=num_inference_steps, etas=eta,
                                     prompt=prompt, cfg_scale=cfg_scale, prog_bar=prog_bar, noise=noise)


def reverse_step(model, model_output, timestep, sample, eta=0, variance_noise=None):
    """DDPM-style reverse step: no clipping, direction coefficient sqrt(1 - a_prev - eta*var)
    (src/ddpm_inversion.py:203-240)."""
    if eta > 0 and variance_noise is None:
        variance_noise = torch.randn(model_output.shape, device=model_output.device)
    prev, _ = ops.guided_step(sample, model_output, model.scheduler.coeffs(int(timestep), eta, "ddpm"),
                              noise=variance_noise if eta > 0 else None, want_x0=False)
    return prev


def inversion_reverse_process(model, xT, eta=0, zs=None, prompt: Optional[str] = None, cfg_scale: float = 3.5,
                              prog_bar=False):
    xt = xT.expand(1, -1, -1, -1) if xT.dim() == 3 else xT
    if zs.dim() == 5 and tuple(zs.shape[1:]) != tuple(xt.shape):
        raise ValueError(f"zs (T', B, C, H, W) {tuple(zs.shape)} does not match the batch xT {tuple(xt.shape)}")
    if _is_batch(xt):
        check_batch(model, xt.shape[0], prompt is not None)
    context = encode_text(model, prompt) if prompt is not None else None
    ts = [int(t) for t in model.scheduler.timesteps][-zs.shape[0]:]
    for idx, t in enumerate(tqdm(ts) if prog_bar else ts):
        eps = get_noise_pred(model, xt, torch.tensor(t), context, cfg_scale)
        xt = reverse_step(model, eps, t, xt, eta=eta, variance_noise=get_variance_noise(zs, idx, eta))
    return xt, zs


def sample(model, zs, xts, Tskip=36, eta=1, prompt: Optional[str] = None, cfg_scale: float = 3.5, prog_bar=True):
    """Regenerate from xts[Tskip] with the extracted noise maps zs[Tskip:] (batched: 5-D xts / zs -> (B,C,H,W))."""
    x0, _ = inversion_reverse_process(model, xT=xts[Tskip], eta=eta, zs=zs[Tskip:], prompt=prompt,
                                      cfg_scale=cfg_scale, prog_bar=prog_bar)
    return x0[None] if x0.dim() < 4 else x0
