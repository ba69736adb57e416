"""CPU tests of the batched real-image editing path: the shape and argument validation that runs before any device
call (batch against the noise predictor's max_batch, injected noise shape, 5-D xts / zs pairing, mask batch)."""
from types import SimpleNamespace

import pytest
import torch


def _model(max_batch=None, T=10):
    from b200edit.scheduler import DDIMScheduler
    s = DDIMScheduler.from_preset("ddpm", clip_sample=False)
    s.set_timesteps(T)
    unet = SimpleNamespace(config=SimpleNamespace(in_channels=3, sample_size=8))
    if max_batch is not None:
        unet.max_batch = max_batch
    return SimpleNamespace(unet=unet, scheduler=s, device=torch.device("cpu"))


def test_batch_above_the_predictors_max_batch_raises():
    import ddpm_inversion as dp
    dp.check_batch(_model(4), 4, cfg=False)
    dp.check_batch(_model(4), 2, cfg=True)
    dp.check_batch(_model(1), 1, cfg=True)             # batch 1 keeps the reference's path unchecked
    dp.check_batch(_model(None), 64, cfg=True)         # a predictor without max_batch (a torch module) is not limited
    with pytest.raises(ValueError, match="max_batch 4"):
        dp.check_batch(_model(4), 5, cfg=False)
    with pytest.raises(ValueError, match="classifier-free guidance"):
        dp.check_batch(_model(4), 3, cfg=True)
    with pytest.raises(ValueError, match="max_batch"):
        dp.invert(_model(2), torch.zeros(3, 3, 8, 8), num_inference_steps=10, eta=1.0, prog_bar=False)
    with pytest.raises(ValueError, match="max_batch"):
        dp.inversion_reverse_process(_model(2), torch.zeros(3, 3, 8, 8), eta=1.0, zs=torch.zeros(4, 3, 3, 8, 8))


def test_wrong_injected_noise_shape_raises():
    import ddpm_inversion as dp
    m = _model(8)
    x0 = torch.zeros(3, 3, 8, 8)
    for bad in (torch.zeros(10, 3, 8, 8), torch.zeros(10, 2, 3, 8, 8), torch.zeros(9, 3, 3, 8, 8)):
        with pytest.raises(ValueError, match=r"noise must be \(T, B, C, H, W\)"):
            dp.sample_xts_from_x0(m, x0, num_inference_steps=10, noise=bad)
        with pytest.raises(ValueError, match="noise must be"):
            dp.invert(m, x0, num_inference_steps=10, eta=1.0, prog_bar=False, noise=bad)


def test_regeneration_zs_must_match_the_batch():
    import ddpm_inversion as dp
    with pytest.raises(ValueError, match="does not match the batch"):
        dp.sample(_model(8), torch.zeros(4, 2, 3, 8, 8), torch.zeros(5, 3, 3, 8, 8), Tskip=1, prog_bar=False)


def test_pipeline_batch_validation():
    from diffusion_classes import DDPM
    from SegDiffEditPipeline import SegDiffEditPipeline
    m = _model(4)
    pipe = SegDiffEditPipeline(DDPM(m), None)
    xts, zs = torch.zeros(11, 3, 3, 8, 8), torch.zeros(10, 3, 3, 8, 8)
    with pytest.raises(ValueError, match="needs zs of shape"):
        pipe.edit_image(xt=xts[0], eta=1.0, zs=zs[:, 0], xts=xts, Tskip=2, mask=torch.ones(1, 3, 8, 8), resynthesize=False)
    with pytest.raises(ValueError, match="needs zs of shape"):
        pipe.edit_image(xt=xts[0], eta=1.0, zs=zs[:, :2], xts=xts, Tskip=2, mask=torch.ones(1, 3, 8, 8), resynthesize=False)
    with pytest.raises(ValueError, match="mask batch must be 1 or the image batch 3"):
        pipe.edit_image(xt=xts[0], eta=1.0, zs=zs, xts=xts, Tskip=2, mask=torch.ones(2, 3, 8, 8), resynthesize=False)
    with pytest.raises(ValueError, match="mask batch must be 1 or the image batch 3"):
        pipe.edit_image(xt=torch.zeros(3, 3, 8, 8), eta=0, mask=torch.ones(2, 3, 8, 8), resynthesize=False)
    with pytest.raises(ValueError, match="max_batch 4"):
        pipe.prepare_real_image_edit(torch.zeros(5, 3, 8, 8), eta=1.0, inversion_method="ddpm", prog_bar=False)
