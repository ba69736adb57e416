"""Batched real-image editing on the device: B images inverted, parsed, masked and edited in one call equal B
single-image calls.  The noise predictor is teacher-forced (recorded eps replayed, per image stacked) wherever the
comparison is bit for bit."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import loops
from test_gpu_pipeline import make_model, osched

pytestmark = pytest.mark.gpu
T_ = torch.from_numpy


def _batch_inputs(g, preset, B, T, seed):
    """Image 0 = the golden x0, the others perturbed copies; per-image forward noise and eps."""
    gen = torch.Generator().manual_seed(seed)
    x0 = T_(g[f"{preset}/x0"])[0]
    x0s = torch.stack([x0] + [(x0 + 0.3 * torch.randn(x0.shape, generator=gen)).clamp(-1, 1) for _ in range(B - 1)])
    noise = torch.randn((T, B) + tuple(x0.shape), generator=gen)
    noise[:, 0] = T_(g[f"{preset}/fwd_noises"])
    return x0s, noise, gen


def _eq(a, b):
    return np.array_equal(a.cpu().numpy(), b.cpu().numpy(), equal_nan=True)


@pytest.mark.parametrize("preset", ["ddpm", "sd"])
@pytest.mark.parametrize("B", [1, 3])
def test_teacher_forced_inversion_and_regeneration_equal_single_image_calls(golden, preset, B):
    import ddim_inversion as di
    import ddpm_inversion as dp
    g = golden("inversion")
    T = int(g["T"])
    x0s, noise, gen = _batch_inputs(g, preset, B, T, seed=10 + B)
    shape = tuple(x0s.shape[1:])
    for eta in (1.0, 0.6):
        eps = torch.randn((T, B) + shape, generator=gen)
        eps[:, 0] = T_(g[f"{preset}/eta{eta}/inv_eps"])
        xT, zs, xts = dp.invert(make_model(eps.numpy(), preset, T, clip=False), x0s.cuda(), num_inference_steps=T,
                                eta=eta, prog_bar=False, noise=noise.cuda() if B > 1 else noise[:, 0].cuda())
        if B > 1:
            assert xT.shape == (B,) + shape and zs.shape == (T, B) + shape and xts.shape == (T + 1, B) + shape
        else:
            assert xT.shape == (1,) + shape and zs.shape == (T,) + shape and xts.shape == (T + 1,) + shape
            zs, xts = zs[:, None], xts[:, None]
        for b in range(B):
            xT1, zs1, xts1 = dp.invert(make_model(eps[:, b].numpy(), preset, T, clip=False), x0s[b].cuda(),
                                       num_inference_steps=T, eta=eta, prog_bar=False, noise=noise[:, b].cuda())
            assert _eq(xT[b], xT1[0]) and _eq(zs[:, b], zs1) and _eq(xts[:, b], xts1), (eta, b)
            rep = iter(eps[:, b])
            _, ozs, oxts = loops.invert_ddpm(osched(preset, T, False), lambda x, t: next(rep)[None], x0s[b][None],
                                             noise[:, b], eta)
            assert _eq(zs[:, b], ozs) and _eq(xts[:, b], oxts), (eta, b)
        for tskip in (0, 7):
            seps = torch.randn((T - tskip, B) + shape, generator=gen)
            xr = dp.sample(make_model(seps.numpy(), preset, T, clip=False), zs if B > 1 else zs[:, 0],
                           xts if B > 1 else xts[:, 0], Tskip=tskip, eta=eta, prog_bar=False)
            assert xr.shape == (B,) + shape
            for b in range(B):
                xr1 = dp.sample(make_model(seps[:, b].numpy(), preset, T, clip=False), zs[:, b], xts[:, b], Tskip=tskip,
                                eta=eta, prog_bar=False)
                assert _eq(xr[b], xr1[0]), (eta, tskip, b)
    deps = torch.randn((T, B) + shape, generator=gen)
    xd = di.ddim_inversion(make_model(deps.numpy(), preset, T, clip=False), x0s.cuda())
    for b in range(B):
        assert _eq(xd[b], di.ddim_inversion(make_model(deps[:, b].numpy(), preset, T, clip=False), x0s[b:b + 1].cuda())[0])


@pytest.mark.parametrize("B", [1, 3])
def test_teacher_forced_batched_edit_equals_single_image_edits(golden, B):
    import ddpm_inversion as dp
    from attr_functions import SingleColorAttrFunc
    from diffusion_classes import DDPM
    from SegDiffEditPipeline import SegDiffEditPipeline
    g = golden("inversion")
    T, tskip = int(g["T"]), 7
    x0s, noise, gen = _batch_inputs(g, "ddpm", B, T, seed=30 + B)
    shape = tuple(x0s.shape[1:])
    eps = torch.randn((T, B) + shape, generator=gen)
    _, zs, xts = dp.invert(make_model(eps.numpy(), "ddpm", T, clip=False), x0s.cuda(), num_inference_steps=T, eta=1.0,
                           prog_bar=False, noise=noise.cuda() if B > 1 else noise[:, 0].cuda())
    if B == 1:
        zs, xts = zs[:, None], xts[:, None]
    mask = (torch.rand((B,) + shape, generator=gen) > 0.5).float().cuda()
    geps = torch.randn((T - tskip, B) + shape, generator=gen)

    def edit(e, z, x, m):
        f = SingleColorAttrFunc(target=0.6, color_idx=1, loss_scale=50.0, per_sample=True, use_mask=True, mask_attr_grad=True)
        pipe = SegDiffEditPipeline(DDPM(make_model(e.numpy(), "ddpm", T, clip=False)), None)
        return pipe.edit_image(xt=x[0], eta=1.0, zs=z, xts=x, mask=m, attr_func=f, Tskip=tskip, inversion_method="ddpm",
                               prog_bar=False, output_type="tensor")

    full = edit(geps, zs, xts, mask)
    assert full.imgs.shape == (B,) + shape
    for b in range(B):
        one = edit(geps[:, b], zs[:, b], xts[:, b], mask[b:b + 1])
        assert torch.equal(full.imgs[b], one.imgs[0]), b
        assert all(torch.equal(h[b], h1[0]) for h, h1 in zip(full.pred_original_samples, one.pred_original_samples))
    # noise resynthesis draws maps of their own shape: (B, C, H, W) and (T', B, C, H, W)
    pipe = SegDiffEditPipeline(DDPM(make_model(geps.numpy(), "ddpm", T, clip=False)), None)
    xt2, zs2 = pipe.edit_noise_maps(xts[tskip], zs[tskip:], mask, True)
    assert xt2.shape == (B,) + shape and zs2.shape == (T - tskip, B) + shape
    keep = mask == 0
    assert torch.equal(xt2[keep], xts[tskip][keep]) and torch.equal(zs2[:, keep], zs[tskip:, keep])
    assert not torch.equal(zs2[:, ~keep], zs[tskip:, ~keep])


def test_batched_inversion_round_trip_ddpm256():
    """test_gpu_pipeline's round trip for a batch of 4 at DDPM-256: regenerating from xts[0] with the extracted zs and
    the recorded predictions reproduces every xts[k] of every image."""
    import ddpm_inversion as dp
    from b200edit.scheduler import DDIMScheduler
    from oracle.unet2d import ToyEpsModel
    s = DDIMScheduler.from_preset("ddpm", clip_sample=False)
    s.set_timesteps(50)
    toy = ToyEpsModel(3, 256).cuda()
    rec = []

    class Recorder:
        config, in_channels, sample_size, device = toy.config, 3, 256, torch.device("cuda")

        def __call__(self, sample, timestep, **_):
            out = toy(sample, timestep)
            rec.append(out["sample"].detach().clone())
            return out

    model = SimpleNamespace(unet=Recorder(), scheduler=s, device=torch.device("cuda"))
    x0 = (torch.randn(4, 3, 256, 256, generator=torch.Generator().manual_seed(7)) * 0.5).clamp(-1, 1).cuda()
    xT, zs, xts = dp.invert(model, x0, num_inference_steps=50, eta=1, prog_bar=False)
    assert len(rec) == 50 and rec[0].shape == (4, 3, 256, 256)
    assert torch.isfinite(zs).all() and torch.isfinite(xts[:50]).all()
    assert torch.equal(xT, xts[0]) and float(zs[-1].abs().max()) == 0.0
    eps_by_idx = rec[::-1]
    xt = xts[0]
    worst = [0.0] * 4
    for idx, t in enumerate([int(t) for t in s.timesteps][:-1]):
        xt = dp.reverse_step(model, eps_by_idx[idx], t, xt, eta=1, variance_noise=zs[idx])
        for b in range(4):
            ref = xts[idx + 1, b]
            worst[b] = max(worst[b], (xt[b] - ref).abs().max().item() / max(1.0, ref.abs().max().item()))
    print(f"batched round trip, worst relative deviation per image: {['%.3e' % w for w in worst]}")
    assert max(worst) < 5e-4


@pytest.fixture(scope="module")
def parsers():
    from b200edit.bisenet import BiSeNet
    out = {}
    for precision in ("fp16", "fp32"):
        for S in (256, 512):
            out[(precision, S)] = BiSeNet(19, S, max_batch=4, precision=precision).init_random(3)
    return out


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
@pytest.mark.parametrize("S", [256, 512])
@pytest.mark.parametrize("B", [1, 3, 8])
def test_parser_labels_equal_the_argmax_of_the_logits(parsers, precision, S, B):
    net = parsers[(precision, S)]
    x = torch.randn(B, 3, S, S, generator=torch.Generator().manual_seed(B * S)).cuda()
    labels = net.labels(x)
    assert labels.shape == (B, S, S) and labels.dtype == torch.int64
    ref = net(x)[0].argmax(1)
    assert torch.equal(labels, ref)
    assert len(torch.unique(ref)) > 1


def _taps(n_in, n_out):
    s = np.float32((n_in - 1) / (n_out - 1))
    f = (s * np.arange(n_out, dtype=np.float32)).astype(np.float32)
    i0 = f.astype(np.int64)
    return i0, np.where(i0 < n_in - 1, i0 + 1, i0), f - i0


@pytest.mark.parametrize("planes", [1, 3])
def test_bilinear_argmax_ties_and_nan(planes):
    """Ties keep the first maximum; a NaN anywhere in a pixel's taps makes that channel (the first NaN one) the label,
    as torch.argmax does on the logits."""
    from b200edit import ops
    Hi, P, K, S = 5, 8, 6, 9
    gen = torch.Generator().manual_seed(5)
    hi = torch.randint(-10, 10, (1, Hi, Hi, P), generator=gen).float()
    lo = torch.zeros_like(hi)
    hi[..., 2] = hi[..., 4] = 1000.0             # tie between channels 2 and 4 -> 2
    hi[..., 6:] = 5000.0                        # channels >= K do not count
    expect = np.full((S, S), 2)
    lo4 = np.where(np.arange(Hi) < 2, 0.5, 0.125)
    if planes == 3:                              # the lo plane decides: channel 4 wins where its lo is larger
        lo[..., 2] = 0.25
        lo[..., 4] = torch.from_numpy(lo4).float()[None, :, None]
    hi[0, 1, 1, 5] = float("nan")
    hi[0, 3, 3, 3] = hi[0, 3, 3, 1] = float("nan")
    h0, h1, lh = _taps(Hi, S)
    for oy in range(S):
        for ox in range(S):
            rows, cols = {h0[oy], h1[oy]}, {h0[ox], h1[ox]}
            if planes == 3:
                # channel 4's interpolated lo against channel 2's 0.25 (never equal at these weights)
                expect[oy, ox] = 4 if (1 - lh[oy]) * lo4[h0[oy]] + lh[oy] * lo4[h1[oy]] > 0.25 else 2
            if 3 in rows and 3 in cols:
                expect[oy, ox] = 1
            elif 1 in rows and 1 in cols:
                expect[oy, ox] = 5
    x = torch.cat([hi, lo, hi], -1) if planes == 3 else hi
    got = ops.bilinear_argmax(x.to(ops.act_dtype()).cuda(), K, S, planes=planes)
    assert got.shape == (1, S, S)
    assert np.array_equal(got[0].cpu().numpy(), expect)


def test_segmentation_model_batch_and_stale_gradient():
    from b200edit._C import B2EError
    from b200edit.bisenet import BiSeNet
    from models import SegmentationModel
    seg = SegmentationModel(seed=4)
    imgs = torch.rand(3, 3, 256, 256, generator=torch.Generator().manual_seed(9)).cuda() * 2 - 1
    maps = seg(imgs)
    assert maps.shape == (3, 512, 512) and maps.dtype == torch.int64
    for b in range(3):
        assert torch.equal(maps[b], seg(imgs[b:b + 1]))
    # a caller-supplied torch network gets argmax(1)
    conv = torch.nn.Conv2d(3, 19, 1).cuda()
    mine = SegmentationModel(net=lambda x: (conv(x),))
    with torch.no_grad():
        assert torch.equal(mine(imgs), conv(mine.process(imgs)).argmax(1))
    # labels overwrite the activations: the gradient of an earlier kept forward is refused
    net = BiSeNet(19, 128, max_batch=2).init_random(1).enable_grad()
    x = torch.randn(2, 3, 128, 128).cuda()
    y = net.forward_keep(x)
    net.labels(x)
    with pytest.raises(B2EError, match="another forward"):
        net.input_grad(torch.ones_like(y))


def test_batched_masks_equal_single_map_calls_and_goldens(golden):
    from b200edit import ops
    from mask_creator import MaskCreator
    g = golden("mask")
    names = sorted({str(k).split("/")[0] for k in g["keys"]})
    rng = np.random.RandomState(3)
    rand = [np.kron(rng.randint(0, 19, size=(65, 65)), np.ones((8, 8), dtype=np.int64))[:512, :512] for _ in range(3)]
    stack = torch.from_numpy(np.stack([g[f"seg/{n}"].astype(np.int64) for n in names] + rand)).cuda()
    n = 0
    for k in g["keys"]:
        name, cls, d, dil = str(k).split("/")
        classes, d = [int(c) for c in cls[1:].split("_")], int(d[1:])
        got = ops.mask_from_seg(stack, classes, dil == "dil1", (d, d))
        assert got.shape == (len(stack), 3, d, d)
        for i in range(len(stack)):
            assert torch.equal(got[i:i + 1], ops.mask_from_seg(stack[i], classes, dil == "dil1", (d, d))), (k, i)
        ref = np.unpackbits(g["mask/" + str(k)])[: d * d].reshape(d, d).astype(np.float32)
        for c in range(3):
            assert np.array_equal(got[names.index(name), c].cpu().numpy(), ref), k
        n += 1
    assert n == 60
    for classes in ([3], [1, 2, 17], [5, 5, 6], []):
        m = MaskCreator(dilate_mask=True, resize_size=(48, 40)).create_mask(stack, classes, channels=4)
        assert m.shape == (len(stack), 4, 48, 40)
        for i in range(len(stack)):
            assert torch.equal(m[i:i + 1], ops.mask_from_seg(stack[i], classes, True, (48, 40), channels=4))


def _native(family):
    from models import create_diffusion_model
    if family == "ddpm":
        cfg = dict(sample_size=32, in_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1,
                   down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"))
        return create_diffusion_model("ddpm", sample_clipping=False, max_batch=4, seed=1, unet_config=cfg), None
    if family == "ldm":
        cfg = dict(sample_size=16, in_channels=3, out_channels=3, block_out_channels=(32, 96), layers_per_block=1,
                   down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"),
                   attention_head_dim=32, flip_sin_to_cos=True, freq_shift=0, downsample_padding=1)
        vq = dict(latent_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1, norm_num_groups=32,
                  norm_eps=1e-6, num_vq_embeddings=64, sample_size=16)
        return create_diffusion_model("ldm", sample_clipping=False, max_batch=4, seed=2, unet_config=cfg, vq_config=vq), None
    from test_gpu_unet_cond import SMALL, FakeTextEncoder, FakeTokenizer
    vq = dict(latent_channels=4, out_channels=3, block_out_channels=(64, 128), layers_per_block=1, norm_num_groups=32,
              norm_eps=1e-6, sample_size=16)
    w = create_diffusion_model("sd", sample_clipping=False, max_batch=4, seed=5, unet_config=SMALL, vq_config=vq,
                               tokenizer=FakeTokenizer(), text_encoder=FakeTextEncoder(64).cuda())
    return w, "a face"


def _close(a, b):
    return bool(((a - b).abs() <= 1e-2 * torch.clamp(b.abs(), min=1.0)).all())


@pytest.mark.parametrize("family", ["ddpm", "ldm", "sd"])
def test_native_real_image_edit_of_a_batch(family, monkeypatch):
    from attr_functions import SingleColorAttrFunc
    from models import SegmentationModel
    from SegDiffEditPipeline import SegDiffEditPipeline
    w, prompt = _native(family)
    T, tskip, B = 10, 4, 3
    w.scheduler.set_timesteps(T)
    pipe = SegDiffEditPipeline(w, SegmentationModel(seed=2, max_batch=4))
    imgs = (torch.rand(B, 3, 32, 32, generator=torch.Generator().manual_seed(6)) * 2 - 1).cuda()
    seg0 = pipe.segmentation_model(imgs[:1])
    cls = [int(torch.mode(seg0.flatten()).values)]             # a class the random parser does produce
    kw = dict(eta=1.0, inversion_method="ddpm", classes=cls, prompt=prompt, cfg_scale=3.5 if prompt else None,
              prog_bar=False)
    # the inversion's forward noise: image b's draw at the k-th call depends on (k, b) only, so that a batched run and
    # the single-image runs see the same noise per image
    state = {}
    real = torch.randn_like

    def randn_like(x, **_):
        k = state["k"] = state["k"] + 1
        return torch.stack([torch.randn(x.shape[1:], generator=torch.Generator().manual_seed(1000 * k + state["b0"] + b))
                            for b in range(x.shape[0])]).to(x.device)

    def run(x, b0=0):
        state.update(k=0, b0=b0)
        monkeypatch.setattr(torch, "randn_like", randn_like)
        try:
            xt, zs, xts, mask, seg = pipe.prepare_real_image_edit(x, **kw)
        finally:
            monkeypatch.setattr(torch, "randn_like", real)
        f = SingleColorAttrFunc(target=0.5, color_idx=0, loss_scale=30.0, per_sample=True, use_mask=True,
                                mask_attr_grad=True)
        out = pipe.edit_image(xt=xt, eta=1.0, zs=zs, xts=xts, mask=mask, attr_func=f, Tskip=tskip, prompt=prompt,
                              cfg_scale=3.5 if prompt else None, inversion_method="ddpm", prog_bar=False,
                              output_type="tensor")
        return xt, zs, xts, mask, seg, out.imgs

    xt, zs, xts, mask, seg, imgs_out = run(imgs)
    C, d = xt.shape[1], w.data_dimensionality
    assert xt.shape == (B, C, d, d) and zs.shape == (T, B, C, d, d) and xts.shape == (T + 1, B, C, d, d)
    assert seg.shape == (B, 512, 512) and mask.shape == (B, C, d, d) and imgs_out.shape == (B, 3, 32, 32)
    assert torch.isfinite(xt).all() and torch.isfinite(zs).all() and torch.isfinite(xts[:T]).all()
    assert torch.isfinite(imgs_out).all()
    latents = w.encode(imgs)
    for b in range(B):
        xt1, _, _, mask1, seg1, img1 = run(imgs[b:b + 1], b0=b)
        if torch.equal(seg[b], seg1):
            assert torch.equal(mask[b], mask1[0]), b
        assert _close(latents[b], w.encode(imgs[b:b + 1])[0]) and _close(xt[b], xt1[0]), b
        assert _close(imgs_out[b], img1[0]), b
