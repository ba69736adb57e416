"""GPU numerics of the native LPIPS (vgg) distance and its input gradient against the oracle restatement of
``lpips.LPIPS(net='vgg')`` (oracle/lpips.py) in fp32 on the GPU (TF32 off) with the same seeded weights, and the
``use_lpips`` guidance: the native path (no autograd) against the generic autograd path through the oracle network.

Bars: fp32-accurate forward - distance relative error <= 2e-4, input gradient relative RMS <= 2e-2 with cosine >= 0.999;
16-bit forward - distance <= 5e-3, gradient <= 0.2 / cosine >= 0.98 and no worse than torch's bf16 autograd + 5e-3."""
import pytest
import torch

pytestmark = pytest.mark.gpu
tv = pytest.importorskip("torchvision")


def rel(a, b):
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()


def cos(a, b):
    return torch.nn.functional.cosine_similarity(a.reshape(1, -1).double(), b.reshape(1, -1).double()).item()


def make_pair(S, B, precision, seed=0):
    from b200edit.lpips import LPIPS, lpips_random_state_dict
    from oracle.lpips import LPIPS as OracleLPIPS
    sd = lpips_random_state_dict(seed)
    net = LPIPS(input_size=S, max_batch=B, precision=precision)
    net.load_state_dict(sd)
    oracle = OracleLPIPS()
    oracle.load_state_dict(sd)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return net, oracle.cuda()


def grads(fn, x0, x1):
    x = x0.clone().requires_grad_(True)
    d = fn(x, x1)
    g, = torch.autograd.grad(d.sum(), x)
    return d.detach().float().reshape(-1), g.float()


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("S,B,RB", [(64, 1, 1), (64, 4, 1), (64, 4, 4), (256, 1, 1), (256, 4, 1), (256, 4, 4), (512, 1, 1),
                                    (512, 4, 1), (512, 4, 4)])
def test_distance_and_input_gradient_vs_oracle(S, B, RB, precision):
    net, oracle = make_pair(S, B, precision, seed=S + B)
    g = torch.Generator().manual_seed(S * 10 + B + RB)
    x0 = (torch.rand(B, 3, S, S, generator=g) * 2 - 1).cuda()
    x1 = (torch.rand(RB, 3, S, S, generator=g) * 2 - 1).cuda()
    dn, gn = grads(net, x0, x1)
    dr, gr = grads(oracle, x0, x1)
    d_err = ((dn - dr).abs() / dr.abs()).max().item()
    tag = f"LPIPS {S}x{S} B={B} ref={RB} [{precision}]"
    assert torch.isfinite(dn).all() and torch.isfinite(gn).all()
    if precision == "fp32":
        print(f"{tag}: distance rel-err {d_err:.3e} | gradient rel-rms {rel(gn, gr):.3e} cos {cos(gn, gr):.6f}")
        assert d_err <= 2e-4
        assert rel(gn, gr) <= 2e-2 and cos(gn, gr) >= 0.999
    else:
        o16 = oracle.bfloat16()
        _, g16 = grads(lambda a, b: o16(a.bfloat16(), b.bfloat16()).float(), x0, x1)
        print(f"{tag}: distance rel-err {d_err:.3e} | gradient rel-rms {rel(gn, gr):.3e} cos {cos(gn, gr):.5f} "
              f"torch-bf16 {rel(g16, gr):.3e} cos {cos(g16, gr):.5f}")
        assert d_err <= 5e-3
        assert rel(gn, gr) <= 0.2 and cos(gn, gr) >= 0.98 and rel(gn, gr) <= rel(g16, gr) + 5e-3


def test_gradient_finite_on_all_zero_tap_pixels():
    """Left half of the image drives every relu1_2 channel to zero (positive conv1_1 weights on a negative input,
    non-positive biases): there the exact Jacobian of the normalisation is I / eps; the ReLU mask removes it before
    any 16-bit store.  (torch's sqrt backward is NaN there, but its ReLU backward is a select that drops it, so the
    oracle's gradient stays finite and is compared everywhere.)"""
    from b200edit.lpips import LPIPS, lpips_random_state_dict
    from oracle.lpips import LPIPS as OracleLPIPS
    sd = lpips_random_state_dict(7)
    sd["net.slice1.0.weight"] = sd["net.slice1.0.weight"].abs()
    for k in list(sd):
        if k.startswith("net.") and k.endswith(".bias"):
            sd[k] = -sd[k].abs()
    S = 64
    net = LPIPS(input_size=S, max_batch=1, precision="fp32")
    net.load_state_dict(sd)
    oracle = OracleLPIPS()
    oracle.load_state_dict(sd)
    oracle = oracle.cuda()
    g = torch.Generator().manual_seed(3)
    x0 = (torch.rand(1, 3, S, S, generator=g) * 2 - 1)
    x0[..., : S // 2] = -1.0
    x0, x1 = x0.cuda(), (torch.rand(1, 3, S, S, generator=g) * 2 - 1).cuda()
    dn, gn = grads(net, x0, x1)
    dr, gr = grads(oracle, x0, x1)
    assert torch.isfinite(gn).all() and torch.isfinite(dn).all()
    assert ((dn - dr).abs() / dr.abs()).max().item() <= 2e-4
    with torch.no_grad():
        tap1 = oracle.net(oracle.scaling_layer(x0))[0]
    zero_px = (tap1.abs().amax(1) == 0).float().mean().item()
    print(f"all-zero tap pixels: {zero_px:.3f} of relu1_2 | gradient rel-rms {rel(gn, gr):.3e} cos {cos(gn, gr):.6f}")
    assert zero_px > 0.3 and torch.isfinite(gr).all()
    assert rel(gn, gr) <= 2e-2 and cos(gn, gr) >= 0.999


def test_two_runs_are_bit_identical_and_stale_backward_raises():
    from b200edit._C import B2EError
    net, _ = make_pair(128, 2, "fp32", seed=5)
    g = torch.Generator().manual_seed(9)
    x0 = (torch.rand(2, 3, 128, 128, generator=g) * 2 - 1).cuda()
    x1 = (torch.rand(1, 3, 128, 128, generator=g) * 2 - 1).cuda()
    d1, g1 = grads(net, x0, x1)
    d2, g2 = grads(net, x0, x1)
    assert torch.equal(d1, d2) and torch.equal(g1, g2)
    x = x0.clone().requires_grad_(True)
    d = net(x, x1)
    net(x0, x1)                                  # another forward overwrites the activations
    with pytest.raises(B2EError):
        torch.autograd.grad(d.sum(), x)
    x1b = x1.clone()
    x1b += 0.5                                    # in-place change of the reference: the cache is recomputed
    dn = net(x0, x1b).reshape(-1)
    dr = net(x0, x1b.clone()).reshape(-1)
    assert torch.equal(dn, dr) and not torch.equal(dn, d1)


def test_new_reference_at_a_reused_address_is_not_mistaken_for_the_cached_one():
    """A metric loop frees each reference before the next one is allocated, typically at the same address with version 0:
    every pair must be scored against its own reference."""
    net, oracle = make_pair(64, 1, "fp32", seed=13)
    g = torch.Generator().manual_seed(6)
    x0 = (torch.rand(1, 3, 64, 64, generator=g) * 2 - 1).cuda()
    for _ in range(3):
        b = (torch.rand(1, 3, 64, 64, generator=g) * 2 - 1).cuda()
        got, want = net(x0, b), oracle(x0, b)
        assert (got - want).abs().max().item() <= 2e-4 * want.abs().max().item()
        del b


def test_one_channel_mask_stays_valid_until_the_backward():
    """A (1, 1, S, S) mask is expanded into a temporary the engine's backward reads (the -mask chain): it must stay
    alive across allocations made between the forward and the backward."""
    net, oracle = make_pair(64, 2, "fp32", seed=17)
    g = torch.Generator().manual_seed(8)
    x0 = (torch.rand(2, 3, 64, 64, generator=g) * 2 - 1).cuda()
    x1 = (torch.rand(1, 3, 64, 64, generator=g) * 2 - 1).cuda()
    m1 = (torch.rand(1, 1, 64, 64, generator=g) > 0.5).float().cuda()
    x = x0.clone().requires_grad_(True)
    d = net(x, x1, mask=(m1 > 0.5).float())               # caller-side temporary, expanded to 3 channels inside
    junk = [torch.full((1 << 20,), 7.0, device="cuda") for _ in range(8)]
    gn, = torch.autograd.grad(d.sum(), x)
    del junk
    xr = x0.clone().requires_grad_(True)
    dr = oracle(1 - m1 * xr, x1)
    gr, = torch.autograd.grad(dr.sum(), xr)
    print(f"1-channel mask: distance rel-err {((d.detach() - dr.detach()).abs() / dr.abs()).max().item():.3e} | "
          f"gradient rel-rms {rel(gn, gr):.3e} cos {cos(gn, gr):.6f}")
    assert ((d.detach() - dr.detach()).abs() / dr.abs()).max().item() <= 2e-4
    assert rel(gn, gr) <= 2e-2 and cos(gn, gr) >= 0.999


def test_metric_with_model():
    import metrics
    net, oracle = make_pair(64, 2, "fp32", seed=11)
    g = torch.Generator().manual_seed(4)
    a, b = [(torch.rand(2, 3, 64, 64, generator=g) * 2 - 1).cuda() for _ in range(2)]
    got = metrics.lpips(a, b, model=net)
    want = oracle(a, b)
    assert got.shape == (2, 1, 1, 1)
    assert ((got - want).abs() / want.abs()).max().item() <= 2e-4


def _guidance_case(name, mask_c=3, B=1):
    from b200edit.lpips import lpips_random_state_dict
    from models import create_diffusion_model, get_lpips
    from oracle.lpips import LPIPS as OracleLPIPS
    if name == "ddpm":
        cfg = dict(sample_size=32, in_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1,
                   down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"))
        w = create_diffusion_model("ddpm", sample_clipping=True, max_batch=B, seed=1, unet_config=cfg)
        S, lat = 32, 32
    else:
        cfg = dict(sample_size=16, in_channels=3, out_channels=3, block_out_channels=(32, 96), layers_per_block=1,
                   down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"),
                   attention_head_dim=32, flip_sin_to_cos=True, freq_shift=0, downsample_padding=1)
        vq = dict(latent_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1, norm_num_groups=32,
                  norm_eps=1e-6, num_vq_embeddings=256, sample_size=16)
        w = create_diffusion_model("ldm", sample_clipping=False, max_batch=1, seed=2, unet_config=cfg, vq_config=vq,
                                   with_encoder=False)
        S, lat = 32, 16
    sd = lpips_random_state_dict(12)
    native = get_lpips(input_size=S, max_batch=B, state_dict=sd)
    oracle = OracleLPIPS()
    oracle.load_state_dict(sd)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator().manual_seed(31)
    mask = (torch.rand(B, mask_c, S, S, generator=g) > 0.4).float().cuda()
    x_0 = (torch.rand(1, 3, S, S, generator=g) * 2 - 1).cuda()
    xt = torch.randn(B, 3, lat, lat, generator=g).cuda()
    return w, native, oracle.cuda(), mask, x_0, xt


@pytest.mark.parametrize("mask_c", [3, 1])
@pytest.mark.parametrize("name", ["ddpm", "ldm"])
def test_use_lpips_native_path_matches_autograd_path(name, mask_c, monkeypatch):
    from attr_functions import MultiColorAttrFunc
    from SegDiffEditPipeline import SegDiffEditPipeline
    w, native, oracle, mask, x_0, xt = _guidance_case(name, mask_c)
    w.scheduler.set_timesteps(6)
    kw = dict(mask_pred_original_sample=True, use_lpips=True, lambda_=0.7, x_0=x_0, mask=mask)
    eps = w.unet(xt, int(w.scheduler.timesteps[2])).sample
    t = int(w.scheduler.timesteps[2])

    def nudge(model):
        f = MultiColorAttrFunc(0.8, 0.2, 0.3, loss_scale=50.0, lpips_model=model, **kw)
        out, _ = f.apply(xt, None, eps, t, 2, w, **kw)
        return out - xt
    ref = nudge(oracle)                                  # generic: autograd through the oracle network
    real_grad = torch.autograd.grad

    def no_autograd(*a, **k):
        raise AssertionError("the native LPIPS guidance path must not call torch.autograd.grad")
    monkeypatch.setattr(torch.autograd, "grad", no_autograd)
    got = nudge(native)
    print(f"use_lpips nudge [{name}, {mask_c}-channel mask]: native vs autograd rel-rms {rel(got, ref):.3e} cos {cos(got, ref):.6f}")
    assert torch.isfinite(got).all() and ref.abs().max() > 0
    assert rel(got, ref) <= 2e-2 and cos(got, ref) >= 0.999
    # the whole edit on the native path
    f = MultiColorAttrFunc(0.8, 0.2, 0.3, loss_scale=50.0, t1=0, t2=6, use_mask=True, mask_pred_original_sample=True,
                           use_lpips=True, lambda_=0.7, x_0=x_0, lpips_model=native)
    out = SegDiffEditPipeline(w, None).edit_image(xt=xt, attr_func=f, prog_bar=False, output_type="tensor", mask=mask)
    assert torch.isfinite(out.imgs).all()
    monkeypatch.setattr(torch.autograd, "grad", real_grad)


def test_use_lpips_native_path_batched():
    """B = 3 with a per-image mask through the native combine kernel, against autograd of the same loss written out
    (colour loss of the masked prediction + lambda_ * sum over the images of the oracle LPIPS; the reference's own
    autograd call accepts only one image here, its loss being (B, 1, 1, 1))."""
    from attr_functions import MultiColorAttrFunc, color_loss
    B = 3
    w, native, oracle, mask, x_0, xt = _guidance_case("ddpm", 3, B)
    w.scheduler.set_timesteps(6)
    t = int(w.scheduler.timesteps[2])
    eps = w.unet(xt, t).sample
    c = w.scheduler.coeffs(t, 0.0, "ddim")
    kw = dict(mask_pred_original_sample=True, use_lpips=True, lambda_=0.7, x_0=x_0, mask=mask)
    f = MultiColorAttrFunc(0.8, 0.2, 0.3, loss_scale=50.0, lpips_model=native, **kw)
    got = f.apply(xt, None, eps, t, 2, w, **kw)[0] - xt
    x = xt.detach().clone().requires_grad_(True)
    pred = (x - c.sqrt_b_t * eps) / c.sqrt_a_t
    loss = 50.0 * (color_loss(mask * pred, 0.8, 0.2, 0.3) + 0.7 * oracle(1 - mask * pred, x_0).sum())
    ref = -torch.autograd.grad(loss, x)[0] * c.a_t_sq
    for b in range(B):
        print(f"use_lpips nudge [ddpm, B={B}, image {b}]: rel-rms {rel(got[b], ref[b]):.3e} cos {cos(got[b], ref[b]):.6f}")
        assert rel(got[b], ref[b]) <= 2e-2 and cos(got[b], ref[b]) >= 0.999
