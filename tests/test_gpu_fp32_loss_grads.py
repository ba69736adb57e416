"""fp32-accurate backward of the loss networks (``grad_precision="fp32"``): the ResNet attribute predictor, the BiSeNet face
parser and LPIPS-VGG differentiate on split operands - split hi + lo gradients through split dgrad weights, every
element-wise backward kernel in fp32 - against float64.

Bars.  Every error is the relative RMS of the input gradient against autograd through the same network in float64 on the
CPU (torchvision / oracle modules, BatchNorm folded the same way), on the same inputs:

  A   rel-rms <= max(1e-4, 3 e32), e32 = torch float32 autograd's own distance from float64, measured in the same test.
      Why 3x: the split forward is 3-4x further from float64 than torch fp32 (DESIGN §2); ReLU / max-pool masks that
      flip scale with the square root of that distance (<= 2x), and the rest is margin for the backward's own rounding.
  B   rel-rms <= 0.25 x the error of the same network with grad_precision=None (the 16-bit backward) on the same inputs:
      the feature must measurably improve on the default.
  C   rel-rms <= the 16-bit backward's error on the same inputs (never worse than the default).

A and B hold where the 16-bit backward's rounding is what separates the engine from float64 - the ResNet-18 case, 1.0e-3
-> 1.4e-5 on a B200.  For ResNet-50, BiSeNet and LPIPS the split backward removes that rounding too, but the error left is
not the backward's (DESIGN §7: LPIPS's is concentrated in a few pixels, the trace of single ReLU masks that the split
forward and float64 set differently; BiSeNet's is spread evenly and does not move with the backward's precision).  Those
cases are held to C, with A / B printed beside it.

The forward of a grad_precision="fp32" engine is bit-identical to a grad_precision=None engine with the same weights, and
two input_grad calls give identical bits.  Guided updates (the native paths, torch.autograd.grad trapped) against the
reference procedure AttrFunc._apply_autograd through float64 networks: max |diff| <= max(1e-4, 3 e32) max |update|, with
e32 the same chain through float32 networks.  Every check prints its measured value beside its bar."""
from types import SimpleNamespace

import pytest
import torch

from oracle.bisenet import BiSeNet as OracleBiSeNet, seeded_weights

pytestmark = pytest.mark.gpu
tv = pytest.importorskip("torchvision")


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()


def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


def _cpu_grad(fn, x, w):
    x = x.clone().requires_grad_(True)
    (g,) = torch.autograd.grad((fn(x) * w).sum(), x)
    return g


def _check(tag, g_new, g_now, g32, g64, fp32_bar):
    """fp32_bar: assert bars A and B; otherwise bar C (A and B printed)."""
    e_new, e_now, e32 = rel(g_new, g64), rel(g_now, g64), rel(g32, g64)
    bar_a = max(1e-4, 3 * e32)
    print(f"{tag}: grad_precision='fp32' rel-rms {e_new:.3e} | bar A {bar_a:.3e} (torch fp32 {e32:.3e}) | bar B "
          f"{0.25 * e_now:.3e} | bar C {e_now:.3e} (16-bit backward) | asserted: {'A, B' if fp32_bar else 'C'}")
    assert torch.isfinite(g_new).all() and g64.abs().max() > 0
    if fp32_bar:
        assert e_new <= bar_a, (tag, e_new, bar_a)
        assert e_new <= 0.25 * e_now, (tag, e_new, e_now)
    else:
        assert e_new <= e_now, (tag, e_new, e_now)


# ------------------------------------------------------------------ 1. input gradient against float64 autograd
def make_resnet_reference(kind, num_classes, seed):
    torch.manual_seed(seed)
    net = (tv.models.resnet50 if kind == "resnet50" else tv.models.resnet18)()
    net.fc = torch.nn.Linear(net.fc.in_features, num_classes)
    g = torch.Generator().manual_seed(seed + 1)
    for mod in net.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):   # a trained network's statistics are not (0, 1)
            mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
            mod.running_var.copy_(torch.rand(mod.num_features, generator=g) * 0.5 + 0.75)
            mod.weight.data.copy_(torch.rand(mod.num_features, generator=g) * 0.5 + 0.75)
            mod.bias.data.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
    return net.eval()


def _resnet(kind, K, S, B, ref, grad_precision):
    from b200edit.resnet import ResNet
    net = ResNet("bottleneck" if kind == "resnet50" else "basic", (3, 4, 6, 3) if kind == "resnet50" else (2, 2, 2, 2), K, S,
                 max_batch=B, precision="fp32", grad_precision=grad_precision)
    net.load_torchvision_state_dict(ref.state_dict())
    return net


@pytest.mark.parametrize("kind,S,B,K,seed", [("resnet18", 64, 2, 16, 1), ("resnet50", 256, 2, 80, 2), ("resnet50", 512, 1, 80, 3)])
def test_resnet_input_gradient_matches_float64(kind, S, B, K, seed):
    ref = make_resnet_reference(kind, K, seed)
    g = torch.Generator().manual_seed(seed + 2)
    x = torch.rand(B, 3, S, S, generator=g) * 2 - 1
    w = torch.randn(B, K, generator=g)
    grads = []
    for gp in ("fp32", None):
        net = _resnet(kind, K, S, B, ref, gp)
        net.forward_keep(x.cuda())
        grads.append(net.input_grad(w.cuda()).cpu())
        del net
    g32 = _cpu_grad(ref, x, w)
    g64 = _cpu_grad(ref.double(), x.double(), w.double())
    _check(f"{kind} {S}x{S} B={B}", grads[0], grads[1], g32, g64, fp32_bar=kind == "resnet18")


def _bisenet_oracle(seed):
    o = seeded_weights(OracleBiSeNet(19).eval(), seed)
    o.conv_out.conv_out.weight.data.mul_(0.02)   # logits of O(1): an unsaturated softmax, as a trained parser has
    return o


@pytest.mark.parametrize("S", [128, 256])
def test_bisenet_input_gradient_matches_float64(S):
    from b200edit.bisenet import MultiResBiSeNet
    B, seed = 2, 7
    o = _bisenet_oracle(seed)
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, 3, S, S, generator=g)
    w = torch.randn(B, 19, S, S, generator=g)
    grads = []
    for gp in ("fp32", None):
        m = MultiResBiSeNet(19, max_batch=B, grad_precision=gp)
        m.load_reference_state_dict(o.state_dict())
        e = m.engine(S, grad=True)
        assert e.grad_precision == gp and e.precision == "fp32"
        e.forward_keep(x.cuda())
        grads.append(e.input_grad(w.cuda()).cpu())
        del m, e
    g32 = _cpu_grad(lambda t: o(t)[0], x, w)
    o64 = o.double()
    g64 = _cpu_grad(lambda t: o64(t)[0], x.double(), w.double())
    _check(f"bisenet {S}x{S} B={B}", grads[0], grads[1], g32, g64, fp32_bar=False)


def _lpips_pair(S, B, seed, grad_precision):
    from b200edit.lpips import LPIPS, lpips_random_state_dict
    sd = lpips_random_state_dict(seed)
    net = LPIPS(input_size=S, max_batch=B, precision="fp32", grad_precision=grad_precision)
    net.load_state_dict(sd)
    return net, sd


@pytest.mark.parametrize("S,RB,masked", [(64, 1, True), (64, 2, False), (256, 1, False), (256, 2, True)])
def test_lpips_input_gradient_matches_float64(S, RB, masked):
    from oracle.lpips import LPIPS as OracleLPIPS
    B, seed = 2, S + RB
    g = torch.Generator().manual_seed(seed + 1)
    x0 = torch.rand(B, 3, S, S, generator=g) * 2 - 1
    x1 = torch.rand(RB, 3, S, S, generator=g) * 2 - 1
    mask = (torch.rand(B, 3, S, S, generator=g) > 0.4).float() if masked else None
    wd = torch.rand(B, generator=g) + 0.5
    grads = []
    for gp in ("fp32", None):
        net, sd = _lpips_pair(S, B, seed, gp)
        net(x0.cuda(), x1.cuda(), mask=None if mask is None else mask.cuda())
        grads.append(net.input_grad(wd.cuda()).cpu())
        del net
    o = OracleLPIPS()
    o.load_state_dict(sd)
    fn = (lambda m: (lambda t: m(t if mask is None else 1 - mask.to(t.dtype) * t, x1.to(t.dtype)).reshape(-1)))
    g32 = _cpu_grad(fn(o), x0, wd)
    g64 = _cpu_grad(fn(o.double()), x0.double(), wd.double())
    _check(f"lpips {S}x{S} B={B} ref={RB} mask={masked}", grads[0], grads[1], g32, g64, fp32_bar=False)


# ------------------------------------------------------------------ 2. the forward is unchanged, the backward deterministic
def test_forward_is_bit_identical_and_backward_deterministic():
    from b200edit.bisenet import MultiResBiSeNet
    g = torch.Generator().manual_seed(41)
    ref = make_resnet_reference("resnet50", 80, 4)
    x = (torch.rand(2, 3, 128, 128, generator=g) * 2 - 1).cuda()
    d = torch.randn(2, 80, generator=g).cuda()
    a, b = _resnet("resnet50", 80, 128, 2, ref, "fp32"), _resnet("resnet50", 80, 128, 2, ref, None)
    la, lb = a.forward_keep(x), b(x)
    g1 = a.input_grad(d)
    a.forward_keep(x)
    g2 = a.input_grad(d)
    print(f"resnet50 128x128: logits max|diff| {(la - lb).abs().max().item():.1e} (bar 0); two input_grad calls max|diff| "
          f"{(g1 - g2).abs().max().item():.1e} (bar 0)")
    assert torch.equal(la, lb) and torch.equal(g1, g2)

    o = _bisenet_oracle(42)
    ms = [MultiResBiSeNet(19, max_batch=2, grad_precision=gp).load_reference_state_dict(o.state_dict()) for gp in ("fp32", None)]
    x = torch.randn(2, 3, 128, 128, generator=g).cuda()
    e0, e1 = ms[0].engine(128, grad=True), ms[1].engine(128, grad=True)
    la, lb = e0.forward_keep(x), e1.forward_keep(x)
    d = torch.randn_like(la)
    g1 = e0.input_grad(d)
    e0.forward_keep(x)
    g2 = e0.input_grad(d)
    assert ms[0].engine(128).grad_precision is None          # the forward-only label engine is untouched
    assert torch.equal(ms[0].labels(x), ms[1].labels(x))
    print(f"bisenet 128x128: logits max|diff| {(la - lb).abs().max().item():.1e} (bar 0); two input_grad calls max|diff| "
          f"{(g1 - g2).abs().max().item():.1e} (bar 0)")
    assert torch.equal(la, lb) and torch.equal(g1, g2)

    (na, _), (nb, _) = _lpips_pair(64, 2, 5, "fp32"), _lpips_pair(64, 2, 5, None)
    x0, x1 = (torch.rand(2, 3, 64, 64, generator=g) * 2 - 1).cuda(), (torch.rand(1, 3, 64, 64, generator=g) * 2 - 1).cuda()
    da, db = na(x0, x1), nb(x0, x1)
    w = torch.ones(2, device="cuda")
    g1 = na.input_grad(w)
    na(x0, x1)
    g2 = na.input_grad(w)
    print(f"lpips 64x64: distance max|diff| {(da - db).abs().max().item():.1e} (bar 0); two input_grad calls max|diff| "
          f"{(g1 - g2).abs().max().item():.1e} (bar 0)")
    assert torch.equal(da, db) and torch.equal(g1, g2)


# ------------------------------------------------------------------ 3. guided updates against float64 autograd
class _NoAutograd:
    def __enter__(self):
        self.real = torch.autograd.grad

        def no_autograd(*a, **k):
            raise AssertionError("torch.autograd.grad called on the native guidance path")
        torch.autograd.grad = no_autograd

    def __exit__(self, *exc):
        torch.autograd.grad = self.real


def _as(net, dtype):
    """A torch module evaluated in ``dtype`` behind an fp32 interface (autograd flows through the casts)."""
    return lambda *xs: _cast_out(net(*(x.to(dtype) for x in xs)))


def _cast_out(out):
    return tuple(o.float() if torch.is_tensor(o) else o for o in out) if isinstance(out, tuple) else out.float()


def _update_check(tag, dn, d64, d32):
    scale = d64.abs().max().item()
    err, e32 = (dn - d64).abs().max().item() / scale, (d32 - d64).abs().max().item() / scale
    bar = max(1e-4, 3 * e32)
    print(f"{tag}: max|diff| / max|update| = {err:.2e} (bar {bar:.2e}; torch fp32 chain {e32:.2e}; max|update| {scale:.2e})")
    assert scale > 0 and torch.isfinite(dn).all() and err <= bar, (tag, err, bar)


def _ddpm(S, B):
    from models import create_diffusion_model
    cfg = dict(sample_size=S, in_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1,
               down_block_types=("DownBlock2D", "DownBlock2D"), up_block_types=("UpBlock2D", "UpBlock2D"))
    w = create_diffusion_model("ddpm", sample_clipping=False, max_batch=B, seed=1, unet_config=cfg)
    w.scheduler.set_timesteps(10)
    return w


def _updates(make_f, native, refs, w, xt, eps, t, kw=None):
    """(native update with autograd trapped, [update of AttrFunc._apply_autograd through each reference network])"""
    kw = dict(kw or {})
    kw.setdefault("mask", None)
    coeffs = w.scheduler.coeffs(t, 0.0, "ddim")
    with _NoAutograd():
        xn, _ = make_f(native).apply(xt=xt.clone(), zt=None, model_output=eps, timestep=torch.tensor(t), step_idx=0, model=w, **kw)
    outs = []
    for r, model in refs:
        xa, _ = make_f(r)._apply_autograd(xt.clone(), None, eps, coeffs, model, **kw)
        outs.append(xa - xt)
    return xn - xt, outs


def test_classifier_guidance_update_matches_float64():
    from attr_functions import ClassifierAttrFunc
    B, S = 2, 64
    _no_tf32()
    ref = make_resnet_reference("resnet18", 80, 6)
    native = _resnet("resnet18", 80, S, B, ref, "fp32")
    w = _ddpm(S, B)
    g = torch.Generator().manual_seed(61)
    xt, eps = torch.randn(B, 3, S, S, generator=g).cuda(), torch.randn(B, 3, S, S, generator=g).cuda()
    r32 = ref.cuda()
    r64 = make_resnet_reference("resnet18", 80, 6).double().cuda()
    make = lambda p: ClassifierAttrFunc(p, idx_for_class=31, idx_of_interest=0, loss_scale=50.0, per_sample=True)   # noqa: E731
    dn, (d64, d32) = _updates(make, native, [(_as(r64, torch.float64), w), (r32, w)], w, xt, eps, int(w.scheduler.timesteps[5]))
    _update_check("ClassifierAttrFunc(per_sample=True), ResNet-18 64x64, B=2", dn, d64, d32)


def test_net_attr_guidance_update_matches_float64():
    from attr_functions import NetAttrFunc
    from b200edit.bisenet import MultiResBiSeNet
    from models import SegmentationModel
    B, S = 2, 256
    _no_tf32()
    o = _bisenet_oracle(62)
    native = MultiResBiSeNet(19, max_batch=B, grad_precision="fp32").load_reference_state_dict(o.state_dict())
    w = _ddpm(S, B)
    g = torch.Generator().manual_seed(63)
    xt, eps = torch.randn(B, 3, S, S, generator=g).cuda(), torch.randn(B, 3, S, S, generator=g).cuda()
    o32 = o.cuda()
    o64 = _bisenet_oracle(62).double().cuda()

    def make(net):
        return NetAttrFunc(SegmentationModel(net=net, image_size=(S, S)), idx_for_class=[1, 10], loss_scale=1e4, per_sample=True)
    dn, (d64, d32) = _updates(make, native, [(_as(o64, torch.float64), w), (o32, w)], w, xt, eps, int(w.scheduler.timesteps[-1]))
    _update_check("NetAttrFunc(per_sample=True), BiSeNet 256x256, B=2", dn, d64, d32)


def test_lpips_regularised_colour_guidance_update_matches_float64():
    from attr_functions import MultiColorAttrFunc
    from b200edit.lpips import lpips_random_state_dict
    from models import get_lpips
    from oracle.lpips import LPIPS as OracleLPIPS
    S = 64
    _no_tf32()
    sd = lpips_random_state_dict(64)
    native = get_lpips(input_size=S, max_batch=1, state_dict=sd, grad_precision="fp32")
    o32, o64 = OracleLPIPS(), OracleLPIPS()
    o32.load_state_dict(sd)
    o64.load_state_dict(sd)
    o32, o64 = o32.cuda(), o64.double().cuda()
    w = _ddpm(S, 1)
    g = torch.Generator().manual_seed(65)
    xt, eps = torch.randn(1, 3, S, S, generator=g).cuda(), torch.randn(1, 3, S, S, generator=g).cuda()
    mask = (torch.rand(1, 3, S, S, generator=g) > 0.4).float().cuda()
    x_0 = (torch.rand(1, 3, S, S, generator=g) * 2 - 1).cuda()
    # targets outside the image range keep sign(img - target) constant: the colour part of d(loss)/d(image) is exact and
    # the update carries the LPIPS gradient's error (lambda_ large enough for that term to dominate)
    kw = dict(mask_pred_original_sample=True, use_lpips=True, lambda_=50.0, x_0=x_0, mask=mask)
    make = lambda m: MultiColorAttrFunc(40.0, -30.0, 50.0, loss_scale=1.0, lpips_model=m, **kw)   # noqa: E731
    dn, (d64, d32) = _updates(make, native, [(_as(o64, torch.float64), w), (o32, w)], w, xt, eps, int(w.scheduler.timesteps[2]), kw)
    _update_check("use_lpips colour guidance, LPIPS 64x64", dn, d64, d32)


def test_sd_chain_guided_step_on_split_operands_matches_float64():
    """SD chain with precision="fp32", decoder_grad_precision="fp32" and a grad_precision="fp32" predictor: every link
    of the guided step (decoder forward and backward, classifier forward and backward) on split operands."""
    from attr_functions import ClassifierAttrFunc
    from diffusion_classes import SD
    from models import create_diffusion_model
    from oracle.vqmodel import VQModel as OracleVQ
    B = 2
    _no_tf32()
    vcfg = dict(latent_channels=4, out_channels=3, block_out_channels=(64, 64, 128), layers_per_block=1, norm_num_groups=32,
                norm_eps=1e-6, num_vq_embeddings=0, sample_size=16)
    ucfg = dict(sample_size=16, in_channels=4, out_channels=4, block_out_channels=(64, 128), layers_per_block=1,
                cross_attention_dim=64, attention_head_dim=2, norm_num_groups=32, norm_eps=1e-5)
    torch.manual_seed(71)
    odec = OracleVQ(**vcfg).eval()
    sd = odec.state_dict()
    w = create_diffusion_model("sd", sample_clipping=False, max_batch=B, seed=3, unet_config=ucfg,
                               vq_config={k: v for k, v in vcfg.items() if k != "num_vq_embeddings"}, vq_state_dict=sd,
                               precision="fp32", decoder_grad_precision="fp32", with_encoder=False, text_encoder=SimpleNamespace())
    S_img = 64
    ref = make_resnet_reference("resnet50", 80, 7)
    native = _resnet("resnet50", 80, S_img, B, ref, "fp32")
    refs = []
    for dtype in (torch.float64, torch.float32):
        dec = OracleVQ(**vcfg).eval()
        dec.load_state_dict(sd)
        dec = dec.to(dtype).cuda()
        shim = SimpleNamespace(decode=lambda z, d=dec, dt=dtype: SimpleNamespace(sample=d.decode(z.to(dt)).sample.float()))
        w_ref = SD(SimpleNamespace(unet=w.unet, scheduler=w.scheduler, device=torch.device("cuda"), vqvae=shim, vae=shim,
                                   tokenizer=None, text_encoder=None))
        refs.append((_as(make_resnet_reference("resnet50", 80, 7).to(dtype).cuda(), dtype), w_ref))
    g = torch.Generator().manual_seed(72)
    xt = torch.randn(B, 4, 16, 16, generator=g).cuda() * 0.18215
    eps = torch.randn(B, 4, 16, 16, generator=g).cuda() * 0.18215
    w.scheduler.set_timesteps(10)
    make = lambda p: ClassifierAttrFunc(p, idx_for_class=31, idx_of_interest=0, loss_scale=50.0, per_sample=True)   # noqa: E731
    dn, (d64, d32) = _updates(make, native, refs, w, xt, eps, int(w.scheduler.timesteps[-3]))
    _update_check("SD chain (split decoder gradient + split classifier gradient), B=2", dn, d64, d32)
