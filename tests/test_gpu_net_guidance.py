"""GPU: per-sample guidance of the network strategies (``NetAttrFunc`` / ``ClassifierAttrFunc`` with ``per_sample=True``).

* The batched loss heads against the oracle head looped over images, and bit-for-bit batch invariance.
* ``apply`` through the native ResNet-50 / BiSeNet (the kernel-to-kernel path, ``AttrFunc._apply_native_network``) against
  fp32 torch autograd of the reference loss on each image alone, with the bars of tests/test_gpu_resnet.py and
  tests/test_gpu_bisenet.py (fp32-accurate forward: relative RMS <= 2e-2, cosine >= 0.999).
* The native path uses no autograd, on the identity decoder (DDPM), the VQ decoder (LDM) and the KL decoder (SD), and
  agrees with the per-sample autograd path on the same engines.
* Fall-backs and errors."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import step_math as sm

pytestmark = pytest.mark.gpu

DDPM64 = dict(sample_size=64, in_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1,
              down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"))
DDPM256 = dict(sample_size=256, in_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1,
               down_block_types=("DownBlock2D", "DownBlock2D"), up_block_types=("UpBlock2D", "UpBlock2D"))


def rel(a, b):
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()


def cos(a, b):
    return torch.nn.functional.cosine_similarity(a.flatten(), b.flatten(), dim=0).item()


def torchvision_resnet50(seed):
    tv = pytest.importorskip("torchvision")
    torch.manual_seed(seed)
    net = tv.models.resnet50()
    net.fc = torch.nn.Linear(net.fc.in_features, 80)
    g = torch.Generator().manual_seed(seed + 1)
    for mod in net.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):   # a trained network's statistics are not (0, 1)
            mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
            mod.running_var.copy_(torch.rand(mod.num_features, generator=g) * 0.5 + 0.75)
            mod.weight.data.copy_(torch.rand(mod.num_features, generator=g) * 0.5 + 0.75)
            mod.bias.data.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
    return net.eval()


@pytest.fixture(scope="module")
def predictor_pair():
    """(native fp32-accurate ResNet-50 at 64x64, max_batch 4; the torchvision module with the same weights on the GPU)."""
    from b200edit.resnet import ResNet
    ref = torchvision_resnet50(5)
    native = ResNet("bottleneck", (3, 4, 6, 3), 80, 64, max_batch=4, precision="fp32")
    native.load_torchvision_state_dict(ref.state_dict())
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return native, ref.cuda()


@pytest.fixture(scope="module")
def parser_pair():
    """(MultiResBiSeNet with max_batch 4; the oracle BiSeNet with the same weights on the GPU).  Logits of O(1): an
    unsaturated softmax, as a trained parser has."""
    from b200edit.bisenet import MultiResBiSeNet
    from oracle.bisenet import BiSeNet as OracleBiSeNet, seeded_weights
    oracle = seeded_weights(OracleBiSeNet(19).eval(), 8)
    oracle.conv_out.conv_out.weight.data.mul_(0.02)
    native = MultiResBiSeNet(19, max_batch=4)
    native.load_reference_state_dict(oracle.state_dict())
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return native, oracle.cuda()


@pytest.fixture(scope="module")
def ddpm64():
    from models import create_diffusion_model
    w = create_diffusion_model("ddpm", sample_clipping=False, max_batch=4, seed=1, unet_config=DDPM64)
    w.scheduler.set_timesteps(10)
    return w


def _inputs(B, C, S, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, C, S, S, generator=g).cuda(), torch.randn(B, C, S, S, generator=g).cuda()


def _apply(f, w, xt, eps, t, **kw):
    kw.setdefault("mask", None)
    x2, _ = f.apply(xt=xt.clone(), zt=None, model_output=eps, timestep=torch.tensor(t), step_idx=0, model=w, **kw)
    return (x2 - xt).detach()


class _NoAutograd:
    def __enter__(self):
        self.real = torch.autograd.grad

        def no_autograd(*a, **k):
            raise AssertionError("torch.autograd.grad called on the native network guidance path")
        torch.autograd.grad = no_autograd

    def __exit__(self, *exc):
        torch.autograd.grad = self.real


# ----------------------------------------------------------------------------- 1. batched heads vs the oracle
@pytest.mark.parametrize("B", [1, 3, 8])
@pytest.mark.parametrize("S", [64, 256])
@pytest.mark.parametrize("classes", [[17], [1, 10, 13], list(range(0, 19, 2))])
def test_batched_seg_area_head_vs_oracle(B, S, classes):
    from b200edit import ops
    logits = 3.0 * torch.randn(B, 19, S, S, generator=torch.Generator().manual_seed(B * S + len(classes)))
    loss, grad = ops.seg_area_head(logits.cuda(), classes, per_sample=True)
    assert loss.shape == (B,) and grad.shape == logits.shape
    for b in range(B):
        lb = logits[b:b + 1].clone().requires_grad_(True)
        ref = sm.segmentation_area_loss(lb, classes)
        (gr,) = torch.autograd.grad(ref, lb)
        assert np.allclose(loss[b].item(), ref.item(), rtol=1e-5, atol=0)
        gr = gr.numpy()
        assert np.allclose(grad[b:b + 1].cpu().numpy(), gr, rtol=1e-5, atol=1e-5 * np.abs(gr).max())


@pytest.mark.parametrize("reg", [(None, None, None), (15, 1, torch.tensor([0.3, -0.6])), (31, 0, torch.tensor([0.2, 0.1]))])
def test_batched_classifier_head_is_the_batch_one_head_of_every_row(reg):
    from b200edit import ops
    lg = torch.randn(6, 80, generator=torch.Generator().manual_seed(3)).cuda()
    loss, grad = ops.classifier_head(lg, 31, 0, reg, per_sample=True)
    for b in range(6):
        lb, gb = ops.classifier_head(lg[b:b + 1], 31, 0, reg)       # pinned to the reference's goldens
        assert loss[b].item() == lb.item()
        assert torch.equal(grad[b:b + 1], gb)
        x = lg[b:b + 1].clone().requires_grad_(True)
        ref = sm.classifier_logit_loss(x, 31, 0, (reg[0], reg[1], None if reg[2] is None else reg[2].cuda()))
        (gr,) = torch.autograd.grad(ref, x)
        assert loss[b].item() == ref.item() and torch.equal(grad[b:b + 1], gr)


def test_grad_scale_is_a_multiply_of_the_unscaled_gradient():
    from b200edit import ops
    lg = 3.0 * torch.randn(3, 19, 64, 64, generator=torch.Generator().manual_seed(4)).cuda()
    for scale in (1e4, 37.3, -2.5):
        l1, g1 = ops.seg_area_head(lg, [1, 10], per_sample=True)
        ls, gs = ops.seg_area_head(lg, [1, 10], per_sample=True, grad_scale=scale)
        assert torch.equal(l1, ls) and torch.equal(gs, g1 * scale)
        c = torch.randn(3, 80, generator=torch.Generator().manual_seed(5)).cuda()
        reg = (3, 1, torch.tensor([0.5, -0.25]))
        l1, g1 = ops.classifier_head(c, 7, 1, reg, per_sample=True)
        ls, gs = ops.classifier_head(c, 7, 1, reg, per_sample=True, grad_scale=scale)
        assert torch.equal(l1, ls) and torch.equal(gs, g1 * scale)


# ----------------------------------------------------------------------------- 2. batch invariance
@pytest.mark.parametrize("S", [64, 256])
def test_batched_seg_area_head_is_batch_invariant(S):
    from b200edit import ops
    lg = 3.0 * torch.randn(5, 19, S, S, generator=torch.Generator().manual_seed(S)).cuda()
    loss, grad = ops.seg_area_head(lg, [17, 1], per_sample=True, grad_scale=3.0)
    for b in range(5):
        lb, gb = ops.seg_area_head(lg[b:b + 1], [17, 1], per_sample=True, grad_scale=3.0)
        assert torch.equal(loss[b:b + 1], lb) and torch.equal(grad[b:b + 1], gb)
    l1, g1 = ops.seg_area_head(lg[2:3], [17, 1], per_sample=True)
    l0, g0 = ops.seg_area_head(lg[2:3], [17, 1])
    assert l1[0].item() == l0.item() and torch.equal(g1, g0)


# ----------------------------------------------------------------------------- 3. / 4. per-sample apply vs fp32 autograd
def test_per_sample_classifier_guidance_through_the_native_resnet(predictor_pair, ddpm64):
    from attr_functions import ClassifierAttrFunc
    native, ref = predictor_pair
    xt, eps = _inputs(3, 3, 64, 9)
    t = int(ddpm64.scheduler.timesteps[5])
    f = ClassifierAttrFunc(native, idx_for_class=31, idx_of_interest=0, loss_scale=50.0, per_sample=True)
    with _NoAutograd():
        dn = _apply(f, ddpm64, xt, eps, t)
    fr = ClassifierAttrFunc(ref, idx_for_class=31, idx_of_interest=0, loss_scale=50.0)
    for b in range(3):
        dr = _apply(fr, ddpm64, xt[b:b + 1], eps[b:b + 1], t)
        print(f"per-sample ClassifierAttrFunc image {b}: rel-rms {rel(dn[b:b + 1], dr):.3e} cos {cos(dn[b:b + 1], dr):.6f}")
        assert dn[b].abs().max() > 0 and dr.abs().max() > 0
        assert rel(dn[b:b + 1], dr) <= 2e-2 and cos(dn[b:b + 1], dr) >= 0.999


def test_per_sample_net_attr_guidance_through_the_native_bisenet(parser_pair):
    from attr_functions import NetAttrFunc
    from models import SegmentationModel, create_diffusion_model
    native, oracle = parser_pair
    w = create_diffusion_model("ddpm", sample_clipping=False, max_batch=3, seed=1, unet_config=DDPM256)
    w.scheduler.set_timesteps(10)
    xt, eps = _inputs(3, 3, 256, 9)
    t = int(w.scheduler.timesteps[-1])     # late step (alpha_bar ~ 1) and a large scale: the area loss is normalised by 256^2
    f = NetAttrFunc(SegmentationModel(net=native, image_size=(256, 256)), idx_for_class=[1, 10], loss_scale=1e4,
                    per_sample=True)
    with _NoAutograd():
        dn = _apply(f, w, xt, eps, t)
    fr = NetAttrFunc(SegmentationModel(net=oracle, image_size=(256, 256)), idx_for_class=[1, 10], loss_scale=1e4)
    for b in range(3):
        dr = _apply(fr, w, xt[b:b + 1], eps[b:b + 1], t)
        print(f"per-sample NetAttrFunc image {b}: rel-rms {rel(dn[b:b + 1], dr):.3e} cos {cos(dn[b:b + 1], dr):.6f}")
        assert dn[b].abs().max() > 0 and dr.abs().max() > 0
        assert rel(dn[b:b + 1], dr) <= 2e-2 and cos(dn[b:b + 1], dr) >= 0.999


# ----------------------------------------------------------------------------- 5. independence of the other images
def test_per_sample_nudge_does_not_depend_on_the_batch(predictor_pair, parser_pair, ddpm64):
    """Image b's nudge in a batch of 4 against a batch-1 run on image b.  Convolution split-K choices depend on the
    grid, so bits may differ; the bar is relative RMS <= 1e-3 (measured on a B200: 0, bit-identical, for both networks
    at 64x64)."""
    from attr_functions import ClassifierAttrFunc, NetAttrFunc
    from models import SegmentationModel
    native, _ = predictor_pair
    parser, _ = parser_pair
    xt, eps = _inputs(4, 3, 64, 11)
    t = int(ddpm64.scheduler.timesteps[5])
    cases = {
        "ClassifierAttrFunc": ClassifierAttrFunc(native, idx_for_class=31, idx_of_interest=0, loss_scale=50.0, per_sample=True),
        "NetAttrFunc": NetAttrFunc(SegmentationModel(net=parser, image_size=(64, 64)), idx_for_class=[1, 10], loss_scale=1e4,
                                   per_sample=True),
    }
    for tag, f in cases.items():
        d4 = _apply(f, ddpm64, xt, eps, t)
        for b in range(4):
            d1 = _apply(f, ddpm64, xt[b:b + 1], eps[b:b + 1], t)
            print(f"{tag} image {b}: batch-4 vs batch-1 nudge rel-rms {rel(d4[b:b + 1], d1):.3e}")
            assert d1.abs().max() > 0 and rel(d4[b:b + 1], d1) <= 1e-3


# ----------------------------------------------------------------------------- 6. no autograd on every decoder family
def _latent_model(family):
    from b200edit.scheduler import DDIMScheduler
    from b200edit.vqmodel import AutoencoderKL, VQModel
    from diffusion_classes import LDM, SD
    if family == "ldm":
        dec = VQModel(latent_channels=3, out_channels=3, block_out_channels=(32, 96), layers_per_block=1, norm_num_groups=32,
                      norm_eps=1e-6, num_vq_embeddings=512, sample_size=32, max_batch=3)
        Cl = 3
    else:
        dec = AutoencoderKL(latent_channels=4, out_channels=3, block_out_channels=(64, 64, 128), layers_per_block=1,
                            norm_num_groups=32, norm_eps=1e-6, sample_size=16, max_batch=3)
        Cl = 4
    dec.init_random(21)
    dec.enable_grad()
    sch = DDIMScheduler.from_preset(family)
    sch.set_timesteps(10)
    S = dec.config.sample_size
    pipe_obj = SimpleNamespace(unet=SimpleNamespace(config=SimpleNamespace(in_channels=Cl, sample_size=S), in_channels=Cl,
                                                    sample_size=S),
                               scheduler=sch, device=torch.device("cuda"), vqvae=dec, vae=dec, tokenizer=None, text_encoder=None)
    w = LDM(pipe_obj) if family == "ldm" else SD(pipe_obj)
    assert dec.out_size == 64
    return w, Cl, S


@pytest.mark.parametrize("family", ["ddpm", "ldm", "sd"])
def test_native_network_guidance_runs_without_autograd(family, predictor_pair, parser_pair, ddpm64):
    """The native path against the per-sample autograd path on the same engines (network wrapped in a lambda, which the
    native path cannot see through): only the x0' arithmetic (torch's CUDA division multiplies by the reciprocal) and
    the update arithmetic differ.  Measured on a B200: DDPM 1.1e-3 .. 1.3e-3 relative RMS / cosine 0.999999 (the one-ulp
    x0' difference moves a few ReLU masks of the fp32-accurate networks), LDM and SD 3e-8 .. 8e-8."""
    from attr_functions import ClassifierAttrFunc, NetAttrFunc
    native, _ = predictor_pair
    parser, _ = parser_pair
    if family == "ddpm":
        w, Cl, S, scale = ddpm64, 3, 64, 1.0
    else:
        w, Cl, S = _latent_model(family)
        scale = 1.0 if family == "ldm" else 0.18215
    xt, eps = _inputs(3, Cl, S, 31)
    xt, eps = xt * scale, eps * scale
    t = int(w.scheduler.timesteps[-3])
    lmask = (torch.rand(1, Cl, S, S, generator=torch.Generator().manual_seed(32)) > 0.4).float().cuda()
    seg = lambda net: SimpleNamespace(net=net)                                           # noqa: E731
    cases = [
        ("classifier", lambda p: ClassifierAttrFunc(p, idx_for_class=31, idx_of_interest=0, loss_scale=50.0, per_sample=True,
                                                     regularize_idx_idx_score=(15, 1, torch.tensor([0.3, -0.6]))),
         native, {}),
        ("net-attr", lambda p: NetAttrFunc(seg(p), idx_for_class=[1, 10], loss_scale=1e4, per_sample=True), parser, {}),
        ("net-attr masked gradient", lambda p: NetAttrFunc(seg(p), idx_for_class=[4], loss_scale=1e4, per_sample=True), parser,
         dict(mask=lmask, mask_attr_grad=True)),
    ]
    for tag, make, net, kw in cases:
        f = make(net)
        with _NoAutograd():
            dn = _apply(f, w, xt, eps, t, **kw)
        da = _apply(make(lambda x, net=net: net(x)), w, xt, eps, t, **kw)
        r, c = rel(dn, da), cos(dn, da)
        print(f"{family} {tag}: native vs autograd per-sample nudge rel-rms {r:.3e} cos {c:.6f}")
        for b in range(3):
            assert dn[b].abs().max() > 0
        assert r <= 5e-3 and c >= 0.9999, (family, tag, r, c)


# ----------------------------------------------------------------------------- 7. fall-backs and errors
def test_fallbacks_stay_per_sample(predictor_pair, ddpm64):
    from attr_functions import ClassifierAttrFunc
    native, ref = predictor_pair
    xt, eps = _inputs(3, 3, 64, 41)
    t = int(ddpm64.scheduler.timesteps[5])
    mask = (torch.rand(1, 3, 64, 64, generator=torch.Generator().manual_seed(42)) > 0.4).float().cuda()
    x_0 = torch.randn(3, 3, 64, 64, generator=torch.Generator().manual_seed(43)).cuda()
    # mask_pred_original_sample + L2: autograd through the native predictor's own autograd node
    f = ClassifierAttrFunc(native, idx_for_class=31, loss_scale=50.0, per_sample=True, use_l2=True)
    d = _apply(f, ddpm64, xt, eps, t, mask=mask, mask_pred_original_sample=True, use_l2=True, lambda_=0.1, x_0=x_0)
    assert all(d[b].abs().max() > 0 for b in range(3))
    # nudge_zt: both the sample and the noise get every image's gradient
    f = ClassifierAttrFunc(native, idx_for_class=31, loss_scale=50.0, per_sample=True, nudge_zt=True)
    zt = torch.randn(3, 3, 64, 64, generator=torch.Generator().manual_seed(44)).cuda()
    x2, z2 = f.apply(xt=xt.clone(), zt=zt.clone(), model_output=eps, timestep=torch.tensor(t), step_idx=0, model=ddpm64,
                     mask=None)
    for b in range(3):
        assert (x2 - xt)[b].abs().max() > 0 and torch.allclose(x2 - xt, z2 - zt, rtol=1e-5, atol=1e-6)
    # a torch module: per-sample autograd, image b's nudge is the batch-1 nudge of image b
    f = ClassifierAttrFunc(ref, idx_for_class=31, loss_scale=50.0, per_sample=True)
    d = _apply(f, ddpm64, xt, eps, t)
    fr = ClassifierAttrFunc(ref, idx_for_class=31, loss_scale=50.0)
    for b in range(3):
        dr = _apply(fr, ddpm64, xt[b:b + 1], eps[b:b + 1], t)
        # cuDNN picks its convolution algorithms by batch size: measured 2.5e-3 on a B200, so the fp32 bars of
        # tests/test_gpu_resnet.py apply
        assert dr.abs().max() > 0 and rel(d[b:b + 1], dr) <= 2e-2 and cos(d[b:b + 1], dr) >= 0.999


def test_errors(predictor_pair, parser_pair):
    from attr_functions import ClassifierAttrFunc, NetAttrFunc
    from b200edit import ops
    from b200edit._C import B2EError
    from models import create_diffusion_model
    native, _ = predictor_pair
    parser, _ = parser_pair
    w = create_diffusion_model("ddpm", sample_clipping=False, max_batch=5, seed=1, unet_config=DDPM64)
    w.scheduler.set_timesteps(10)
    t = int(w.scheduler.timesteps[5])
    xt, eps = _inputs(5, 3, 64, 51)
    with pytest.raises(ValueError):           # B > the predictor's max_batch (4)
        _apply(ClassifierAttrFunc(native, idx_for_class=31, per_sample=True), w, xt, eps, t)
    with pytest.raises(ValueError):           # B > the parser's max_batch (4)
        _apply(NetAttrFunc(SimpleNamespace(net=parser), idx_for_class=[1], per_sample=True), w, xt, eps, t)
    with pytest.raises(B2EError):             # class id out of range, on the native path
        _apply(NetAttrFunc(SimpleNamespace(net=parser), idx_for_class=[19], per_sample=True), w, xt[:2], eps[:2], t)
    with pytest.raises(B2EError):
        _apply(ClassifierAttrFunc(native, idx_for_class=40, per_sample=True), w, xt[:2], eps[:2], t)
    with pytest.raises(ValueError):
        ops.seg_area_head(torch.randn(19, 8, 8, device="cuda"), [1], per_sample=True)
    with pytest.raises(ValueError):
        ops.classifier_head(torch.randn(2, 79, device="cuda"), 3, 0, per_sample=True)
