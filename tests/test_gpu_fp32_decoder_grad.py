"""fp32-accurate decoder gradient: the split VQ / KL decoder in gradient mode, its fp32 attention backward, and guidance
through it, against float64.

In the fp32-accurate mode (precision="fp32") every activation is a split 16-bit pair hi + lo and every GEMM weight is
packed [W_hi | W_hi | W_lo] x 2^10.  In gradient mode the decoder's dgrad twins are packed the same way, gradients travel
as split tensors, and GroupNorm / upsample / col2im backward and the mid-block attention backward run in fp32.  Bars
(e = 2^-24, u = the 16-bit unit roundoff: 2^-11 fp16, 2^-8 bf16):

  attention backward (b2e_attention_bwd_fp32, single head, T tokens, C channels) against float64 autograd of
      softmax(q k^T / sqrt(C)) v on the exact hi + lo inputs.  Every output is a sum of products evaluated in fp32:
        dV = P^T dO,   dK = dS^T (q / sqrt(C)),   dQ = dS k / sqrt(C),   dS = P o (dP - D),  dP = dO v^T,  D = rowsum(dO o O).
      First-order running-error estimate, each fp32 operation one relative error <= e with independent signs, so errors
      of a sum add in quadrature (quad(a, b) = sqrt(sum_t (a_t b_t)^2) over the contraction):
        P      relative error (4Z + 8) e (Z = max |scaled logit|: the fp32 logit, the exp, the max and 1 / l);
        dP, D  sums over C terms: sqrt(C) e (rss(dO o v_k) + rss(dO o O_q)), with O a split tensor;
        dS     sigma_qk = P_qk ((4Z + 8) |dP - D| + sqrt(C) (rss(dO o v_k) + rss(dO o O_q)));
        sums over T terms add sqrt(T) e quad of the exact terms:
          sigma(dQ) = quad(sigma, k / sqrt(C)) + sqrt(T) quad(dS, k / sqrt(C)),
          sigma(dK) = quad(sigma^T, q / sqrt(C)) + (sqrt(T) + 1) quad(dS^T, q / sqrt(C))  (+1: the pre-scaled q),
          sigma(dV) = (4Z + 8 + sqrt(T)) quad(P^T, dO).
      The outputs are stored as hi + lo: u^2 |G| (and u^2 once more for O inside D).  A quadrature sum is a standard
      deviation, so the bar allows four of them:
        bar(G) = 4 e max sigma(G) + 2 u^2 max |G|.
      The bar must be at least 10x below the error of the 16-bit backward (torch float16 autograd on the hi
      planes) on the same inputs.  Mutation check: the same call with d_o's lo plane zeroed misses the bar.  Two calls
      give identical bits (no atomics).
  decoder gradient d(loss)/d(latent) (the smooth dense loss of test_gpu_vqdecoder._grad_pair) against autograd through
      oracle/vqmodel.py in float64 with the same weights: relative RMS <= 1e-4, the decoder's fp32-mode bar, and <= 0.1x
      the relative RMS of the 16-bit engine's gradient on the same inputs.  torch float32 autograd's own distance from
      float64 is printed beside it as the yardstick.
  forward in gradient mode: decode_keep(z) of the split decoder in gradient mode equals decode(z) of a forward-only
      split decoder with the same weights bit for bit (the gradient mode changes no forward arithmetic).
  guided update (AttrFunc.apply, no autograd) on an fp32 pipeline built with decoder_grad_precision="fp32", against the
      reference's procedure (AttrFunc._apply_autograd) through the float64 oracle decoder: targets outside the image
      range keep sign(img - target) constant, so d(loss)/d(image) is exact and the update carries only the decoder
      gradient's error (and, for the L2 variant, the fp32 forward's): max |diff| <= 1e-4 max |update|.

Every check prints its measured error beside its bar."""
from types import SimpleNamespace

import pytest
import torch

from oracle.vqmodel import LDM_VQ_CONFIG, SD_VAE_CONFIG, VQModel as OracleVQ

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -24
SMALL_VQ = dict(latent_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1, norm_num_groups=32,
                norm_eps=1e-6, num_vq_embeddings=512, sample_size=16)
SMALL_KL = dict(latent_channels=4, out_channels=3, block_out_channels=(64, 64, 128), layers_per_block=1, norm_num_groups=32,
                norm_eps=1e-6, num_vq_embeddings=0, sample_size=16)
SMALL_UNET = dict(sample_size=16, in_channels=3, out_channels=3, block_out_channels=(32, 96), layers_per_block=1,
                  down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"),
                  attention_head_dim=32, flip_sin_to_cos=True, freq_shift=0, downsample_padding=1)
SMALL_SD_UNET = dict(sample_size=16, in_channels=4, out_channels=4, block_out_channels=(64, 128), layers_per_block=1,
                     cross_attention_dim=64, attention_head_dim=2, norm_num_groups=32, norm_eps=1e-5)


def _factory_kw(family):
    """The noise predictor is not run by these tests: small configs; SD gets a placeholder text encoder (no CLIP built)."""
    if family == "ldm":
        return dict(unet_config=SMALL_UNET)
    return dict(unet_config=SMALL_SD_UNET, text_encoder=SimpleNamespace())


def _factory_vq(vcfg):
    return {k: v for k, v in vcfg.items() if not (k == "num_vq_embeddings" and v == 0)}   # AutoencoderKL has no quantiser


def _rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()


def _unit_roundoff():
    from b200edit import ops
    return 2.0 ** -8 if ops.act_dtype() == torch.bfloat16 else 2.0 ** -11


# ------------------------------------------------------------------ 1. attention backward kernel
def _split(x):
    from b200edit import ops
    return ops.split_planes(x.float())


def _exact(s):
    from b200edit import ops
    return ops.merge_planes(s).double()   # hi + lo is exact in float64


@pytest.mark.parametrize("B,T,C", [(1, 4096, 512), (2, 256, 128), (2, 64, 64)])
def test_attention_backward_matches_float64(B, T, C):
    from b200edit import ops
    P = (C + 63) // 64 * 64
    g = torch.Generator().manual_seed(T + C)
    q, k, v = (torch.randn(B, T, C, generator=g) * s for s in (1.5, 1.0, 1.0))
    dO = torch.randn(B, T, C, generator=g)      # O(1), as the decoder's power-of-two gradient scale leaves it
    pad = lambda x: torch.nn.functional.pad(x, (0, P - C))   # noqa: E731
    qkv_s = _split(torch.cat([pad(q), pad(k), pad(v)], dim=-1).cuda())      # (B, T, 9P): [hi | lo | hi] of q | k | v
    qkv = _exact(qkv_s)
    q64, k64, v64 = (qkv[..., i * P:i * P + C].clone().requires_grad_(True) for i in range(3))
    scale = 1.0 / C ** 0.5
    s64 = q64 @ k64.transpose(1, 2) * scale
    p64 = torch.softmax(s64, dim=-1)
    o64 = p64 @ v64
    dO_s = _split(pad(dO).cuda())
    dO64 = _exact(dO_s)[..., :C]
    grads = torch.autograd.grad(o64, (q64, k64, v64), dO64)
    o_s = _split(pad(o64.detach()).float())
    dq, dk, dv = ops.attention_bwd_fp32(qkv_s, o_s, dO_s, channels=C)
    got = [_exact(t)[..., :C] for t in (dq, dk, dv)]
    for t in (dq, dk, dv):
        assert (_exact(t)[..., C:] == 0).all()
    # first-order running-error scale of every output (see the module docstring), in float64
    with torch.no_grad():
        Z = s64.abs().max().item()
        o_ex = _exact(o_s)[..., :C]
        qs, ks = q64 * scale, k64 * scale
        dP, D = dO64 @ v64.transpose(1, 2), (dO64 * o_ex).sum(-1, keepdim=True)
        dS = p64 * (dP - D)
        rss_dP = ((dO64 ** 2) @ (v64 ** 2).transpose(1, 2)).sqrt()
        rss_D = ((dO64 * o_ex) ** 2).sum(-1, keepdim=True).sqrt()
        sig_dS = p64 * ((4 * Z + 8) * (dP - D).abs() + C ** 0.5 * (rss_dP + rss_D))
        quad = lambda a, b: ((a ** 2) @ (b ** 2)).sqrt()   # noqa: E731  sqrt(sum_t (a_t b_t)^2) over the contraction
        pT, dST, sigT = p64.transpose(1, 2), dS.transpose(1, 2), sig_dS.transpose(1, 2)
        sigma = [(quad(sig_dS, ks) + T ** 0.5 * quad(dS, ks)).max().item(),
                 (quad(sigT, qs) + (T ** 0.5 + 1) * quad(dST, qs)).max().item(),
                 ((4 * Z + 8) * quad(pT, dO64) + T ** 0.5 * quad(pT, dO64)).max().item()]
    u = _unit_roundoff()
    # 16-bit backward on the same inputs: torch float16 autograd on the hi planes
    q16, k16, v16 = (t.detach().half().requires_grad_(True) for t in (q64, k64, v64))
    o16 = torch.softmax((q16 @ k16.transpose(1, 2)).float() * scale, dim=-1).half() @ v16
    g16 = torch.autograd.grad(o16, (q16, k16, v16), dO64.half())
    # mutation: d_o without its lo plane
    dO_hi = dO_s.clone()
    dO_hi[..., P:2 * P] = 0
    mut = ops.attention_bwd_fp32(qkv_s, o_s, dO_hi, channels=C)
    again = ops.attention_bwd_fp32(qkv_s, o_s, dO_s, channels=C)
    for name, gn, gr, sg, gh, gm in zip("qkv", got, grads, sigma, g16, mut):
        err = (gn - gr).abs().max().item()
        bar = 4 * EPS32 * sg + 2 * u * u * gr.abs().max().item()
        err16 = (gh.double() - gr).abs().max().item()
        err_mut = (_exact(gm)[..., :C] - gr).abs().max().item()
        print(f"attention backward B={B} T={T} C={C} d{name}: max-abs {err:.3e} bar {bar:.3e} (Z {Z:.1f}, sigma {sg:.3e}) | "
              f"16-bit {err16:.3e} | without dO's lo plane {err_mut:.3e}")
        assert torch.isfinite(gn).all() and err <= bar
        assert bar <= 0.1 * err16
        assert err_mut > bar
    assert all(torch.equal(a, b) for a, b in zip(again, (dq, dk, dv)))


# ------------------------------------------------------------------ 2. / 3. decoder gradient and forward
def _oracle(cfg, seed):
    torch.manual_seed(seed)
    oracle = OracleVQ(**cfg).eval()
    if cfg["num_vq_embeddings"]:
        oracle.quantize.embedding.weight.data.uniform_(-2.0, 2.0)
    return oracle


def _native(cfg, B, precision, sd):
    from b200edit.vqmodel import VQModel
    m = VQModel(**cfg, max_batch=B, precision=precision)
    m.load_state_dict(sd)
    return m


def _loss(img, w):   # test_gpu_vqdecoder._grad_pair's smooth loss with a dense, sign-changing gradient
    return (img * w).sum() / img[0].numel() + (img ** 2).mean()


def _latent_grad(m, z, w):
    m.enable_grad()
    zn = z.clone().requires_grad_(True)
    (g,) = torch.autograd.grad(_loss(m.decode(zn).sample, w), zn)
    return g


@pytest.mark.parametrize("tag,cfg,B", [("small vq", SMALL_VQ, 1), ("small vq", SMALL_VQ, 2), ("small kl", SMALL_KL, 2),
                                       ("ldm vq", dict(LDM_VQ_CONFIG), 1), ("sd kl", dict(SD_VAE_CONFIG, num_vq_embeddings=0), 1)])
def test_split_decoder_gradient_matches_float64(tag, cfg, B):
    seed = 60 + B + cfg["sample_size"] + len(cfg["block_out_channels"])
    oracle = _oracle(cfg, seed)
    sd = oracle.state_dict()
    g = torch.Generator().manual_seed(seed + 1)
    z = torch.randn(B, cfg["latent_channels"], cfg["sample_size"], cfg["sample_size"], generator=g).cuda()
    S_out = cfg["sample_size"] << (len(cfg["block_out_channels"]) - 1)
    w = torch.randn(B, cfg["out_channels"], S_out, S_out, generator=g).cuda()
    g32 = _latent_grad(_native(cfg, B, "fp32", sd), z, w)
    g16 = _latent_grad(_native(cfg, B, None, sd), z, w)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    o64 = oracle.double().cuda()
    z64 = z.double().requires_grad_(True)
    (gref,) = torch.autograd.grad(_loss(o64.decode(z64).sample, w.double()), z64)
    o32 = _oracle(cfg, seed).cuda()
    z32 = z.clone().requires_grad_(True)
    (gt32,) = torch.autograd.grad(_loss(o32.decode(z32).sample, w), z32)
    rel, rel16, relt = _rel(g32, gref), _rel(g16, gref), _rel(gt32, gref)
    print(f"{tag} decoder gradient B={B}: fp32-accurate rel-rms {rel:.3e} (bar 1e-4, 0.1x 16-bit = {0.1 * rel16:.3e}) | "
          f"16-bit engine {rel16:.3e} | torch fp32 autograd {relt:.3e}")
    assert torch.isfinite(g32).all() and rel <= 1e-4 and rel <= 0.1 * rel16


@pytest.mark.parametrize("tag,cfg", [("small vq", SMALL_VQ), ("small kl", SMALL_KL), ("ldm vq", dict(LDM_VQ_CONFIG))])
def test_gradient_mode_leaves_the_split_forward_unchanged(tag, cfg):
    oracle = _oracle(cfg, 77)
    sd = oracle.state_dict()
    B = 2
    z = torch.randn(B, cfg["latent_channels"], cfg["sample_size"], cfg["sample_size"],
                    generator=torch.Generator().manual_seed(78)).cuda()
    fwd = _native(cfg, B, "fp32", sd)
    grad = _native(cfg, B, "fp32", sd).enable_grad()
    a = fwd.decode(z).sample
    b = grad.decode_keep(z)
    print(f"{tag}: gradient-mode decode_keep vs forward-only decode, max |diff| {(a - b).abs().max().item():.3e} (bar: 0, bit-exact)")
    assert torch.equal(a, b)


# ------------------------------------------------------------------ 4. guided update through the split decoder
class _Float64Decoder:
    """The oracle decoder in float64 behind the decode(...).sample contract (the reference's autograd path)."""

    def __init__(self, m):
        self.m = m.double().cuda()

    def decode(self, z):
        return SimpleNamespace(sample=self.m.decode(z.double()).sample.float())


def _guided_cases(Cl, S, S_img, B, g):
    from attr_functions import MultiColorAttrFunc, SingleColorAttrFunc
    lmask = (torch.rand(1, Cl, S, S, generator=g) > 0.4).float().cuda()
    imask = (torch.rand(1, 3, S_img, S_img, generator=g) > 0.4).float().cuda()
    x_0 = torch.randn(B, 3, S_img, S_img, generator=g).cuda()
    return {
        "single": (SingleColorAttrFunc(target=50.0, color_idx=0, loss_scale=300.0), {}),
        "multi": (MultiColorAttrFunc(40.0, -30.0, 50.0, loss_scale=3.0), {}),
        "masked gradient": (SingleColorAttrFunc(target=50.0, color_idx=1, loss_scale=300.0), dict(mask=lmask, mask_attr_grad=True)),
        "masked prediction + L2": (SingleColorAttrFunc(target=50.0, color_idx=0, loss_scale=300.0, use_l2=True),
                                   dict(mask=imask, mask_pred_original_sample=True, use_l2=True, lambda_=0.3, x_0=x_0)),
    }


@pytest.mark.parametrize("family,vcfg,B", [("ldm", SMALL_VQ, 2), ("sd", SMALL_KL, 2), ("ldm", dict(LDM_VQ_CONFIG), 1)])
def test_guided_update_through_the_split_decoder_matches_float64(family, vcfg, B):
    from diffusion_classes import LDM, SD
    from models import create_diffusion_model
    oracle = _oracle(vcfg, 91 + vcfg["sample_size"])
    kw = _factory_kw(family)
    w = create_diffusion_model(family, sample_clipping=False, max_batch=B, seed=3, vq_config=_factory_vq(vcfg),
                               vq_state_dict=oracle.state_dict(),
                               precision="fp32", decoder_grad_precision="fp32", with_encoder=False, **kw)
    dec = w.vqvae if family == "ldm" else w.vae
    Cl, S = vcfg["latent_channels"], vcfg["sample_size"]
    S_img = S << (len(vcfg["block_out_channels"]) - 1)
    shim = _Float64Decoder(oracle)
    ref_obj = SimpleNamespace(unet=w.unet, scheduler=w.scheduler, device=torch.device("cuda"), vqvae=shim, vae=shim,
                              tokenizer=None, text_encoder=None)
    w64 = LDM(ref_obj) if family == "ldm" else SD(ref_obj)
    sch = w.scheduler
    sch.set_timesteps(10)
    g = torch.Generator().manual_seed(92)
    sc = 1.0 if family == "ldm" else 0.18215
    xt = torch.randn(B, Cl, S, S, generator=g).cuda() * sc
    eps = torch.randn(B, Cl, S, S, generator=g).cuda() * sc
    t = torch.tensor(int(sch.timesteps[-3]))
    for tag, (f, fkw) in _guided_cases(Cl, S, S_img, B, g).items():
        coeffs = sch.coeffs(int(t), 0.0, "ddim")
        real_grad = torch.autograd.grad

        def no_autograd(*a, **k):
            raise AssertionError("torch.autograd.grad called on the native analytic guidance path")

        torch.autograd.grad = no_autograd
        try:
            xn, _ = f.apply(xt=xt.clone(), zt=None, model_output=eps, timestep=t, step_idx=0, model=w, **fkw)
        finally:
            torch.autograd.grad = real_grad
        xa, _ = f._apply_autograd(xt.clone(), None, eps, coeffs, w64, **fkw)
        du, dr = xn - xt, xa - xt
        err = (du - dr).abs().max().item() / dr.abs().max().item()
        print(f"{family} {tag} (latent {S}, B={B}): fp32 decoder-gradient update vs float64 autograd: max|diff| / max|update| = "
              f"{err:.2e} (bar 1e-4; max|update| {dr.abs().max().item():.2e})")
        assert dr.abs().max() > 0 and err <= 1e-4, (family, tag, err)
    assert w.native_decoder()[0] is dec


# ------------------------------------------------------------------ 5. wiring and defaults
@pytest.mark.parametrize("family", ["ldm", "sd"])
def test_decoder_grad_precision_wiring(family):
    from b200edit._C import B2EError
    from models import create_diffusion_model
    vcfg = SMALL_VQ if family == "ldm" else SMALL_KL
    kw = _factory_kw(family)
    w = create_diffusion_model(family, max_batch=1, seed=3, vq_config=_factory_vq(vcfg), precision="fp32", decoder_grad_precision="fp32",
                               with_encoder=False, **kw)
    dec, twin = (w.vqvae, w.guidance_vqvae) if family == "ldm" else (w.vae, w.guidance_vae)
    assert twin is None and not dec.forward_only and dec.precision == "fp32"
    assert w.native_decoder()[0] is dec
    z = torch.randn(1, vcfg["latent_channels"], 16, 16, generator=torch.Generator().manual_seed(4)).cuda()
    img = dec.decode_keep(z)
    dec.decode(z * 0.5)             # an intervening forward on the same engine
    with pytest.raises(B2EError, match="another forward"):
        dec.latent_grad(torch.ones_like(img))
