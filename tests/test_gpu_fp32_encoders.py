"""fp32-accurate VQ / KL encoders and CLIP text encoder, and the causal fp32 tiled attention under CLIP, against float64.

The fp32-accurate mode keeps every activation as a split 16-bit pair hi + lo and packs every GEMM weight as
[W_hi | W_hi | W_lo]; element-wise ops, normalisations and attention run in fp32 on the CUDA cores.  The bars are the
project's fp32-mode bars:

  causal attention (path "fp32_tiled_causal"): the fp32-tiled bar of test_gpu_attention.py, (e (8Z + 64) + u^2) R with
      e = 2^-24, u the 16-bit unit roundoff, R = max |V| over the valid keys, Z = max |scaled logit| over the unmasked
      scores.  The reference takes the exact hi + lo inputs and the inputs of test_gpu_attention.make_inputs, whose causal
      regime makes every future key outweigh the diagonal.  Mutation check: the float64 reference with the diagonal
      moved by one key either way differs from the kernel's output by more than the bar.
  CLIP last hidden state: max-abs <= 1e-4 max(1, max|h|) and relative RMS <= 5e-5, the UNet fp32 bars, against
      transformers' CLIPTextModel run in float64 with the same weights.
  encoders (latent, or the KL moments' mean): max-abs <= 1e-4 max(1, max|latent|) and relative RMS <= 1e-4, the
      decoder fp32 bars, against oracle/vqmodel.py run in float64 with the same weights.
  LDM inversion (edit-friendly DDPM inversion, eta = 1, injected noise, 10 steps), against the float64 chain oracle
      encoder -> oracle UNet -> oracle.loops.invert_ddpm with the same noise and the same fp32 scheduler coefficients:
    xts[i] = sqrt(a_t) x0 + sqrt(1 - a_t) n_t is a linear map of x0 with a coefficient <= 1, so the encoder bar holds
      for rows 0 .. T - 1 of xts.  Row T is the x0 "corrected" by the last step, whose variance is 0: NaN, as in the
      reference, and not compared.
    zs[i] = (x_{t-1} - mu) / (eta sigma_t), mu = sp (x_t - sb eps) / sa + cdir eps, with sa = sqrt(a_t),
      sb = sqrt(1 - a_t), sp = sqrt(a_prev), cdir = sqrt(1 - a_prev - eta sigma_t^2).  The x0 part of x_{t-1} and of
      sp x_t / sa is the same, sp x0, so an error in x0 cancels; an eps error de moves z by |dz/de| de with
      |dz/de| = |cdir - sp sb / sa| / (eta sigma_t).  With the UNet eps bar de <= 1e-4 max(1, max|eps_t|) and the fp32
      roundings of the step (a few e relative on each term of the numerator):
        bar_z(t) = (|cdir - sp sb / sa| de + 8 e (|x_{t-1}| + sp (|x_t| + sb |eps|) / sa + cdir |eps|)) / (eta sigma_t)
      with the magnitudes taken as the maxima of the float64 chain.  zs[T - 1] is zero in both.
  SD text conditioning: prep_text through a fake tokenizer and the native CLIP at the CLIP bar, then one CFG noise
      prediction: each half of the doubled batch at the UNet bar against the float64 conditional oracle UNet fed with the
      float64 text embedding, and the combination e_u + s (e_c - e_u) at (1 + 2 s) times the larger of the two bars.

Every check prints its measured error beside its bar."""
import pytest
import torch

import test_gpu_attention as ta
from oracle.vqmodel import LDM_VQ_CONFIG, SD_VAE_CONFIG, VQModel as OracleVQ

EPS32 = 2.0 ** -24
CAUSAL = "fp32_tiled_causal"

CAUSAL_CASES = [
    # CLIP text encoder: 12 heads of 64, 128 padded token rows, valid_k text tokens
    *[ta._mh(CAUSAL, f"clip-12h-vk{vk}", 2, 1, 128, 12, 64, valid_k=vk, causal=True) for vk in (1, 20, 77)],
    # two heads over 77 tokens: a ragged last 32-query block, no key padding
    ta._mh(CAUSAL, "small-2h-t77", 1, 1, 77, 2, 64, causal=True),
]

SMALL_CLIP = dict(vocab_size=1000, hidden_size=128, intermediate_size=512, num_hidden_layers=2, num_attention_heads=2,
                  max_position_embeddings=77)
SMALL_VQ = dict(latent_channels=3, out_channels=3, block_out_channels=(32, 96), layers_per_block=1, norm_num_groups=32,
                norm_eps=1e-6, num_vq_embeddings=512, sample_size=16)
SMALL_KL = dict(latent_channels=4, out_channels=3, block_out_channels=(64, 128, 128), layers_per_block=1, norm_num_groups=32,
                norm_eps=1e-6, num_vq_embeddings=0, sample_size=8)


def _errors(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    err = (got - ref).abs().max().item()
    rel = ((got - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt()).item()
    return err, rel, ref.abs().max().item()


def check_bars(got, ref, rel_bar, tag):
    """max-abs <= 1e-4 max(1, max|ref|) and relative RMS <= rel_bar"""
    assert got.shape == ref.shape and torch.isfinite(got).all()
    err, rel, scale = _errors(got, ref)
    bar = 1e-4 * max(1.0, scale)
    print(f"{tag}: max-abs {err:.3e} (bar {bar:.3e}) rel-rms {rel:.3e} (bar {rel_bar:.1e}) | max|ref| {scale:.3f}")
    assert err <= bar and rel <= rel_bar, (err, bar, rel, rel_bar)


def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


# ----------------------------------------------------------------------------------------------------- causal kernel
@pytest.mark.gpu
@pytest.mark.parametrize("regime", ta.REGIMES)
@pytest.mark.parametrize("case", CAUSAL_CASES, ids=str)
def test_causal_fp32_tiled_attention_matches_float64(case, regime):
    torch.cuda.set_device(0)
    u = ta.unit_roundoff()
    q, k, v = ta.make_inputs(case, regime)
    out = ta.run_case(case, q, k, v)
    torch.cuda.synchronize()
    C, P = case.heads * case.d, case.P
    for pl in (out[..., i * P:(i + 1) * P] for i in range(3)):
        assert pl[..., C:].numel() == 0 or (pl[..., C:] == 0).all().item(), "pitch tail not zeroed"
    from b200edit import ops
    got = ops.merge_planes(out)[..., :C].double()
    assert torch.isfinite(got).all().item(), "unwritten (NaN) or non-finite output"
    qr, kr, vr = (ta.kernel_view(x, case.path)[0].cuda() for x in (q, k, v))
    ref, Z = ta.reference(case, qr, kr, vr)
    ref = ref.reshape(case.B, case.Tq, C)
    err = (got - ref).abs().max().item()
    R = ta.value_range(case, vr)
    b = ta.bar(case.path, u, R, Z)
    print(f"{case} {regime}: max err {err:.3e}  bar {b:.3e}  ({err / b:.3f} of the bar; R {R:.2f} Z {Z:.1f})")
    assert err <= b, (err, b)
    if case.vk > 1:
        for fault in ("diag_next", "diag_prev"):
            alt, _ = ta.reference(case, qr, kr, vr, fault=fault)
            diff = (got - alt.reshape(case.B, case.Tq, C)).abs().nan_to_num(0.0).max().item()
            print(f"{case} {regime}: reference with {fault} differs from the kernel by {diff:.3e} = {diff / b:.0f} x bar")
            assert diff > b, (fault, diff, b)


@pytest.mark.gpu
def test_causal_path_refuses_non_causal_calls_and_others_refuse_causal():
    from b200edit import ops
    from b200edit._C import B2EError
    torch.cuda.set_device(0)
    qkv = torch.zeros(1, 128, 3 * 64, device="cuda")
    kw = dict(hw=(1, 128), heads=1, head_dim=64, q_col=0, k_col=64, v_col=128, out_pitch=64)
    with pytest.raises(B2EError, match="unknown path"):
        ops.attention_f16(qkv, qkv, causal=False, path=CAUSAL, **kw)
    for path in ("fp32_split", "fp32_tiled"):
        with pytest.raises(B2EError, match="causal"):
            ops.attention_f16(qkv, qkv, causal=True, path=path, **kw)


# ----------------------------------------------------------------------------------------------------- CLIP
def _clip_pair(cfg, B, L, seed):
    from b200edit.clip import CLIPTextModel
    from transformers import CLIPTextConfig, CLIPTextModel as RefCLIP
    torch.manual_seed(seed)
    ref = RefCLIP(CLIPTextConfig(hidden_act="quick_gelu", attn_implementation="eager", **cfg)).eval()
    native = CLIPTextModel(**cfg, max_batch=B, precision="fp32")
    assert native.precision == "fp32"
    native.load_state_dict(ref.state_dict())
    ids = torch.randint(0, cfg["vocab_size"], (B, L), generator=torch.Generator().manual_seed(seed + 1)).cuda()
    got = native(ids)[0]
    torch.cuda.synchronize()
    with torch.no_grad():
        want = ref.double().cuda()(ids)[0]
    return got, want


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name,B,L", [("small", 1, 77), ("small", 3, 20), ("sd15", 2, 77)])
def test_clip_fp32_matches_transformers_float64(cfg_name, B, L):
    pytest.importorskip("transformers")
    from b200edit.clip import SD15_CLIP_CONFIG
    cfg = SMALL_CLIP if cfg_name == "small" else SD15_CLIP_CONFIG
    got, want = _clip_pair(cfg, B, L, seed=B + L)
    check_bars(got, want, 5e-5, f"clip fp32 {cfg_name} B={B} L={L}")


@pytest.mark.gpu
def test_clip_fp32_token_states_ignore_later_tokens():
    """Token t's state is bit-identical when only tokens after t change (causal mask, row-independent GEMMs)."""
    from b200edit.clip import CLIPTextModel
    enc = CLIPTextModel(**SMALL_CLIP, max_batch=2, precision="fp32").init_random(3)
    ids = torch.randint(0, 1000, (2, 77), generator=torch.Generator().manual_seed(4)).cuda()
    ids2 = ids.clone()
    ids2[:, 40:] = 7
    a, b = enc(ids)[0], enc(ids2)[0]
    assert torch.equal(a[:, :40], b[:, :40]) and not torch.equal(a[:, 40:], b[:, 40:])


# ----------------------------------------------------------------------------------------------------- encoders
def _native_vq(cfg, B, precision="fp32", **kw):
    from b200edit.vqmodel import AutoencoderKL, VQModel
    kl = cfg["num_vq_embeddings"] == 0
    args = {k: v for k, v in cfg.items() if not (kl and k == "num_vq_embeddings")}
    return (AutoencoderKL if kl else VQModel)(**args, max_batch=B, with_encoder=True, encoder_precision=precision, **kw)


def _latent(model, x, kl):
    e = model.encode(x)
    return e.latent_dist.mode() if kl else e.latents


ENCODERS = {"small-vq": (SMALL_VQ, 2), "small-kl": (SMALL_KL, 2), "ldm-vq": (LDM_VQ_CONFIG, 2), "sd-kl": (SD_VAE_CONFIG, 1)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ENCODERS))
def test_fp32_encoder_matches_oracle_float64(name):
    """The full LDM VQ encoder runs at 256 x 256 (B = 2), the full SD KL encoder at 512 x 512 (B = 1): their stride-2
    downsamplers pad (0, 1, 0, 1), and their mid-block attention over 4096 tokens runs on the tiled fp32 kernel."""
    cfg, B = ENCODERS[name]
    torch.manual_seed(B + len(name))
    oracle = OracleVQ(**cfg).eval()
    native = _native_vq(cfg, B)
    assert native.encoder_precision == "fp32" and native._enc.precision == "fp32"
    native.load_state_dict(oracle.state_dict())
    kl = cfg["num_vq_embeddings"] == 0
    S = cfg["sample_size"] << (len(cfg["block_out_channels"]) - 1)
    x = torch.randn(B, cfg["out_channels"], S, S, generator=torch.Generator().manual_seed(11)).clamp(-1, 1).cuda()
    got = _latent(native, x, kl)
    torch.cuda.synchronize()
    _no_tf32()
    with torch.no_grad():
        ref = _latent(oracle.double().cuda(), x.double(), kl)
    check_bars(got, ref, 1e-4, f"{name} encoder fp32 B={B}")


# ----------------------------------------------------------------------------------------------------- pipelines
LDM_UNET = dict(sample_size=16, in_channels=3, out_channels=3, block_out_channels=(64, 128), layers_per_block=1,
                down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"),
                attention_head_dim=32, flip_sin_to_cos=True, freq_shift=0, downsample_padding=1)


@pytest.mark.gpu
def test_ldm_fp32_encode_and_inversion_match_float64_chain():
    import ddpm_inversion as dp
    from models import create_diffusion_model
    from oracle import loops, step_math as sm
    from oracle.unet2d import UNet2DModel as OracleUNet
    from test_gpu_pipeline import osched
    T, B, eta = 10, 2, 1.0
    torch.manual_seed(21)
    ounet, ovq = OracleUNet(**LDM_UNET).eval(), OracleVQ(**SMALL_VQ).eval()
    w = create_diffusion_model("ldm", sample_clipping=False, max_batch=B, unet_config=LDM_UNET, vq_config=SMALL_VQ,
                               state_dict=ounet.state_dict(), vq_state_dict=ovq.state_dict(), decoder_grad=False,
                               precision="fp32", encoder_precision="fp32")
    assert w.vqvae.encoder_precision == "fp32" and w.unet.precision == "fp32"
    g = torch.Generator().manual_seed(22)
    img = (torch.rand(B, 3, 32, 32, generator=g) * 2 - 1).cuda()
    noise = torch.randn(T, B, 3, 16, 16, generator=g)          # fp32 draws; the float64 chain takes the same values
    x0 = w.encode(img)
    _, zs, xts = dp.invert(w, x0, num_inference_steps=T, eta=eta, prog_bar=False, noise=noise.cuda())
    noise = noise.double()
    torch.cuda.synchronize()
    _no_tf32()
    ounet, ovq = ounet.double().cuda(), ovq.double().cuda()
    with torch.no_grad():
        x0_ref = ovq.encode(img.double()).latents.cpu()
    check_bars(x0, x0_ref, 1e-4, "ldm encode fp32")
    bar_x0 = 1e-4 * max(1.0, x0_ref.abs().max().item())
    sched = osched("ldm", T, False)
    eps_max = {}

    def eps_fn(x, t):
        with torch.no_grad():
            e = ounet(x.cuda(), torch.tensor(t))["sample"].cpu()
        eps_max[t] = max(eps_max.get(t, 0.0), e.abs().max().item())
        return e

    refs = [loops.invert_ddpm(sched, eps_fn, x0_ref[b:b + 1], noise[:, b], eta) for b in range(B)]
    xts_ref = torch.stack([r[2] for r in refs], 1)
    zs_ref = torch.stack([r[1] for r in refs], 1)
    err_x = (xts[:T].cpu().double() - xts_ref[:T]).abs().max().item()
    print(f"ldm inversion xts: max-abs {err_x:.3e} (encoder bar {bar_x0:.3e})")
    assert err_x <= bar_x0, (err_x, bar_x0)
    assert torch.equal(zs[-1].cpu(), torch.zeros_like(zs[-1].cpu()))
    for idx in range(T - 1):
        t = int(sched.timesteps[idx])
        c = sm.step_coeffs(sched, t)
        sa, sb, sp = float(c.sqrt_a_t), float(c.sqrt_b_t), float(c.sqrt_a_prev)
        sigma = float(c.variance) ** 0.5
        cdir = (1 - float(c.a_prev) - eta * float(c.variance)) ** 0.5
        de = 1e-4 * max(1.0, eps_max[t])
        mag = (xts_ref[idx + 1].abs().max().item() + sp * (xts_ref[idx].abs().max().item() + sb * eps_max[t]) / sa
               + cdir * eps_max[t])
        bar_z = (abs(cdir - sp * sb / sa) * de + 8 * EPS32 * mag) / (eta * sigma)
        err_z = (zs[idx].cpu().double() - zs_ref[idx]).abs().max().item()
        print(f"ldm inversion zs[{idx}] (t={t}): max-abs {err_z:.3e} (bar {bar_z:.3e}, |dz/de| "
              f"{abs(cdir - sp * sb / sa) / (eta * sigma):.2f})")
        assert err_z <= bar_z, (idx, err_z, bar_z)


@pytest.mark.gpu
def test_sd_fp32_prompt_conditioning_matches_float64_chain():
    pytest.importorskip("transformers")
    from transformers import CLIPTextConfig, CLIPTextModel as RefCLIP
    from diffusion_utils import prep_text
    from models import create_diffusion_model
    from oracle.unet2d_condition import UNet2DConditionModel as OracleCond
    from test_gpu_unet_cond import SMALL, FakeTokenizer
    clip_cfg = dict(SMALL_CLIP, hidden_size=SMALL["cross_attention_dim"], intermediate_size=4 * SMALL["cross_attention_dim"])
    vae = dict(latent_channels=4, out_channels=3, block_out_channels=(64, 128), layers_per_block=1, norm_num_groups=32,
               norm_eps=1e-6, sample_size=16)
    torch.manual_seed(31)
    ocond = OracleCond(**SMALL).eval()
    oclip = RefCLIP(CLIPTextConfig(hidden_act="quick_gelu", attn_implementation="eager", **clip_cfg)).eval()
    w = create_diffusion_model("sd", sample_clipping=False, max_batch=1, unet_config=SMALL, vq_config=vae,
                               state_dict=ocond.state_dict(), decoder_grad=False, tokenizer=FakeTokenizer(),
                               text_encoder_config=clip_cfg, text_encoder_state_dict=oclip.state_dict(), precision="fp32",
                               encoder_precision="fp32")
    assert w.text_encoder.precision == "fp32" and w.vae.encoder_precision == "fp32"
    prompt, s, t = "a photo of a face", 3.5, 500
    emb = prep_text(w, prompt)
    lat = torch.randn(1, 4, 16, 16, generator=torch.Generator().manual_seed(32)).cuda()
    with torch.no_grad():
        both = w.unet(sample=torch.cat([lat] * 2), timestep=torch.tensor(t), encoder_hidden_states=emb)["sample"]
    from diffusion_utils import get_noise_pred
    eps = get_noise_pred(w, lat, torch.tensor(t), emb, s)
    torch.cuda.synchronize()
    _no_tf32()
    ids = FakeTokenizer()(["", prompt]).input_ids.cuda()
    with torch.no_grad():
        emb_ref = oclip.double().cuda()(ids)[0]
        both_ref = ocond.double().cuda()(torch.cat([lat] * 2).double(), torch.tensor(t),
                                         encoder_hidden_states=emb_ref)["sample"]
    check_bars(emb, emb_ref, 5e-5, "sd prep_text (clip fp32)")
    bars = []
    for i, half in enumerate(("uncond", "cond")):
        check_bars(both[i:i + 1], both_ref[i:i + 1], 5e-5, f"sd cfg noise prediction, {half} half")
        bars.append(1e-4 * max(1.0, both_ref[i].abs().max().item()))
    u, c = both_ref.chunk(2)
    ref = u + s * (c - u)
    err = (eps.double() - ref).abs().max().item()
    bar = (1 + 2 * s) * max(bars)
    print(f"sd cfg combination (s={s}): max-abs {err:.3e} (bar {bar:.3e})")
    assert err <= bar, (err, bar)


# ----------------------------------------------------------------------------------------------------- defaults
@pytest.mark.gpu
def test_defaults_keep_the_16bit_encoders():
    from b200edit import _C
    from b200edit.clip import CLIPTextModel
    from b200edit.vqmodel import VQModel
    from models import create_diffusion_model
    fast = _C.fast_precision()
    assert CLIPTextModel(**SMALL_CLIP, max_batch=1).precision == fast
    vq = VQModel(**SMALL_VQ, max_batch=1, with_encoder=True)
    assert vq.encoder_precision == fast and vq._enc.precision == fast and vq.precision == fast
    # precision="fp32" selects the fp32-accurate UNet and decoder, not the encoder
    w = create_diffusion_model("ldm", max_batch=1, unet_config=LDM_UNET, vq_config=SMALL_VQ, decoder_grad=False,
                               precision="fp32")
    assert w.vqvae.precision == "fp32" and w.vqvae.encoder_precision == fast and w.vqvae._enc.precision == fast
    for bad in ("fp8", "bf16" if fast == "fp16" else "fp16"):
        with pytest.raises(ValueError):
            create_diffusion_model("ldm", max_batch=1, unet_config=LDM_UNET, vq_config=SMALL_VQ, encoder_precision=bad)
        with pytest.raises(ValueError):
            CLIPTextModel(**SMALL_CLIP, max_batch=1, precision=bad)
        with pytest.raises(ValueError):
            VQModel(**SMALL_VQ, max_batch=1, with_encoder=True, encoder_precision=bad)


def test_factory_refuses_an_unknown_encoder_precision_before_building():
    """No device needed: the refusal comes before any engine is created."""
    from models import create_diffusion_model
    with pytest.raises(ValueError, match="encoder_precision"):
        create_diffusion_model("ldm", encoder_precision="fp8")

