"""Every attention path of the engine against a float64 reference, at the models' shapes and masking edges.

`ops.attention_f16` runs the engine's own launch sequence of one path (`b2e_attention_f16`): fused tcgen05 attention
(8 or 4 softmax warps), materialised multi-head attention, single-head GEMM attention, the CUDA-core kernel and the two
fp32-accurate kernels.  The reference takes the exact 16-bit inputs the kernel sees (hi + lo for the fp32 paths) and
computes softmax(Q K^T / sqrt(d)) V in float64, one (image, head) at a time, with the same key and causal masks.

Inputs make masking faults visible.  Key and value rows at and after `valid_k` hold +-30 (large logits, large values).
The last valid key gets a dominant scaled logit L (channel 0 of every head is a bias channel: q = 4, k = L sqrt(d) / 4),
its values are +-(2..4), and its other key channels are zero, so L is its exact logit.  Without a causal mask the other
valid value rows lean the other way (-2.5 sign(dominant row) + 0.25 N(0, 1)), so dropping the dominant key moves the
output by up to about 1.5 R.  In causal cases query i is aligned with keys i and i + 1 (logits of about L / 2 each), and
a ramp adds 0.25 (j - i) to the logit of key j: every future key outweighs the diagonal, the more the further it lies
past it, while the diagonal leads the keys a row may see.  Future keys of one row are valid keys of later rows, so their
value rows stay ordinary.  Where the padded paths add zero key rows (fewer than 128 tokens, no masked key), the
dominant logit is -5 and the other valid logits are about -13 (unit-variance q in both regimes: the largest |logit|
stays near 16, where even the bf16 bar of the 16-bit-score paths is below a fifth of R), so an admitted zero-padded key
(logit 0) would outweigh them all.  Three regimes: "unit" (unit-variance q and k, L = 10), "saturated" (q scaled by 2,
L = 30: the largest scaled logit is about 30) and "zero" (q = 0: the output is the mean of the valid V rows).

Tolerances (u = unit roundoff of the build's 16-bit type: 2^-11 fp16, 2^-8 bf16; e = 2^-24; R = max |V| over the valid
keys; Z = max |scaled logit| over the unmasked scores):
  fused:  the kernel rounds P to 16 bit and divides by the sum of the ROUNDED P, so O is an exact convex combination with
          weights perturbed by at most 2u relative: |dO| <= 2uR; the 16-bit output adds uR; fp32 logits and the fp32 P V
          sums stay below one more uR.                                                              bar = 4 u R
  materialised / single-head:  the scores are stored in 16 bit BEFORE scaling, so each scaled logit carries an error
          up to u|z| <= uZ; a weight perturbation of that size moves O by up to 2uZR.  P is stored in 16 bit after the
          normalisation (the P V sum no longer adds to exactly 1): uR; the output rounding: uR.   bar = (2Z + 4) u R
  CUDA core:  fp32 scores, softmax and P V, one 16-bit rounding of the output.           bar = (u + e (8Z + 64)) R
  fp32 split / tiled:  fp32 arithmetic.  The fp32 scores carry a few ulps of |z| (4eZ relative on a weight, 8eZR on O)
          and the fp32 sums over up to 4096 keys about sqrt(4096) e R.  The output is stored as hi + lo: |O - hi| <= u|O|,
          and rounding lo costs u|O - hi| <= u^2 R (2^-22 R in fp16, but 2^-16 R in bf16, where hi + lo holds only 16
          mantissa bits).                                                               bar = (e (8Z + 64) + u^2) R
          (at Z <= 30 this is at least 100x below the fused bar of either build; the test checks it.)
Every case prints its measured error beside its bar.  `test_bars_resolve_masking_faults` shows on the CPU, in float64,
that each bar sees the faults this file is meant to catch: a reference with one extra masked key admitted, with the last
valid key dropped, with the causal diagonal moved by one or the causal mask gone, or (fp32 paths) without the lo plane differs from the true
reference by at least 5x the bar.
"""
import math
from dataclasses import dataclass
from typing import Optional

import pytest
import torch

from b200edit import _C, ops
from b200edit._C import B2EError

EPS32 = 2.0 ** -24
A_BIAS = 4.0      # q value of the bias channel
R_DOM = 4.0       # |value| of the dominant key's value row
BIG = 30.0        # |k| and |v| of masked key rows
V_REST, V_NOISE = 2.5, 0.25   # non-causal cases: the other valid value rows are -V_REST * sign(dominant row) + V_NOISE * N(0, 1)
RAMP = 0.25       # causal cases: logit step per key position
REGIMES = ("unit", "saturated", "zero")


def unit_roundoff() -> float:
    return 2.0 ** -8 if ops.act_dtype() == torch.bfloat16 else 2.0 ** -11


@dataclass(frozen=True)
class Case:
    name: str
    path: str
    B: int
    H: int
    W: int
    heads: int
    d: int
    P: int                      # channel block width: pitch of out, of the q / k / v blocks of the packed tensors
    Tk: Optional[int] = None    # cross-attention: key rows of the kv tensor (None: self-attention over H*W tokens)
    valid_k: Optional[int] = None
    causal: bool = False
    sw: int = 8

    @property
    def Tq(self):
        return self.H * self.W

    @property
    def T_keys(self):
        return self.Tk if self.Tk is not None else self.Tq

    @property
    def vk(self):
        return self.valid_k if self.valid_k is not None else self.T_keys

    @property
    def padded_keys(self):
        """the fused / materialised paths pad the keys to 128-row blocks with zero rows (masked by valid_k)"""
        return self.path in ("fused", "materialised") and self.T_keys % 128 != 0

    def __str__(self):
        return self.name


def _mh(path, name, B, H, W, heads, d, P=None, sw=8, **kw):
    return Case(f"{path}-sw{sw}-{name}" if path == "fused" else f"{path}-{name}", path, B, H, W, heads, d,
                P or heads * d, sw=sw, **kw)


CASES = [
    # LDM-CelebAHQ: 32-channel heads; the 672-channel level has a pitch of 704 (zero tail)
    _mh("fused", "ldm-14h-1024", 2, 32, 32, 14, 32),
    _mh("fused", "ldm-21h-256-pitch704", 2, 16, 16, 21, 32, P=704),
    _mh("fused", "ldm-28h-64", 2, 8, 8, 28, 32),
    # SD 1.5 self-attention: d = 40 / 80 / 160 (D = 64 / 128 / 192)
    _mh("fused", "sd-d40-4096", 1, 64, 64, 8, 40),
    _mh("fused", "sd-d80-1024", 2, 32, 32, 8, 80),
    _mh("fused", "sd-d160-256", 2, 16, 16, 8, 160),
    _mh("fused", "sd-d160-64", 2, 8, 8, 8, 160),
    # SD cross-attention over 128 text rows, valid_k text tokens
    *[_mh("fused", f"sd-cross-d80-vk{vk}", 1, 32, 32, 8, 80, Tk=128, valid_k=vk) for vk in (1, 64, 65, 77, 128)],
    _mh("fused", "sd-cross-d40-4096-vk77", 1, 64, 64, 8, 40, Tk=128, valid_k=77),
    *[_mh("fused", f"sd-cross-d160-256-vk{vk}", 2, 16, 16, 8, 160, Tk=128, valid_k=vk) for vk in (1, 65)],
    _mh("fused", "sd-cross-d160-64-vk77", 2, 8, 8, 8, 160, Tk=128, valid_k=77),
    # CLIP text encoder: causal, 12 heads of 64, 128 token rows, valid_k tokens
    *[_mh("fused", f"clip-causal-vk{vk}", 2, 1, 128, 12, 64, valid_k=vk, causal=True) for vk in (1, 77, 128)],
    # persistent grid of min(items, 148) CTAs: fewer items, exactly 148, 149 (one CTA walks a second item), 3 - 4 per CTA
    _mh("fused", "grid-2-items", 1, 1, 128, 2, 64),
    _mh("fused", "grid-148-items", 37, 1, 128, 4, 64),
    _mh("fused", "grid-149-items", 1, 1, 128, 149, 8),
    _mh("fused", "grid-512-items", 2, 64, 64, 8, 40),
    # D = 192 (single-stage K/V ring) with one key block and with 32
    _mh("fused", "d192-one-key-block", 1, 1, 128, 2, 160),
    _mh("fused", "d192-32-key-blocks", 1, 64, 64, 1, 160),
    # the one-thread-per-row softmax layout
    _mh("fused", "ldm-14h-1024", 2, 32, 32, 14, 32, sw=4),
    _mh("fused", "sd-cross-d80-vk65", 1, 32, 32, 8, 80, sw=4, Tk=128, valid_k=65),
    _mh("fused", "clip-causal-vk77", 2, 1, 128, 12, 64, sw=4, valid_k=77, causal=True),
    _mh("fused", "d192-32-key-blocks", 1, 64, 64, 1, 160, sw=4),
    _mh("fused", "sd-d160-64", 2, 8, 8, 8, 160, sw=4),
    # materialised multi-head attention (head_dim > 192, or B2E_FLASH=0)
    _mh("materialised", "ldm-14h-1024", 2, 32, 32, 14, 32),
    _mh("materialised", "ldm-21h-256-pitch704", 2, 16, 16, 21, 32, P=704),
    _mh("materialised", "sd-d40-4096", 1, 64, 64, 8, 40),
    _mh("materialised", "sd-d160-64", 2, 8, 8, 8, 160),
    *[_mh("materialised", f"sd-cross-d80-vk{vk}", 1, 32, 32, 8, 80, Tk=128, valid_k=vk) for vk in (1, 64, 65, 77, 128)],
    _mh("materialised", "d256-2h-256", 2, 16, 16, 2, 256),
    # single-head GEMM attention: DDPM-256 (C = 512, T = 256, batch 8) and the decoder mid block (T = 4096)
    _mh("single_head", "ddpm-c512-256", 8, 16, 16, 1, 512),
    _mh("single_head", "decoder-mid-c512-4096", 1, 64, 64, 1, 512),
    # CUDA-core kernel: 4-query blocks when 16-query blocks cannot fill the chip
    _mh("cuda_core", "q4-d40", 1, 16, 16, 8, 40),
    _mh("cuda_core", "q16-d40", 2, 32, 32, 8, 40),
    _mh("cuda_core", "q4-d128", 1, 16, 16, 4, 128),
    _mh("cuda_core", "q16-d128", 2, 32, 32, 2, 128),
    _mh("cuda_core", "q4-d512", 1, 8, 8, 1, 512),
    _mh("cuda_core", "q16-d512", 4, 32, 32, 1, 512),
    _mh("cuda_core", "q16-ldm-21h-pitch704", 2, 16, 16, 21, 32, P=704),
    # fp32-accurate kernels
    _mh("fp32_split", "ddpm-c512-256", 2, 16, 16, 1, 512),
    _mh("fp32_split", "ldm-21h-256-pitch704", 2, 16, 16, 21, 32, P=704),
    _mh("fp32_split", "d512-1024", 1, 32, 32, 1, 512),
    _mh("fp32_tiled", "sd-d40-4096", 1, 64, 64, 8, 40),
    _mh("fp32_tiled", "decoder-mid-c512-4096", 1, 64, 64, 1, 512),
    _mh("fp32_tiled", "cross-d80-tq1000-vk77", 1, 25, 40, 8, 80, Tk=128, valid_k=77),
    *[_mh("fp32_tiled", f"cross-d160-vk{vk}", 2, 16, 16, 8, 160, Tk=128, valid_k=vk) for vk in (1, 65)],
    _mh("fp32_tiled", "self-tq100-vk77", 2, 10, 10, 2, 64, valid_k=77),
]


# ----------------------------------------------------------------------------------------------------- inputs
def make_inputs(c: Case, regime: str, seed: int = 0):
    """float64 q (B, Tq, heads, d), k / v (B, Tk, heads, d) before the kernel's 16-bit rounding (see the module docstring)."""
    g = torch.Generator().manual_seed(seed)
    B, Tq, Tk, h, d, vk = c.B, c.Tq, c.T_keys, c.heads, c.d, c.vk
    f64 = torch.float64
    q = torch.randn(B, Tq, h, d, generator=g, dtype=f64)
    k = torch.randn(B, Tk, h, d, generator=g, dtype=f64)
    v = torch.randn(B, Tk, h, d, generator=g, dtype=f64)
    signs_v = torch.randn(B, Tk, h, d, generator=g, dtype=f64).sign()
    signs_k = torch.randn(B, Tk, h, d, generator=g, dtype=f64).sign()
    s_dom = signs_v[:, vk - 1:vk]
    if not c.causal:   # the other valid value rows lean against the dominant one
        v = -V_REST * s_dom + V_NOISE * v
    if regime == "zero":
        q.zero_()
    else:
        L = 10.0 if regime == "unit" else 30.0
        pad_shift = c.padded_keys and vk == Tk
        q *= 1.0 if regime == "unit" or pad_shift else 2.0
        if c.causal:
            # query i aligned with keys i and i + 1 (logits of about L / 2 each), channels 3 ..
            a = 0.5 * L / math.sqrt(d)
            nxt = torch.cat([k[:, 1:Tq, :, 3:], torch.zeros_like(k[:, :1, :, 3:])], dim=1)
            q[..., 3:] += a * (k[:, :Tq, :, 3:] + nxt)
            # ramp, channels 1 and 2: + RAMP * (j - i) on the logit of key j for query i, so that every future key
            # outweighs the diagonal, the more the further it lies past it
            cr = math.sqrt(RAMP * Tq * math.sqrt(d))
            pos = torch.arange(max(Tq, Tk), dtype=f64) / Tq
            q[..., 1], q[..., 2] = cr, -cr * pos[:Tq, None]
            k[..., 1], k[..., 2] = cr * pos[:Tk, None], cr
        q[..., 0] = A_BIAS
        bias = torch.zeros(Tk, dtype=f64)
        bias[vk - 1] = L
        if pad_shift:   # an admitted zero-padded key (logit 0) would outweigh every valid key
            bias[:vk] = -13.0
            bias[vk - 1] = -5.0
        k[..., 0] = bias[:, None] * math.sqrt(d) / A_BIAS
        k[:, vk - 1, :, 1:] = 0.0
    # |v| in (R_DOM / 2, R_DOM]: not representable in 16 bit, so the lo plane of the fp32 paths carries the dominant row too
    v[:, vk - 1] = R_DOM * s_dom[:, 0] * (1.0 - 0.5 * torch.rand(B, h, d, generator=g, dtype=f64))
    k[:, vk:] = BIG * signs_k[:, vk:]
    v[:, vk:] = BIG * signs_v[:, vk:]
    return q, k, v


def kernel_view(x64: torch.Tensor, path: str):
    """The values the kernel computes with: 16-bit rounding, or hi + lo of the fp32-accurate split."""
    if path.startswith("fp32"):
        x32 = x64.float()
        hi = x32.to(ops.act_dtype())
        lo = (x32 - hi.float()).to(ops.act_dtype())
        return hi.double() + lo.double(), hi.double()
    r = x64.to(ops.act_dtype()).double()
    return r, r


# ----------------------------------------------------------------------------------------------------- reference
def allowed_keys(c: Case, rows: torch.Tensor, n_keys: int, fault: Optional[str] = None):
    """[len(rows), n_keys] bool mask of the keys each query row attends to, optionally with one of the masking faults."""
    j = torch.arange(n_keys, device=rows.device)[None, :]
    i = rows[:, None]
    lim = torch.full_like(i, c.vk)
    if c.causal:
        shift = {"diag_next": 2, "diag_prev": 0, "no_causal": n_keys}.get(fault, 1)
        lim = torch.minimum(lim, i + shift)
    m = j < lim
    if fault == "extra":
        m = m | (j == c.vk)
    elif fault == "drop_last":
        m = m & (j != c.vk - 1)
    return m


def reference(c: Case, q, k, v, rows=None, fault=None, images=None, heads=None):
    """float64 softmax(q k^T / sqrt(d), masked) v for the given query rows, one (image, head) at a time.
    Returns out [len(images), len(rows), len(heads), d] and the max |scaled logit| over the unmasked scores.  Rows
    whose fault leaves no key are NaN."""
    Tq, d = q.shape[1], c.d
    rows = torch.arange(Tq, device=q.device) if rows is None else rows.to(q.device)
    images = range(q.shape[0]) if images is None else images
    heads = range(c.heads) if heads is None else heads
    if fault == "extra" and c.vk == k.shape[1]:   # the admitted key is a zero-padded row of the padded paths
        k = torch.cat([k, torch.zeros_like(k[:, :1])], dim=1)
        v = torch.cat([v, torch.zeros_like(v[:, :1])], dim=1)
    allow = allowed_keys(c, rows, k.shape[1], fault)
    scale = 1.0 / math.sqrt(d)
    out = torch.empty(len(images), len(rows), len(heads), d, dtype=q.dtype, device=q.device)
    zmax = 0.0
    for bi, b in enumerate(images):
        for hi, hh in enumerate(heads):
            s = (q[b, rows, hh] @ k[b, :, hh].T) * scale
            zmax = max(zmax, s.abs().masked_fill(~allow, 0).max().item())
            p = torch.softmax(s.masked_fill(~allow, -math.inf), dim=-1)
            out[bi, :, hi] = p @ v[b, :, hh]
    return out, zmax


def value_range(c: Case, v):
    return v[:, :c.vk].abs().max().item()


def bar(path: str, u: float, R: float, Z: float) -> float:
    if path == "fused":
        return 4 * u * R
    if path in ("materialised", "single_head"):
        return (2 * Z + 4) * u * R
    if path == "cuda_core":
        return (u + EPS32 * (8 * Z + 64)) * R
    return (EPS32 * (8 * Z + 64) + u * u) * R


def faults_for(c: Case):
    # with one valid key, dropping it leaves an empty softmax: the finiteness check of the GPU test covers that
    f = ["drop_last"] if c.vk > 1 else []
    if c.vk < c.T_keys or c.padded_keys:
        f.append("extra")
    if c.causal and c.vk > 1:
        f += ["diag_next", "diag_prev", "no_causal"]
    if c.path.startswith("fp32"):
        f.append("no_lo")
    return f


# ----------------------------------------------------------------------------------------------------- CPU checks
def _probe_rows(Tq: int, g: torch.Generator):
    fixed = {0, 1, 2, 31, 32, 63, 64, 65, 76, 77, 78, 127, 128, 129, Tq - 2, Tq - 1}
    rnd = torch.randint(0, Tq, (24,), generator=g).tolist()
    return torch.tensor(sorted(r for r in fixed | set(rnd) if 0 <= r < Tq))


def _logit_max(c: Case, q, k):
    """max |scaled logit| over the unmasked scores, float32 on the CPU, rounded up by 0.1 %"""
    q32, k32 = q.float(), k.float()
    allow = allowed_keys(c, torch.arange(c.Tq), k.shape[1])
    z = 0.0
    for b in range(c.B):
        for hh in range(c.heads):
            s = (q32[b, :, hh] @ k32[b, :, hh].T) / math.sqrt(c.d)
            z = max(z, s.abs().masked_fill(~allow, 0).max().item())
    return z * 1.001


@pytest.mark.parametrize("regime", ("unit", "saturated"))
@pytest.mark.parametrize("case", CASES, ids=str)
def test_bars_resolve_masking_faults(case, regime):
    """The reference with each masking fault (or without the lo plane) differs from the true reference by at least 5x the
    case's bar, on a probe of query rows of the first and last image / head (a lower bound of the full difference)."""
    torch.set_num_threads(max(torch.get_num_threads(), 1))
    u = unit_roundoff()
    q, k, v = make_inputs(case, regime)
    qr, qhi = kernel_view(q, case.path)
    kr, khi = kernel_view(k, case.path)
    vr, vhi = kernel_view(v, case.path)
    R, Z = value_range(case, vr), _logit_max(case, qr, kr)
    b = bar(case.path, u, R, Z)
    if case.path.startswith("fp32"):
        assert 100 * b <= 4 * u * R, (b, 4 * u * R)
    rows = _probe_rows(case.Tq, torch.Generator().manual_seed(1))
    sel = dict(rows=rows, images=sorted({0, case.B - 1}), heads=sorted({0, case.heads - 1}))
    ref, _ = reference(case, qr, kr, vr, **sel)
    for fault in faults_for(case):
        if fault == "no_lo":
            alt, _ = reference(case, qhi, khi, vhi, **sel)
        else:
            alt, _ = reference(case, qr, kr, vr, fault=fault, **sel)
        diff = (alt - ref).abs().nan_to_num(0.0).max().item()
        print(f"{case} {regime} {fault}: fault moves the output by {diff:.3e} = {diff / b:.0f} x bar {b:.3e}")
        assert diff >= 5 * b, (fault, diff, b)


def test_zero_queries_give_the_mean_of_the_valid_values():
    """q = 0: every unmasked key has weight 1 / n, the reference is the mean of the valid value rows (causal: of the
    first min(i + 1, valid_k) rows)."""
    c = next(x for x in CASES if x.causal and x.vk == 77)
    q, k, v = make_inputs(c, "zero")
    ref, _ = reference(c, q, k, v, images=[0], heads=[0])
    csum = v[0, :, 0].cumsum(0)
    n = torch.clamp(torch.arange(c.Tq, dtype=torch.float64) + 1, max=c.vk)
    want = csum[n.long() - 1] / n[:, None]
    assert torch.allclose(ref[0, :, 0], want, rtol=0, atol=1e-12)


def test_attention_hook_validates_arguments_on_the_host():
    """Null pointers and every unsupported combination are refused before anything touches memory or the device."""
    lib = _C.lib
    fake = 1 << 20   # never dereferenced: every call below is refused on the host

    def call(q=fake, qp=192, qc=0, kv=fake, kp=192, kc=64, vc=128, out=fake, op=64, B=1, H=8, W=8, Tk=64, vk=64, heads=1,
             d=64, causal=0, path=0, sw=8):
        return lib.b2e_attention_f16(q, qp, qc, kv, kp, kc, vc, out, op, B, H, W, Tk, vk, heads, d, causal, path, sw, None)

    assert call(q=None) == -1 and b"null pointer" in lib.b2e_last_error()
    assert call(kv=None) == -1 and call(out=None) == -1
    assert call(path=6) == -1 and b"unknown path" in lib.b2e_last_error()
    assert call(vk=0) == -1 and b"valid_k" in lib.b2e_last_error()
    assert call(vk=65) == -1 and b"valid_k" in lib.b2e_last_error()
    assert call(sw=6) == -1
    assert call(kc=160) == -1                                   # key window past the pitch
    assert call(op=32) == -1                                    # out pitch below heads * d
    for path in (1, 2, 3, 4, 5):                                # causal on a non-fused path
        assert call(causal=1, path=path) == -2 and b"causal" in lib.b2e_last_error()
    for path in (2, 3, 4):                                      # packed-qkv paths: q and k / v in different tensors
        assert call(kv=fake + 4096, path=path) == -2 and b"packed" in lib.b2e_last_error()
        assert call(vk=63, path=path) == -2                     # ... and no key mask
    assert call(path=2, heads=2, d=32) == -2                    # single-head path with two heads
    assert call(path=2, H=8, W=8) == -2                         # 64 tokens: no 128-row GEMM tiling
    assert call(qp=3 * 256, kp=3 * 256, kc=256, vc=512, op=256, d=256, path=0) == -2   # head_dim > 192 on the fused path
    assert b"head_dim" in lib.b2e_last_error()
    assert call(H=10, W=20, Tk=200, vk=200) == -2               # 200 tokens: not a multiple of 128
    assert b"tokens" in lib.b2e_last_error()
    assert call(H=10, W=20, Tk=200, vk=200, path=1) == -2


# ----------------------------------------------------------------------------------------------------- GPU checks
def _layout(c: Case, q, k, v, dtype):
    """The engine's operand layout: self-attention reads one packed [q | k | v] tensor of 3P channels per token,
    cross-attention a q tensor of P channels and a [k | v] tensor of 2P channels; zero channel tails."""
    B, Tq, Tk, C, P = c.B, c.Tq, c.T_keys, c.heads * c.d, c.P
    if c.Tk is None:
        qkv = torch.zeros(B, Tq, 3 * P, dtype=dtype)
        qkv[..., :C] = q.reshape(B, Tq, C).to(dtype)
        qkv[..., P:P + C] = k.reshape(B, Tk, C).to(dtype)
        qkv[..., 2 * P:2 * P + C] = v.reshape(B, Tk, C).to(dtype)
        qkv = qkv.cuda()
        return qkv, qkv, dict(q_col=0, k_col=P, v_col=2 * P)
    qt = torch.zeros(B, Tq, P, dtype=dtype)
    qt[..., :C] = q.reshape(B, Tq, C).to(dtype)
    kvt = torch.zeros(B, Tk, 2 * P, dtype=dtype)
    kvt[..., :C] = k.reshape(B, Tk, C).to(dtype)
    kvt[..., P:P + C] = v.reshape(B, Tk, C).to(dtype)
    return qt.cuda(), kvt.cuda(), dict(q_col=0, k_col=0, v_col=P)


def run_case(c: Case, q, k, v, out=None):
    fp32 = c.path.startswith("fp32")
    qt, kvt, cols = _layout(c, q, k, v, torch.float32 if fp32 else ops.act_dtype())
    if out is None:
        out = torch.full((c.B, c.Tq, (3 if fp32 else 1) * c.P), float("nan"), dtype=ops.act_dtype(), device="cuda")
    return ops.attention_f16(qt, kvt, hw=(c.H, c.W), heads=c.heads, head_dim=c.d, out_pitch=c.P, valid_k=c.valid_k,
                             causal=c.causal, path=c.path, softmax_warps=c.sw, out=out, **cols)


@pytest.mark.gpu
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("case", CASES, ids=str)
def test_attention_path_matches_float64(case, regime):
    torch.cuda.set_device(0)
    u = unit_roundoff()
    q, k, v = make_inputs(case, regime)
    out = run_case(case, q, k, v)
    torch.cuda.synchronize()
    C, P = case.heads * case.d, case.P
    planes = [out[..., i * P:(i + 1) * P] for i in range(3)] if case.path.startswith("fp32") else [out]
    for pl in planes:   # the consumer convolutions read the whole pitch: its tail must be exactly zero
        tail = pl[..., C:]
        assert tail.numel() == 0 or (tail == 0).all().item(), "pitch tail not zeroed"
    got = (ops.merge_planes(out) if case.path.startswith("fp32") else out.float())[..., :C]
    assert torch.isfinite(got).all().item(), "unwritten (NaN) or non-finite output"
    qr, kr, vr = (kernel_view(x, case.path)[0].cuda() for x in (q, k, v))
    ref, Z = reference(case, qr, kr, vr)
    ref = ref.reshape(case.B, case.Tq, C)
    err = (got.double() - ref).abs().max().item()
    R = value_range(case, vr)
    b = bar(case.path, u, R, Z)
    print(f"{case} {regime} [{ops.act_dtype()}]: max err {err:.3e}  bar {b:.3e}  ({err / b:.3f} of the bar; R {R:.2f} Z {Z:.1f})")
    assert err <= b, (err, b)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in CASES if c.path == "fused"], ids=str)
def test_fused_attention_is_deterministic(case):
    torch.cuda.set_device(0)
    q, k, v = make_inputs(case, "unit", seed=3)
    a = run_case(case, q, k, v)
    b = run_case(case, q, k, v)
    assert torch.equal(a, b)


@pytest.mark.gpu
def test_unsupported_combinations_raise_and_launch_nothing():
    torch.cuda.set_device(0)
    dt = ops.act_dtype()
    qkv = torch.zeros(1, 256, 3 * 64, dtype=dt, device="cuda")
    qt = torch.zeros(1, 256, 64, dtype=dt, device="cuda")
    kvt = torch.zeros(1, 256, 128, dtype=dt, device="cuda")
    qkv32 = torch.zeros(1, 256, 3 * 64, device="cuda")
    big = torch.zeros(1, 256, 3 * 256, dtype=dt, device="cuda")
    odd = torch.zeros(1, 200, 3 * 64, dtype=dt, device="cuda")
    self_cols = dict(q_col=0, k_col=64, v_col=128, out_pitch=64)
    bad = [
        ("causal materialised", dict(q=qkv, kv=qkv, hw=(16, 16), heads=1, head_dim=64, causal=True, path="materialised", **self_cols)),
        ("causal single-head", dict(q=qkv, kv=qkv, hw=(16, 16), heads=1, head_dim=64, causal=True, path="single_head", **self_cols)),
        ("causal CUDA core", dict(q=qkv, kv=qkv, hw=(16, 16), heads=1, head_dim=64, causal=True, path="cuda_core", **self_cols)),
        ("causal fp32 split", dict(q=qkv32, kv=qkv32, hw=(16, 16), heads=1, head_dim=64, causal=True, path="fp32_split", **self_cols)),
        ("causal fp32 tiled", dict(q=qkv32, kv=qkv32, hw=(16, 16), heads=1, head_dim=64, causal=True, path="fp32_tiled", **self_cols)),
        ("valid_k 0", dict(q=qkv, kv=qkv, hw=(16, 16), heads=1, head_dim=64, valid_k=0, **self_cols)),
        ("valid_k > Tk", dict(q=qkv, kv=qkv, hw=(16, 16), heads=1, head_dim=64, valid_k=257, **self_cols)),
        ("fused head_dim 256", dict(q=big, kv=big, hw=(16, 16), heads=1, head_dim=256, q_col=0, k_col=256, v_col=512,
                                    out_pitch=256)),
        ("200 tokens fused", dict(q=odd, kv=odd, hw=(10, 20), heads=1, head_dim=64, **self_cols)),
        ("200 tokens materialised", dict(q=odd, kv=odd, hw=(10, 20), heads=1, head_dim=64, path="materialised", **self_cols)),
        ("200 tokens single-head", dict(q=odd, kv=odd, hw=(10, 20), heads=1, head_dim=64, path="single_head", **self_cols)),
        ("split q / kv single-head", dict(q=qt, kv=kvt, hw=(16, 16), heads=1, head_dim=64, q_col=0, k_col=0, v_col=64,
                                          out_pitch=64, path="single_head")),
        ("split q / kv CUDA core", dict(q=qt, kv=kvt, hw=(16, 16), heads=1, head_dim=64, q_col=0, k_col=0, v_col=64,
                                        out_pitch=64, path="cuda_core")),
        ("split q / kv fp32 split", dict(q=qkv32[..., :64].contiguous(), kv=qkv32[..., :128].contiguous(), hw=(16, 16), heads=1,
                                         head_dim=64, q_col=0, k_col=0, v_col=64, out_pitch=64, path="fp32_split")),
        ("masked keys CUDA core", dict(q=qkv, kv=qkv, hw=(16, 16), heads=1, head_dim=64, valid_k=100, path="cuda_core", **self_cols)),
    ]
    for what, kw in bad:
        n0 = _C.launch_count()
        with pytest.raises(B2EError):
            ops.attention_f16(**kw)
        torch.cuda.synchronize()
        assert _C.launch_count() == n0, f"{what}: launched before refusing"
