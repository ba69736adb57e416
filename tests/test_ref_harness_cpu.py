"""The config-2 harness of the reference arm (oracle/ref_harness.py: the reference's OWN diffusion_loop / get_noise_pred /
get_variance_noise / reverse_step / AttrFunc.apply from baseline/_ref/src, composed in the order of
src/SegDiffEditPipeline.py:248-296) must agree BIT-EXACTLY with the oracle loop the GPU parity tests check the CUDA
path against (oracle.loops.guided_edit_loop, mode="ddpm") - this pins the timed path's checker to the unmodified
reference.  The live comparison runs in a subprocess (the reference's bare module names collide with the drop-in
package's) wherever baseline/_ref/src is installed.

Everywhere, the oracle loop is checked against tests/golden/ref_harness.npz: the noise predictions of every step and the
final samples of the same seeded cases.  That file was recorded from the oracle loop (``python
tests/test_ref_harness_cpu.py``) where the unmodified reference could not be run; the live comparison is what ties it to
the reference.  The recorded predictions are replayed (teacher forcing), so the bit-exact check of the step / guidance /
Tskip-window arithmetic does not depend on how the host's convolution kernels sum."""
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden", "ref_harness.npz")
T, TSKIP, S = 50, 36, 16
BATCHES = (1, 3)

SCRIPT = r"""
import sys
sys.path.insert(0, %(repo)r)
from types import SimpleNamespace
import torch
from oracle import ref_harness as rh
ref = rh.load_reference()
from oracle import loops
from oracle.ddim_scheduler import DDIMScheduler
from oracle.unet2d import ToyEpsModel
T, Tskip, S = 50, 36, 16
for B in (1, 3):
    sch = DDIMScheduler.from_preset("ddpm")
    sch.config.clip_sample = False
    sch.set_timesteps(T)
    unet = ToyEpsModel(3, S, seed=5)
    w = ref.DDPM(SimpleNamespace(unet=unet, scheduler=sch, device=torch.device("cpu")))
    g = torch.Generator().manual_seed(11 + B)
    xt = torch.randn(B, 3, S, S, generator=g)
    zs = 3.0 * torch.randn(T, 3, S, S, generator=g)
    n = T - Tskip
    x_ref, _ = rh.config2_regeneration(ref, w, xt, zs[Tskip:], n, eta=1.0, loss_scale=50.0)

    def eps_fn(x, t):
        with torch.no_grad():
            return unet(x, torch.tensor(t))["sample"]

    x_or, _, _ = loops.guided_edit_loop(sch, eps_fn, xt, eta=1.0, zs=zs[Tskip:], mode="ddpm",
                                        guidance=loops.color_guidance([0.8, None, None], [1, 1, 1], 50.0, 0, 10 ** 9))
    assert torch.equal(x_ref.detach(), x_or), (B, (x_ref.detach() - x_or).abs().max().item())
print("HARNESS_OK")
"""


def oracle_regeneration(B, eps_fn=None):
    """The seeded case of SCRIPT through the oracle loop.  eps_fn(x, t, model) -> eps replaces the model call when given.
    Returns (final samples, [eps of every step])."""
    from oracle import loops
    from oracle.ddim_scheduler import DDIMScheduler
    from oracle.unet2d import ToyEpsModel
    sch = DDIMScheduler.from_preset("ddpm")
    sch.config.clip_sample = False
    sch.set_timesteps(T)
    unet = ToyEpsModel(3, S, seed=5)
    g = torch.Generator().manual_seed(11 + B)
    xt = torch.randn(B, 3, S, S, generator=g)
    zs = 3.0 * torch.randn(T, 3, S, S, generator=g)
    eps_seen = []

    def step_eps(x, t):
        if eps_fn is not None:
            e = eps_fn(x, t, unet)
        else:
            with torch.no_grad():
                e = unet(x, torch.tensor(t))["sample"]
        eps_seen.append(e)
        return e

    x, _, _ = loops.guided_edit_loop(sch, step_eps, xt, eta=1.0, zs=zs[TSKIP:], mode="ddpm",
                                     guidance=loops.color_guidance([0.8, None, None], [1, 1, 1], 50.0, 0, 10 ** 9))
    return x, eps_seen


def test_config2_harness_of_reference_functions_equals_oracle_loop(golden):
    g = golden("ref_harness")
    for B in BATCHES:
        eps = torch.from_numpy(g[f"B{B}/eps"])
        assert eps.shape == (T - TSKIP, B, 3, S, S)

        def replay(x, t, model, it=iter(eps)):
            e = next(it)
            with torch.no_grad():
                live = model(x, torch.tensor(t))["sample"]
            assert torch.allclose(live, e, rtol=1e-5, atol=1e-6), (B, t, (live - e).abs().max().item())
            return e

        x, seen = oracle_regeneration(B, replay)
        assert len(seen) == T - TSKIP
        assert np.array_equal(x.numpy(), g[f"B{B}/x"]), (B, np.abs(x.numpy() - g[f"B{B}/x"]).max())
    if os.path.isfile(os.path.join(REPO, "baseline", "_ref", "src", "SegDiffEditPipeline.py")):
        r = subprocess.run([sys.executable, "-c", SCRIPT % {"repo": REPO}], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "HARNESS_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


if __name__ == "__main__":
    sys.path.insert(0, REPO)
    out = {}
    for B in BATCHES:
        x, eps = oracle_regeneration(B)
        out[f"B{B}/x"] = x.numpy()
        out[f"B{B}/eps"] = torch.stack(eps).numpy()
    np.savez_compressed(GOLDEN, **out)
    print(GOLDEN, {k: v.shape for k, v in out.items()})
