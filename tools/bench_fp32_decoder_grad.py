#!/usr/bin/env python
"""Cost of the fp32-accurate decoder gradient against the 16-bit gradient twin of a precision="fp32" pipeline: the LDM VQ
decoder (256 x 256 images, B = 8) and the SD KL decoder (512 x 512, B = 8 or the largest batch that fits, stated).

    python tools/bench_fp32_decoder_grad.py [--out profiles/fp32_decoder_grad_b200.json] [--window 2.0]

Per decoder and set-up ("twin": the split decoder forward-only + a 16-bit decoder in gradient mode with the same weights,
what create_diffusion_model(precision="fp32") builds by default; "fp32": the split decoder itself in gradient mode,
decoder_grad_precision="fp32"):
  - ms per decode_keep + latent_grad (CUDA events, warm-up, windows of at least --window seconds);
  - the device bytes the set-up's engines allocate when built (weights and dgrad twins; free-memory difference) and
    the workspace bytes of the gradient engine;
  - the per-op backward breakdown of one call (B2E_PROFILE_BWD=1 in a child process, its stderr parsed).
Then one guided, config-3-shaped edit step (LDM, B = 8, colour guidance masked in latent space, analytic path) in an
fp32 pipeline with either set-up.  The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import re
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "diffusion-image-editing_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
import torch  # noqa: E402

from b200edit._C import lib  # noqa: E402
from b200edit.vqmodel import LDM_VQ_CONFIG, SD_VAE_CONFIG, AutoencoderKL, VQModel  # noqa: E402

DECODERS = {"ldm": (VQModel, LDM_VQ_CONFIG), "sd": (AutoencoderKL, SD_VAE_CONFIG)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def time_fn(fn, window):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 1
    while True:
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / 1e3
        if s >= window:
            return s / n * 1e3, n
        n = max(n * 2, int(n * window / max(s, 1e-6) * 1.1) + 1)


def build(family, setup, B):
    """-> (engines, gradient engine, device bytes the engines allocated when built)."""
    cls, cfg = DECODERS[family]
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    main = cls(**cfg, max_batch=B, precision="fp32").init_random(1)
    if setup == "fp32":
        engines, g = [main], main.enable_grad()
    else:
        twin = cls(**cfg, max_batch=B, precision=None)
        twin.load_state_dict(main.random_state_dict(1), strict=False)
        engines, g = [main, twin], twin.enable_grad()
    torch.cuda.synchronize()
    return engines, g, free0 - torch.cuda.mem_get_info()[0]


def inputs(family, B):
    cfg = DECODERS[family][1]
    g = torch.Generator("cuda").manual_seed(0)
    z = torch.randn(B, cfg["latent_channels"], cfg["sample_size"], cfg["sample_size"], device="cuda", generator=g)
    S = cfg["sample_size"] << (len(cfg["block_out_channels"]) - 1)
    return z, torch.randn(B, cfg["out_channels"], S, S, device="cuda", generator=g) * 1e-6


def measure(family, setup, B, window):
    engines, g, built_bytes = build(family, setup, B)
    z, dimg = inputs(family, B)

    def step():
        g.decode_keep(z)
        return g.latent_grad(dimg)

    ms, n = time_fn(step, window)
    out = dict(decoder=family, setup=setup, batch=B, ms_per_decode_keep_plus_latent_grad=ms, calls_timed=n,
               engine_bytes_at_build=int(built_bytes), grad_workspace_bytes=int(lib.b2e_unet_workspace_bytes(g._h)),
               engines=len(engines))
    del engines, g
    torch.cuda.empty_cache()
    return out


def profile_child(family, setup, B):
    """One backward with B2E_PROFILE_BWD=1 in a child process: the per-op lines it prints to stderr."""
    env = dict(os.environ, B2E_PROFILE_BWD="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", family, setup, str(B)], env=env,
                       capture_output=True, text=True)
    ops = []
    for line in r.stderr.splitlines():
        m = re.match(r"BWD\s+(\d+)\s+([\d.]+) us\s+([\d.]+) TF/s\s+([\d.]+) GB/s\s+(.*)", line)
        if m:
            ops.append(dict(idx=int(m.group(1)), us=float(m.group(2)), tflops=float(m.group(3)), gbs=float(m.group(4)),
                            desc=m.group(5).strip()))
    groups = {}
    for o in ops:
        key = "conv" if "conv" in o["desc"] else o["desc"].split(" (")[0]
        groups[key] = groups.get(key, 0.0) + o["us"]
    return dict(returncode=r.returncode, total_us=sum(o["us"] for o in ops), by_kind_us=groups, ops=ops,
                stderr_tail=r.stderr[-2000:] if r.returncode else "")


def child(family, setup, B):
    engines, g, _ = build(family, setup, B)
    z, dimg = inputs(family, B)
    for _ in range(2):       # the second call is the one whose breakdown counts (the first loads modules)
        g.decode_keep(z)
        g.latent_grad(dimg)
    torch.cuda.synchronize()


def largest_batch(family, want):
    for B in (want, 4, 2, 1):
        try:
            engines, g, _ = build(family, "fp32", B)
            z, dimg = inputs(family, B)
            g.decode_keep(z)
            g.latent_grad(dimg)
            torch.cuda.synchronize()
            del engines, g
            torch.cuda.empty_cache()
            return B
        except (RuntimeError, torch.OutOfMemoryError):
            torch.cuda.empty_cache()
    raise RuntimeError(f"{family}: no batch fits")


def guided_step(setup, B, window):
    """One config-3-shaped guided step (LDM, masked colour guidance through the decoder) via AttrFunc.apply."""
    from attr_functions import SingleColorAttrFunc
    from models import create_diffusion_model
    w = create_diffusion_model("ldm", sample_clipping=False, max_batch=B, seed=3, precision="fp32", with_encoder=False,
                               decoder_grad_precision="fp32" if setup == "fp32" else None)
    w.scheduler.set_timesteps(50)
    g = torch.Generator("cuda").manual_seed(1)
    xt = torch.randn(B, 3, 64, 64, device="cuda", generator=g)
    eps = torch.randn(B, 3, 64, 64, device="cuda", generator=g)
    mask = (torch.rand(1, 3, 64, 64, device="cuda", generator=g) > 0.5).float()
    t = torch.tensor(int(w.scheduler.timesteps[10]))
    f = SingleColorAttrFunc(target=0.8, color_idx=0, loss_scale=200.0, use_mask=True, mask_attr_grad=True)
    ms, n = time_fn(lambda: f.apply(xt=xt, zt=None, model_output=eps, timestep=t, step_idx=0, model=w, mask=mask,
                                    mask_attr_grad=True), window)
    return dict(setup=setup, batch=B, ms_per_guided_step=ms, steps_timed=n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "fp32_decoder_grad_b200.json"))
    ap.add_argument("--window", type=float, default=2.0)
    ap.add_argument("--child", nargs=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp32_decoder_grad: no CUDA device")
    if a.child:
        return child(a.child[0], a.child[1], int(a.child[2]))
    res = dict(gpu=gpu_info(), window_s=a.window, decoders=[], backward_profiles=[], guided_step=[])
    for family in ("ldm", "sd"):
        B = largest_batch(family, 8)
        for setup in ("twin", "fp32"):
            res["decoders"].append(measure(family, setup, B, a.window))
            res["backward_profiles"].append(dict(decoder=family, setup=setup, batch=B, **profile_child(family, setup, B)))
            print(json.dumps(res["decoders"][-1]), flush=True)
    for setup in ("twin", "fp32"):
        res["guided_step"].append(guided_step(setup, 8, a.window))
        print(json.dumps(res["guided_step"][-1]), flush=True)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
