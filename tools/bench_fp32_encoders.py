#!/usr/bin/env python
"""Cost of the fp32-accurate encoders against the 16-bit ones: the LDM VQ encoder at 256 x 256 (B = 8), the SD KL
encoder at 512 x 512 (B = 8) and the CLIP text encoder at (2, 77), each in both modes.

    python tools/bench_fp32_encoders.py [--out result.json] [--window 2.0]

CUDA events around back-to-back forwards after a warm-up; every timed window lasts at least --window seconds.  Prints
one JSON document: the GPU's name and power limit (read in the same run), and per network and mode the time per
forward, the workspace bytes of the engine and the executed FLOPs."""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "diffusion-image-editing_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
import torch  # noqa: E402

from b200edit._C import lib  # noqa: E402
from b200edit.clip import SD15_CLIP_CONFIG, CLIPTextModel  # noqa: E402
from b200edit.vqmodel import LDM_VQ_CONFIG, SD_VAE_CONFIG, AutoencoderKL, VQModel  # noqa: E402


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


def bench_encoder(name, cls, cfg, B, precision, window):
    m = cls(**cfg, max_batch=B, with_encoder=True, encoder_precision=precision).init_random(0)
    S = m.out_size
    x = torch.rand(B, 3, S, S, device="cuda", generator=torch.Generator("cuda").manual_seed(0)) * 2 - 1
    ms, n = time_fn(lambda: m._encode_raw(x), window)
    enc = m._enc
    return dict(network=name, precision=enc.precision, batch=B, image=S, ms_per_forward=ms, forwards_timed=n,
                workspace_bytes=int(lib.b2e_unet_workspace_bytes(enc._h)), flops_per_forward=enc.flops_per_sample * B,
                launches_per_forward=enc.launches_per_forward)


def bench_clip(precision, window):
    m = CLIPTextModel(**SD15_CLIP_CONFIG, max_batch=2, precision=precision).init_random(0)
    ids = torch.randint(0, SD15_CLIP_CONFIG["vocab_size"], (2, 77), generator=torch.Generator().manual_seed(0)).cuda()
    ms, n = time_fn(lambda: m(ids), window)
    return dict(network="clip-vit-l14-text", precision=m.precision, batch=2, tokens=77, ms_per_forward=ms, forwards_timed=n,
                workspace_bytes=int(lib.b2e_unet_workspace_bytes(m._h)), flops_per_forward=m.flops_per_sample * 2,
                launches_per_forward=m.launches_per_forward)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--window", type=float, default=2.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp32_encoders: no CUDA device (this measurement has no CPU fall-back)")
    torch.cuda.set_device(0)
    res = dict(gpu=gpu_info(), window_s=a.window, runs=[])
    for precision in (None, "fp32"):
        res["runs"].append(bench_encoder("ldm-vq-encoder", VQModel, LDM_VQ_CONFIG, 8, precision, a.window))
        res["runs"].append(bench_encoder("sd-kl-encoder", AutoencoderKL, SD_VAE_CONFIG, 8, precision, a.window))
        res["runs"].append(bench_clip(precision, a.window))
        torch.cuda.empty_cache()
    by = {(r["network"], r["precision"]): r for r in res["runs"]}
    res["fp32_over_16bit_time"] = {n: by[(n, "fp32")]["ms_per_forward"] / by[(n, p)]["ms_per_forward"]
                                   for (n, p) in by if p != "fp32"}
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
