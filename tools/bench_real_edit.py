"""Batched real-image editing on the B200: one batched call against serial batch-1 calls of the same work.

* DDPM-256 and LDM (CelebA-HQ layouts, random weights), B = 8: the first 8 images of a seeded set go through
  ``prepare_real_image_edit(..., inversion_method="ddpm", eta=1, classes=[17])`` (face parser -> masks -> encoder ->
  edit-friendly DDPM inversion, 50 steps) and ``edit_image(Tskip=36)`` with per-sample masked colour guidance.  Arm
  "batched": one call on all 8 images; arm "serial": 8 batch-1 calls on the same pipeline (the engines re-plan for
  batch 1 once at the start of each serial region).
* The face parser at B = 8, 512 x 512: ``BiSeNet.labels`` (upsampling fused with the argmax) against the logits
  forward followed by ``torch.argmax``.

Each arm is timed with CUDA events over regions of at least --min-seconds after a warm-up; the two arms of a pair
alternate in one process (--rounds regions each), so the spread is measured in the same call as the difference.  The
card's name and power limit are read before and after.

    python tools/bench_real_edit.py --out DIR
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
for p in (REPO, os.path.join(REPO, "diffusion-image-editing_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        q = f"unavailable ({e})"
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q)


def region_ms(fn, min_s):
    """ms per call (CUDA events) over a region of at least min_s seconds of host time."""
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0, n = time.perf_counter(), 0
    a.record()
    while True:
        fn()
        n += 1
        torch.cuda.synchronize()
        if time.perf_counter() - t0 >= min_s:
            break
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n, n


def ab(arms, rounds, min_s, warmup=2):
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    res = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ms, n = region_ms(fn, min_s)
            res[k].append(dict(ms_per_call=ms, calls=n))
    out = {}
    for k, v in res.items():
        ms = [r["ms_per_call"] for r in v]
        out[k] = dict(regions=v, median_ms=sorted(ms)[len(ms) // 2], min_ms=min(ms), max_ms=max(ms),
                      spread=(max(ms) - min(ms)) / min(ms))
    return out


def bench_family(name, args):
    from attr_functions import SingleColorAttrFunc
    from models import SegmentationModel, create_diffusion_model
    from SegDiffEditPipeline import SegDiffEditPipeline
    B = 8
    w = create_diffusion_model(name, sample_clipping=False, max_batch=B, seed=0)
    w.scheduler.set_timesteps(args.steps)
    pipe = SegDiffEditPipeline(w, SegmentationModel(None, 19, (512, 512), max_batch=B))
    images = torch.rand(16, 3, 256, 256, generator=torch.Generator().manual_seed(1)) * 2 - 1
    imgs = images[:B].cuda()
    f = SingleColorAttrFunc(target=0.6, color_idx=0, loss_scale=30.0, per_sample=True, use_mask=True, mask_attr_grad=True)

    def edit(x):
        xt, zs, xts, mask, _ = pipe.prepare_real_image_edit(x, eta=1, inversion_method="ddpm", classes=[17], prog_bar=False)
        return pipe.edit_image(xt=xt, eta=1, zs=zs, xts=xts, mask=mask, attr_func=f, Tskip=args.tskip,
                               inversion_method="ddpm", prog_bar=False, output_type="tensor").imgs

    def serial():
        for b in range(B):
            edit(imgs[b:b + 1])

    res = ab({"batched (one call, B = 8)": lambda: edit(imgs), "serial (8 calls, B = 1)": serial}, args.rounds,
             args.min_seconds)
    res["batched_over_serial"] = res["batched (one call, B = 8)"]["median_ms"] / res["serial (8 calls, B = 1)"]["median_ms"]
    res["config"] = dict(model=f"{name} (random weights, fp16 UNet)", batch=B, inversion_steps=args.steps, tskip=args.tskip,
                         edit_steps=args.steps - args.tskip, classes=[17], parser="BiSeNet 512x512 (fp16, forward only)",
                         guidance="SingleColorAttrFunc(target=0.6, color_idx=0, loss_scale=30, per_sample=True, "
                                  "use_mask=True, mask_attr_grad=True)")
    del pipe, w
    torch.cuda.empty_cache()
    return res


def bench_labels(args):
    from b200edit.bisenet import BiSeNet
    B, S = 8, 512
    net = BiSeNet(19, S, max_batch=B).init_random(0)
    x = torch.randn(B, 3, S, S, generator=torch.Generator().manual_seed(2)).cuda()
    same = bool(torch.equal(net.labels(x), net(x)[0].argmax(1)))
    res = ab({"labels (fused upsample + argmax)": lambda: net.labels(x),
              "logits + torch.argmax": lambda: net(x)[0].argmax(1)}, args.rounds, args.min_seconds, warmup=5)
    res["labels_over_logits"] = (res["labels (fused upsample + argmax)"]["median_ms"]
                                 / res["logits + torch.argmax"]["median_ms"])
    res["config"] = dict(batch=B, size=S, classes=19, precision="fp16", labels_equal_argmax_of_logits=same,
                         logits_bytes=B * 19 * S * S * 4, labels_bytes=B * S * S * 8)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for real_edit_bench.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=2.0)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--tskip", type=int, default=36)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_real_edit: no CUDA device (this measurement needs the GPU)")
    res = dict(card=card())
    res["parser_labels_b8_512"] = bench_labels(args)
    print(json.dumps({k: v.get("median_ms") if isinstance(v, dict) else v for k, v in res["parser_labels_b8_512"].items()
                      if k != "config"}), flush=True)
    for name in ("ddpm", "ldm"):
        res[f"{name}_real_edit_b8"] = r = bench_family(name, args)
        print(name, json.dumps({k: v.get("median_ms") if isinstance(v, dict) else v for k, v in r.items() if k != "config"}),
              flush=True)
    res["card_after"] = card()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "real_edit_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
