"""Per-sample network guidance on the B200: what guiding every image of a batch costs against the default mode.

* SD config-4 shape: ``edit_image`` at batch 8, CFG 7.5, ``ClassifierAttrFunc`` on the 512^2 fp32-accurate ResNet-50
  predictor; per_sample=False (the reference's semantics: the autograd path, only image 0 guided) against per_sample=True
  (the native kernel-to-kernel path, every image guided), and per_sample=True on the autograd path (the predictor in a
  lambda), which separates the cost of the path from the cost of guiding 8 images instead of 1 (in the default mode the
  backward passes of the predictor and the decoder carry zero gradients for images 1..7).  Every arm runs the predictor
  and decoder forward and backward over the whole batch.
* LDM shape: ``edit_image`` at batch 8, ``NetAttrFunc(idx_for_class=[17])`` through the native BiSeNet at 256^2;
  per_sample=True on the native path against per_sample=True on the autograd path (the parser wrapped in a lambda, which
  the native path cannot see through).
* The batched seg-area head alone at B = 8 (19 x 256^2 and 19 x 512^2): bytes moved (logits read + gradient written)
  over CUDA-event time, against the 6 560 GB/s copy bandwidth measured for this project on a B200.

Every ``edit_image`` arm is timed over regions of at least --min-seconds after a warm-up, the two arms alternated in one
process (--rounds regions each), so the run-to-run spread is measured in the same call as the difference.

    python tools/bench_net_guidance.py --out DIR
"""
import argparse
import json
import os
import subprocess
import sys
import time
from types import SimpleNamespace

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
for p in (REPO, os.path.join(REPO, "diffusion-image-editing_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

COPY_GBPS = 6560.0   # measured copy bandwidth of the project's B200 (BASELINE.md)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        q = f"unavailable ({e})"
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q)


def region_ms(fn, min_s):
    """ms per call over a region of at least min_s seconds (host clock around work that ends in a synchronise)."""
    torch.cuda.synchronize()
    t0, n = time.perf_counter(), 0
    while True:
        fn()
        n += 1
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        if el >= min_s:
            return el * 1e3 / n, n


def ab(arms, rounds, min_s, warmup=2):
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    res = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ms, n = region_ms(fn, min_s)
            res[k].append(dict(ms_per_edit=ms, calls=n))
    out = {}
    for k, v in res.items():
        ms = [r["ms_per_edit"] for r in v]
        out[k] = dict(regions=v, median_ms=sorted(ms)[len(ms) // 2], min_ms=min(ms), max_ms=max(ms),
                      spread=(max(ms) - min(ms)) / min(ms))
    return out


def bench_sd(args):
    from attr_functions import ClassifierAttrFunc
    from models import create_diffusion_model, get_pretrained_anyGAN
    from SegDiffEditPipeline import SegDiffEditPipeline
    B, D = 8, args.sd_steps
    predictor = get_pretrained_anyGAN(input_size=512, max_batch=B, precision="fp32")
    w = create_diffusion_model("sd", sample_clipping=False, max_batch=B, seed=0, with_encoder=False)
    w.scheduler.set_timesteps(D)
    text_emb = torch.randn(2, 77, 768, generator=torch.Generator().manual_seed(3)).cuda()   # no tokenizer files offline
    w.additional_prep = lambda model, prompt: text_emb
    pipe = SegDiffEditPipeline(w, None)
    x = torch.randn(B, 4, 64, 64, generator=torch.Generator().manual_seed(4)).cuda()
    arms = {}
    for name, pred, ps in (("per_sample=False (autograd, image 0 guided)", predictor, False),
                           ("per_sample=True (native, all images guided)", predictor, True),
                           ("per_sample=True autograd (predictor in a lambda)", lambda img: predictor(img), True)):
        f = ClassifierAttrFunc(pred, idx_for_class=31, idx_of_interest=0, loss_scale=50.0, t1=0, t2=10 ** 9, per_sample=ps)
        arms[name] = (lambda f=f: pipe.edit_image(xt=x, attr_func=f, prompt="a photo of a face", cfg_scale=7.5, prog_bar=False,
                                                  output_type="tensor"))
    res = ab(arms, args.rounds, args.min_seconds)
    res["config"] = dict(model="sd (SD 1.x layout, random weights, fp16 UNet)", batch=B, denoising_steps_per_edit=D, cfg_scale=7.5,
                         guidance="ClassifierAttrFunc(idx_for_class=31, idx_of_interest=0, loss_scale=50)",
                         predictor="ResNet-50 512x512, fp32-accurate forward")
    del pipe, w, predictor
    torch.cuda.empty_cache()
    return res


def bench_ldm(args):
    from attr_functions import NetAttrFunc
    from models import SegmentationModel, create_diffusion_model
    from SegDiffEditPipeline import SegDiffEditPipeline
    B, D = 8, args.ldm_steps
    w = create_diffusion_model("ldm", sample_clipping=False, max_batch=B, seed=0, with_encoder=False)
    w.scheduler.set_timesteps(D)
    seg = SegmentationModel(None, 19, (512, 512), max_batch=B)
    pipe = SegDiffEditPipeline(w, None)
    x = torch.randn(B, 3, 64, 64, generator=torch.Generator().manual_seed(5)).cuda()
    opaque = SimpleNamespace(net=lambda img: seg.net(img))
    arms = {}
    for name, sm in (("per_sample=True native", seg), ("per_sample=True autograd (parser in a lambda)", opaque)):
        f = NetAttrFunc(sm, idx_for_class=[17], loss_scale=1e4, t1=0, t2=10 ** 9, per_sample=True)
        arms[name] = lambda f=f: pipe.edit_image(xt=x, attr_func=f, prog_bar=False, output_type="tensor")
    res = ab(arms, args.rounds, args.min_seconds)
    res["config"] = dict(model="ldm (CelebAHQ layout, random weights, fp16 UNet, VQ decoder in gradient mode)", batch=B,
                         denoising_steps_per_edit=D, guidance="NetAttrFunc(idx_for_class=[17], loss_scale=1e4, per_sample=True)",
                         parser="BiSeNet 256x256 (MultiResBiSeNet gradient engine, fp32-accurate forward)")
    del pipe, w, seg
    torch.cuda.empty_cache()
    return res


def bench_heads(iters):
    from b200edit import ops
    rows = []
    for S in (256, 512):
        B, Cc = 8, 19
        lg = 3.0 * torch.randn(B, Cc, S, S, device="cuda")
        fn = lambda: ops.seg_area_head(lg, [1, 10, 17], per_sample=True, grad_scale=1e4)   # noqa: E731
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / iters
        nbytes = 2 * B * Cc * S * S * 4     # logits read once, gradient written once
        rows.append(dict(head="seg_area_head_batched (loss + gradient)", B=B, C=Cc, S=S, ms=ms, bytes=nbytes,
                         gbps=nbytes / ms / 1e6, share_of_copy_bw=nbytes / ms / 1e6 / COPY_GBPS,
                         note="host-side allocation and launch included; working set "
                              + ("fits" if nbytes <= 126e6 else "exceeds") + " the 126 MB L2"))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for net_guidance_bench.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=2.0)
    ap.add_argument("--sd-steps", type=int, default=3)
    ap.add_argument("--ldm-steps", type=int, default=4)
    ap.add_argument("--head-iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_net_guidance: no CUDA device (this measurement needs the GPU)")
    res = dict(card=card(), heads=bench_heads(args.head_iters))
    print(json.dumps(res["heads"]), flush=True)
    res["sd_config4_shape"] = bench_sd(args)
    print(json.dumps({k: v.get("median_ms") for k, v in res["sd_config4_shape"].items() if k != "config"}), flush=True)
    res["ldm_shape"] = bench_ldm(args)
    print(json.dumps({k: v.get("median_ms") for k, v in res["ldm_shape"].items() if k != "config"}), flush=True)
    res["card_after"] = card()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "net_guidance_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
