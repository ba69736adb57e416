#!/usr/bin/env python
"""Cost of the fp32-accurate loss-network backward (grad_precision="fp32") against the default 16-bit backward, both under
the fp32-accurate forward (precision="fp32"):

    python tools/bench_fp32_loss_grads.py [--out profiles/fp32_loss_grads_b200.json] [--min-seconds 2.0] [--rounds 3]

  - ms per forward_keep + input_grad at B = 8: ResNet-50 256^2 and 512^2, BiSeNet 256^2 (the differentiated engine of
    MultiResBiSeNet), LPIPS-VGG 256^2 (reference batch 1); the two settings alternated in one process, each timed over
    regions of at least --min-seconds (host clock around work that ends in a synchronise) after a warm-up;
  - the workspace bytes of each engine;
  - config-4-shaped guided edits: SD (random weights), B = 8, CFG 7.5, 3 guided DDIM steps, ClassifierAttrFunc(per_sample=
    True) through a 512^2 ResNet-50, precision="fp32", decoder_grad_precision="fp32"; the predictor's grad_precision None
    vs "fp32" (ms per edit and per step).
The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "diffusion-image-editing_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
import torch  # noqa: E402

from b200edit._C import lib  # noqa: E402

SETTINGS = (None, "fp32")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(torch_device=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip() or q.stderr.strip())


def region_ms(fn, min_s):
    torch.cuda.synchronize()
    t0, n = time.perf_counter(), 0
    while True:
        fn()
        n += 1
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        if el >= min_s:
            return el * 1e3 / n, n


def alternate(arms, rounds, min_s):
    for fn in arms.values():
        fn()
        fn()
    out = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            out[k].append(region_ms(fn, min_s)[0])
    return {k: dict(ms=v, median_ms=sorted(v)[len(v) // 2], spread=(max(v) - min(v)) / min(v)) for k, v in out.items()}


def network(kind, S, B, gp):
    """-> (engine, call of forward_keep + input_grad)."""
    g = torch.Generator("cuda").manual_seed(S)
    x = torch.rand(B, 3, S, S, device="cuda", generator=g) * 2 - 1
    if kind == "resnet50":
        from b200edit.resnet import ResNet
        net = ResNet("bottleneck", (3, 4, 6, 3), 80, S, max_batch=B, precision="fp32", grad_precision=gp).init_random(0)
        d = torch.randn(B, 80, device="cuda", generator=g)
        return net, lambda: net.input_grad(d) if net.forward_keep(x) is not None else None
    if kind == "bisenet":
        from b200edit.bisenet import MultiResBiSeNet
        net = MultiResBiSeNet(19, max_batch=B, grad_precision=gp).engine(S, grad=True)
        d = torch.randn(B, 19, S, S, device="cuda", generator=g)
        return net, lambda: net.input_grad(d) if net.forward_keep(x) is not None else None
    from b200edit.lpips import LPIPS
    net = LPIPS(input_size=S, max_batch=B, precision="fp32", grad_precision=gp)
    net.init_random(0)
    x1 = torch.rand(1, 3, S, S, device="cuda", generator=g) * 2 - 1
    d = torch.ones(B, device="cuda")
    return net, lambda: net.input_grad(d) if net(x, x1) is not None else None


def guided_step(args):
    """edit_image with D = 3 denoising steps (CFG 7.5, every step guided); ms per step = ms per edit / 3."""
    from attr_functions import ClassifierAttrFunc
    from models import create_diffusion_model, get_pretrained_anyGAN
    from SegDiffEditPipeline import SegDiffEditPipeline
    B, D = 8, 3
    w = create_diffusion_model("sd", sample_clipping=False, max_batch=B, seed=0, with_encoder=False, precision="fp32",
                               decoder_grad_precision="fp32")
    w.scheduler.set_timesteps(D)
    text_emb = torch.randn(2, 77, 768, generator=torch.Generator().manual_seed(3)).cuda()   # no tokenizer files offline
    w.additional_prep = lambda model, prompt: text_emb
    pipe = SegDiffEditPipeline(w, None)
    x = torch.randn(B, 4, 64, 64, generator=torch.Generator().manual_seed(4)).cuda()
    arms = {}
    for gp in SETTINGS:
        pred = get_pretrained_anyGAN(input_size=512, max_batch=B, precision="fp32", grad_precision=gp, state_dict_path=None)
        f = ClassifierAttrFunc(pred, idx_for_class=31, idx_of_interest=0, loss_scale=50.0, t1=0, t2=10 ** 9, per_sample=True)
        arms[f"grad_precision={gp}"] = (lambda f=f: pipe.edit_image(xt=x, attr_func=f, prompt="a photo of a face", cfg_scale=7.5,
                                                                    prog_bar=False, output_type="tensor"))
    res = alternate(arms, args.rounds, args.min_seconds)
    for v in res.values():
        v["median_ms_per_step"] = v["median_ms"] / D
    res["config"] = dict(model="sd (SD 1.x layout, random weights), precision='fp32', decoder_grad_precision='fp32'", batch=B,
                         denoising_steps_per_edit=D, cfg_scale=7.5,
                         guidance="ClassifierAttrFunc(idx_for_class=31, per_sample=True), ResNet-50 512x512 (random weights)")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "fp32_loss_grads_b200.json"))
    ap.add_argument("--min-seconds", type=float, default=2.0)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp32_loss_grads: no CUDA device")
    res = dict(gpu=card(), networks=[])
    for kind, S in (("resnet50", 256), ("resnet50", 512), ("bisenet", 256), ("lpips", 256)):
        engines = {gp: network(kind, S, 8, gp) for gp in SETTINGS}
        timed = alternate({f"grad_precision={gp}": fn for gp, (_, fn) in engines.items()}, args.rounds, args.min_seconds)
        for gp, (net, _) in engines.items():
            timed[f"grad_precision={gp}"]["workspace_bytes"] = int(lib.b2e_unet_workspace_bytes(net._h))
        res["networks"].append(dict(network=kind, size=S, batch=8, **timed))
        print(json.dumps(res["networks"][-1]), flush=True)
        del engines
        torch.cuda.empty_cache()
    res["guided_step_config4"] = guided_step(args)
    print(json.dumps(res["guided_step_config4"]), flush=True)
    res["gpu_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
