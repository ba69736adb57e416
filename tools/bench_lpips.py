"""LPIPS (vgg) on the B200: native forward and forward + input gradient against torch eager (oracle restatement +
autograd, cuDNN, fp32 and fp16) at 256^2 / 512^2 and batch 1 / 8, and the cost of ``use_lpips`` in a 50-step DDPM
``edit_image`` at batch 8 against ``use_l2``.  CUDA-event times after warm-up; FLOP/s from shapes (algorithmic VGG
convolution work: 2 * H * W * Cin * Cout * 9 per layer; the backward pass counts the dgrad chain once more).

    python tools/bench_lpips.py [--out profiles/lpips_bench.json] [--iters 20]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
for p in (REPO, os.path.join(REPO, "diffusion-image-editing_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

VGG = ((3, 64, 0), (64, 64, 0), (64, 128, 1), (128, 128, 1), (128, 256, 2), (256, 256, 2), (256, 256, 2), (256, 512, 3),
       (512, 512, 3), (512, 512, 3), (512, 512, 4), (512, 512, 4), (512, 512, 4))


def vgg_flops(S):
    return sum(2.0 * (S >> lv) ** 2 * cin * cout * 9 for cin, cout, lv in VGG)


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        q = f"unavailable ({e})"
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q)


def bench_network(iters):
    from b200edit.lpips import LPIPS, lpips_random_state_dict
    from oracle.lpips import LPIPS as OracleLPIPS
    sd = lpips_random_state_dict(0)
    rows = []
    for S in (256, 512):
        for B in (1, 8):
            fl = vgg_flops(S) * B
            g = torch.Generator().manual_seed(S + B)
            x0 = (torch.rand(B, 3, S, S, generator=g) * 2 - 1).cuda()
            x1 = (torch.rand(1, 3, S, S, generator=g) * 2 - 1).cuda()
            for prec in ("fp32", "fp16"):
                net = LPIPS(input_size=S, max_batch=B, precision=prec)
                net.load_state_dict(sd)
                net(x0, x1)
                f_ms = timed(lambda: net(x0, x1), iters)

                def fb():
                    x = x0.detach().requires_grad_(True)
                    torch.autograd.grad(net(x, x1).sum(), x)
                fb_ms = timed(fb, iters)
                rows.append(dict(impl="native", precision=prec, S=S, B=B, fwd_ms=f_ms, fwd_bwd_ms=fb_ms,
                                 fwd_tflops=fl / f_ms / 1e9, fwd_bwd_tflops=2 * fl / fb_ms / 1e9,
                                 algorithmic_gflop_fwd=fl / 1e9))
                del net
                torch.cuda.empty_cache()
            for prec, dt in (("fp32", torch.float32), ("fp16", torch.float16)):
                torch.backends.cudnn.allow_tf32 = False
                torch.backends.cuda.matmul.allow_tf32 = False
                o = OracleLPIPS()
                o.load_state_dict(sd)
                o = o.cuda().to(dt)
                a, b = x0.to(dt), x1.to(dt)
                with torch.no_grad():
                    f_ms = timed(lambda: o(a, b), iters)

                def fb2():
                    x = a.detach().requires_grad_(True)
                    torch.autograd.grad(o(x, b).sum(), x)
                fb_ms = timed(fb2, iters)
                rows.append(dict(impl="torch-eager-cudnn", precision=prec, S=S, B=B, fwd_ms=f_ms, fwd_bwd_ms=fb_ms,
                                 fwd_tflops=fl / f_ms / 1e9, fwd_bwd_tflops=2 * fl / fb_ms / 1e9,
                                 algorithmic_gflop_fwd=fl / 1e9))
                del o
                torch.cuda.empty_cache()
            print(json.dumps(rows[-4:]), flush=True)
    return rows


def bench_edit(steps=50, B=8):
    from attr_functions import MultiColorAttrFunc
    from models import create_diffusion_model, get_lpips
    from SegDiffEditPipeline import SegDiffEditPipeline
    w = create_diffusion_model("ddpm", sample_clipping=True, max_batch=B, seed=0)
    w.scheduler.set_timesteps(steps)
    S = w.unet.config.sample_size
    g = torch.Generator().manual_seed(1)
    xt = torch.randn(B, 3, S, S, generator=g).cuda()
    mask = (torch.rand(1, 3, S, S, generator=g) > 0.5).float().cuda()
    x_0 = (torch.rand(1, 3, S, S, generator=g) * 2 - 1).cuda()
    lp = get_lpips(input_size=S, max_batch=B)
    out = {}
    for name, kw in (("use_l2", dict(use_l2=True)), ("use_lpips", dict(use_lpips=True, lpips_model=lp))):
        f = MultiColorAttrFunc(0.8, 0.2, 0.3, loss_scale=50.0, t1=0, t2=steps, use_mask=True, mask_pred_original_sample=True,
                               lambda_=0.5, x_0=x_0, **kw)
        pipe = SegDiffEditPipeline(w, None)
        run = lambda: pipe.edit_image(xt=xt, attr_func=f, prog_bar=False, output_type="tensor", mask=mask)   # noqa: E731
        ms = timed(run, 2, warmup=1)
        out[name] = dict(ms_per_edit=ms, ms_per_step=ms / steps)
        print(name, out[name], flush=True)
    out["lpips_overhead_ms_per_guided_step"] = out["use_lpips"]["ms_per_step"] - out["use_l2"]["ms_per_step"]
    out["config"] = dict(model="ddpm (DDPM256 layout, random weights)", batch=B, steps=steps, lpips_precision="fp32")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "lpips_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lpips: no CUDA device (this measurement needs the GPU)")
    res = dict(card=card(), network=bench_network(args.iters), edit=bench_edit())
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["edit"]))


if __name__ == "__main__":
    main()
