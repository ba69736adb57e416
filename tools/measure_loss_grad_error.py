#!/usr/bin/env python
"""How far the loss networks' input gradients (ResNet attribute predictor, BiSeNet face parser, LPIPS-VGG) are from
float64 under the split-operand forward (precision="fp32"), with the 16-bit backward (grad_precision=None) and with the
split-operand backward (grad_precision="fp32").

    python tools/measure_loss_grad_error.py [--out profiles/loss_grad_error_b200.json]

Per case, the relative RMS against autograd through the same network in float64 on the CPU (torchvision ResNet / the
oracle modules, same weights, random output gradient) of
  e_now   - the native input gradient with the 16-bit backward;
  e_split - the same with the split backward;
  e32     - torch float32 autograd on the CPU (the yardstick);
"split_backward_can_help" records e_now >= 2 max(1e-4, 3 e32).  Per backward, where the error sits: the share of the
squared error in the 1 % of pixels with the largest error, and the relative RMS of the other 99 %.  A ReLU / max-pool
mask that the split forward sets differently from float64 changes the gradient in one receptive field only, so such
errors concentrate in few pixels; rounding spreads evenly.  The GPU's name and power limit are read in the same run."""
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


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()


def cpu_grad(fn, x, w):
    x = x.clone().requires_grad_(True)
    (g,) = torch.autograd.grad((fn(x) * w).sum(), x)
    return g


def concentration(g, g64):
    d = (g.detach().double().cpu() - g64).pow(2).sum(1).flatten()       # squared error per pixel (summed over channels)
    s, n = d.sort(descending=True).values, d.numel()
    return dict(top1pct_share=(s[:n // 100].sum() / d.sum()).item(),
                rel_rms_outside_top1pct=(s[n // 100:].sum() / g64.pow(2).sum()).sqrt().item())


def record(res, tag, g_now, g_split, g32, g64):
    e_now, e_split, e32 = rel(g_now, g64), rel(g_split, g64), rel(g32, g64)
    floor = max(1e-4, 3 * e32)
    w_now, w_split = concentration(g_now, g64), concentration(g_split, g64)
    res[tag] = dict(e_now=e_now, e_split=e_split, e32=e32, floor=floor, split_backward_can_help=e_now >= 2 * floor,
                    where_now=w_now, where_split=w_split)
    print(f"{tag}: e_now {e_now:.3e} | e_split {e_split:.3e} | torch fp32 e32 {e32:.3e} | floor {floor:.3e} | top-1% share "
          f"16-bit {w_now['top1pct_share']:.3f} split {w_split['top1pct_share']:.3f} | rest 16-bit "
          f"{w_now['rel_rms_outside_top1pct']:.2e} split {w_split['rel_rms_outside_top1pct']:.2e}", flush=True)


def resnet_reference(kind, num_classes, seed):
    import torchvision as tv
    torch.manual_seed(seed)
    net = (tv.models.resnet50 if kind == "resnet50" else tv.models.resnet18)()
    net.fc = torch.nn.Linear(net.fc.in_features, num_classes)
    g = torch.Generator().manual_seed(seed + 1)
    for mod in net.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):   # a trained network's statistics are not (0, 1)
            mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
            mod.running_var.copy_(torch.rand(mod.num_features, generator=g) * 0.5 + 0.75)
            mod.weight.data.copy_(torch.rand(mod.num_features, generator=g) * 0.5 + 0.75)
            mod.bias.data.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
    return net.eval()


def resnet_case(res, kind, S, B, K, seed):
    from b200edit.resnet import ResNet
    ref = resnet_reference(kind, K, seed)
    g = torch.Generator().manual_seed(seed + 2)
    x = torch.rand(B, 3, S, S, generator=g) * 2 - 1
    w = torch.randn(B, K, generator=g)
    grads = []
    for gp in (None, "fp32"):
        net = ResNet("bottleneck" if kind == "resnet50" else "basic", (3, 4, 6, 3) if kind == "resnet50" else (2, 2, 2, 2), K,
                     S, max_batch=B, precision="fp32", grad_precision=gp)
        net.load_torchvision_state_dict(ref.state_dict())
        net.forward_keep(x.cuda())
        grads.append(net.input_grad(w.cuda()).cpu())
        del net
    record(res, f"{kind} {S}x{S} B={B}", *grads, cpu_grad(ref, x, w), cpu_grad(ref.double(), x.double(), w.double()))


def bisenet_case(res, S, B, seed):
    from b200edit.bisenet import MultiResBiSeNet
    from oracle.bisenet import BiSeNet as OracleBiSeNet, seeded_weights
    o = seeded_weights(OracleBiSeNet(19).eval(), seed)
    o.conv_out.conv_out.weight.data.mul_(0.02)      # logits of O(1): an unsaturated softmax, as a trained parser has
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, 3, S, S, generator=g)
    w = torch.randn(B, 19, S, S, generator=g)
    grads = []
    for gp in (None, "fp32"):
        m = MultiResBiSeNet(19, max_batch=B, grad_precision=gp)
        m.load_reference_state_dict(o.state_dict())
        e = m.engine(S, grad=True)                  # the differentiated engine: split forward
        e.forward_keep(x.cuda())
        grads.append(e.input_grad(w.cuda()).cpu())
        del m, e
    o64 = seeded_weights(OracleBiSeNet(19).eval(), seed)
    o64.conv_out.conv_out.weight.data.mul_(0.02)
    o64 = o64.double()
    record(res, f"bisenet {S}x{S} B={B}", *grads, cpu_grad(lambda t: o(t)[0], x, w),
           cpu_grad(lambda t: o64(t)[0], x.double(), w.double()))


def lpips_case(res, S, B, RB, masked, seed):
    from b200edit.lpips import LPIPS, lpips_random_state_dict
    from oracle.lpips import LPIPS as OracleLPIPS
    sd = lpips_random_state_dict(seed)
    o = OracleLPIPS()
    o.load_state_dict(sd)
    g = torch.Generator().manual_seed(seed + 1)
    x0 = torch.rand(B, 3, S, S, generator=g) * 2 - 1
    x1 = torch.rand(RB, 3, S, S, generator=g) * 2 - 1
    mask = (torch.rand(B, 3, S, S, generator=g) > 0.4).float() if masked else None
    wd = torch.rand(B, generator=g) + 0.5
    grads = []
    for gp in (None, "fp32"):
        net = LPIPS(input_size=S, max_batch=B, precision="fp32", grad_precision=gp)
        net.load_state_dict(sd)
        net(x0.cuda(), x1.cuda(), mask=None if mask is None else mask.cuda())
        grads.append(net.input_grad(wd.cuda()).cpu())
        del net

    def fn(m):
        return lambda t: m(t if mask is None else 1 - mask.to(t.dtype) * t, x1.to(t.dtype)).reshape(-1)
    g32 = cpu_grad(fn(o), x0, wd)
    g64 = cpu_grad(fn(o.double()), x0.double(), wd.double())
    record(res, f"lpips {S}x{S} B={B} ref={RB} mask={masked}", *grads, g32, g64)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "loss_grad_error_b200.json"))
    args = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    res = {"gpu": gpu_info(), "cases": {}}
    print(res["gpu"], flush=True)
    c = res["cases"]
    resnet_case(c, "resnet18", 64, 2, 16, 1)
    resnet_case(c, "resnet50", 256, 2, 80, 2)
    resnet_case(c, "resnet50", 512, 1, 80, 3)
    bisenet_case(c, 128, 2, 7)
    bisenet_case(c, 256, 2, 7)
    lpips_case(c, 64, 2, 1, True, 3)
    lpips_case(c, 256, 2, 2, False, 4)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
