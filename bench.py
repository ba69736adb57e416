#!/usr/bin/env python
"""Benchmark of the guided denoising loop (BASELINE.json metric: guided img-steps/s; DDPM-256, 50-step schedules).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl native|reference] [--config 1|2|3|4]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[1], per GPU): DDPM-256 UNet2DModel (random-init, seed 0), batch 8, the guided
regeneration pass of the edit-friendly DDPM inversion: ``reverse_step`` (eta = 1, extracted-style noise maps z_t) +
``SingleColorAttrFunc(target 0.8, channel 0, loss_scale 50)`` after every step, through the drop-in
``SegDiffEditPipeline.edit_image(inversion_method="ddpm", Tskip=...)``.

One bench "step" = ONE PASS of the hot path over the batch = one ``edit_image`` call of ``--denoise-steps`` (default 50: the
whole 50-step schedule of the metric) guided denoising steps; each denoising step is one UNet forward (tcgen05 kernels) + one
fused step kernel.  K bench steps are timed, so the default driver run (K = 20) holds 1000 denoising steps (~5 s) inside
each timed region and the SM clock settles.  value = images x denoising steps / second over all GPUs (weak scaling: the batch
is sharded per GPU, no data-path collective; one NCCL all_gather of the final images after every pass).

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the roofline arithmetic and the extra keys."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "diffusion-image-editing_b200")

import torch  # noqa: E402

METRIC = "guided img-steps/s (DDPM-256 UNet, 50-step schedule: edit-friendly DDPM regeneration step + colour guidance)"
UNIT = "img-steps/s"
TARGET, CHANNEL, LOSS_SCALE, ETA, T_INFER = 0.8, 0, 50.0, 1.0, 50
T_START = time.time()


def use_package():
    for p in (REPO, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)


def peaks():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), tf_burst=float(p["bf16_tflops"]),
                    tf_sust=float(p["bf16_tflops_sustained"]), src="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms during the timed region (rank 0's GPU)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0, enabled=True):
        self.index, self.rows, self.proc, self.enabled = index, [], None, enabled

    def __enter__(self):
        if not self.enabled:     # only the reporting rank samples: N polling nvidia-smi processes perturb an N-rank run
            return self
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            self.th.join(timeout=1)

    def summary(self):
        sm, pw, reasons, mx = [], [], set(), None
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                pw.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None, "sm_max_mhz": mx,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU reference arm
def cpu_reference_sample(n_denoise, warm, budget_s):
    """The reference's own CPU implementation of the headline step: the UNMODIFIED reference functions from
    baseline/_ref/src (oracle/ref_harness.py: diffusion_loop, get_noise_pred, get_variance_noise, reverse_step,
    AttrFunc.apply in the order of src/SegDiffEditPipeline.py:248-296; UNet2DModel / DDIMScheduler = the oracle
    restatements of the absent diffusers package), fp32, all host threads, batch 1 (the reference is batch-1 by
    construction: src/transforms.py:31, src/utils.py:49-51).  Falls back to the oracle port when baseline/_ref is missing.
    Returns (img-steps/s, denoising steps timed, s/denoising step, kind, description)."""
    if REPO not in sys.path:
        sys.path.append(REPO)
    torch.set_num_threads(os.cpu_count() or 1)
    from oracle import ref_harness as rh
    g = torch.Generator().manual_seed(7)
    x = torch.randn(1, 3, 256, 256, generator=g)
    if rh.available():
        ref = rh.load_reference()
        w = rh.build_ddpm256(ref, clip_sample=False, num_inference_steps=T_INFER)

        def run(n):
            zs = torch.randn(n, 3, 256, 256, generator=g)
            return rh.config2_regeneration(ref, w, x, zs, n, eta=ETA, target=TARGET, color_idx=CHANNEL, loss_scale=LOSS_SCALE)[1]
        kind = "reference"
        what = ("UNMODIFIED reference functions from baseline/_ref/src (diffusion_loop, get_noise_pred, get_variance_noise, "
                "reverse_step, SingleColorAttrFunc.apply composed as src/SegDiffEditPipeline.py:248-296; diffusers' UNet2DModel / "
                "DDIMScheduler = oracle restatements), torch-CPU fp32")
    else:
        from oracle import loops
        from oracle.ddim_scheduler import DDIMScheduler
        from oracle.unet2d import DDPM256_CONFIG, UNet2DModel
        torch.manual_seed(0)
        unet = UNet2DModel(**DDPM256_CONFIG).eval()
        sch = DDIMScheduler.from_preset("ddpm", clip_sample=False)
        sch.set_timesteps(T_INFER)
        guide = loops.color_guidance([TARGET, None, None], [1, 1, 1], LOSS_SCALE, 0, 10 ** 9)

        def eps_fn(xx, t):
            with torch.no_grad():
                return unet(xx, torch.tensor(t))["sample"]

        def run(n):
            zs = torch.randn(n, 3, 256, 256, generator=g)
            t0 = time.perf_counter()
            loops.guided_edit_loop(sch, eps_fn, x, eta=ETA, zs=zs, guidance=guide, mode="ddpm")
            return time.perf_counter() - t0
        kind = "port"
        what = "oracle port of the reference CPU path (baseline/_ref missing), torch-CPU fp32"
    per = run(max(1, warm)) / max(1, warm)
    n = max(1, min(n_denoise, int(budget_s / max(per, 1e-3))))
    dt = run(n)
    return n / dt, n, dt / n, kind, what


def run_reference(args, rank):
    """--impl reference: K bench steps, each a bounded sample (2 denoising steps at batch 1) of the headline workload."""
    if rank != 0:
        return
    per_step = 2
    # one untimed denoising step first (thread pools, oneDNN primitive caches), then K x per_step denoising steps in one
    # go, bounded by a 150 s budget (the sample actually timed is stated in cpu_baseline.sample)
    v, n, per, kind, what = cpu_reference_sample(args.steps * per_step, 1, 150.0)
    cores = torch.get_num_threads()
    sample = (f"{what}; batch 1; {n} denoising steps timed ({per:.2f} s each) = {n / per_step:.1f} of the {args.steps} requested "
              f"bench steps of {per_step} denoising steps each (bounded sample of the 50-step pass), {cores} threads")
    cfg = workload_config(args, 1, per_step)
    cfg["reference_arm"] = "batch 1 (the reference's native batch), 2 denoising steps per bench step"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per * per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(args, batch, denoise_steps):
    return {"workload": "BASELINE configs[1]: DDPM-256 UNet2DModel (random-init) colour-guided regeneration pass of the "
                        "edit-friendly DDPM inversion (reverse_step eta=1 + SingleColorAttrFunc after every step), per-GPU "
                        f"batch {batch}; one bench step = one edit_image call of {denoise_steps} denoising steps",
            "batch_per_gpu": batch, "global_batch": batch * args.gpus, "image": "3x256x256",
            "num_inference_steps": T_INFER, "denoising_steps_per_bench_step": denoise_steps, "eta": ETA,
            "guidance": "SingleColorAttrFunc(target=0.8,color_idx=0,loss_scale=50,per_sample=True): the loss mean runs over "
                        "each image (H*W), not over the batch (B*H*W) as the reference's batch mean would - a batch is B "
                        "independent batch-1 problems and the result does not depend on how the batch is sharded",
            "schedule_note": "the metric's 50-step schedule; reverse_step (DDPM, eta=1) costs the same FLOPs / bytes per step "
                             "as the DDIM eta=0 step (extra.batch1 times that one)",
            "parallelism": f"dp{args.gpus} (batch sharded, final NCCL all_gather)",
            "l2": "per-step working set (UNet activations, GBs) exceeds the 126 MB L2; no explicit flush"}


# --------------------------------------------------------------------------- native arm
class Ctx:
    pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="bench steps = passes of --denoise-steps guided denoising steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8, help="images per GPU")
    ap.add_argument("--denoise-steps", type=int, default=T_INFER, help="guided denoising steps per pass (bench step)")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4],
                    help="BASELINE config to put on the headline line (default 2; 1 / 3 / 4 also appear under 'extra')")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip extra.* (other configs, fp32 mode, eager baseline)")
    ap.add_argument("--step-kernel-batch", type=int, default=256)
    ap.add_argument("--profile-out", default=None, help="write the per-op CUDA-event profile (JSON) here")
    ap.add_argument("--precision", default=None, choices=["fp16", "bf16", "fp32"],
                    help="noise predictor: 16-bit operands (default: what the library is built for, fp16) or the fp32-accurate split mode")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed pass of the headline returned as DIR/<name>.npy "
                         "(float32, rank 0's shard; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the native arm's outputs; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    use_package()
    args.warmup = max(args.warmup, 3)
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from b200edit import _C, ops
    from b200edit.distributed import gather_images

    c = Ctx()
    c.args, c.rank, c.world, c.dev, c.dist, c.gather = args, rank, world, dev, dist, gather_images
    c._C, c.ops = _C, ops
    precision = args.precision or _C.fast_precision()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world > 1:
            t = torch.tensor([v], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return v

    def timed(fn, passes):
        """passes x fn() between CUDA events on the launching (current) stream, barrier + synchronize on both sides, max over ranks.
        -> (ms, launches, what the final pass returned)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _C.launch_count()
        e0.record()
        for _ in range(passes - 1):
            fn()
        last = fn()     # each earlier pass's result is freed as it returns; only the final one is kept
        e1.record()
        barrier()
        launches = _C.launch_count() - n0
        if world > 1:
            lt = torch.tensor([launches], device=dev, dtype=torch.int64)
            dist.all_reduce(lt)
            launches = int(lt.item())
        return max_over_ranks(e0.elapsed_time(e1)), launches, last
    c.barrier, c.timed = barrier, timed

    headline = {1: config1, 2: config2, 3: config3, 4: config4}[args.config]
    with ClockSampler(local_rank, enabled=(rank == 0)) as clk:
        res = headline(c, precision, args.batch if args.config == 2 else None, args.steps, args.warmup, headline=True)
    last_output = res.pop("last_output", None)
    if args.dump_outputs and rank == 0:
        dump_outputs(last_output, args.dump_outputs)
    del last_output
    line = None
    if rank == 0:
        line = {"metric": METRIC if args.config == 2 else res["metric"], "value": res["value"], "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_pass"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": precision if precision != "fp32" else "fp32-accurate (split fp16 hi+lo operands, 3 tensor-core products per GEMM, fp32 accumulation)",
                "data": "synthetic", "config": res["config"], "clocks": clk.summary(), "e2e": res["e2e"],
                "gpu_launches": res["launches"], "timed_region_s": res["timed_region_s"]}
        line.update(res.get("rooflines", {}))
    # ---- extras: the other BASELINE configs, the fp32-accurate mode, the torch-eager GPU baseline (short runs, same process)
    extra = {}
    if not args.no_extras:
        todo = []
        if args.config != 1:
            todo.append(("batch1", lambda: config1(c, precision, 1, 3, 1)))
        if args.config == 2 and precision != "fp32":
            todo.append(("fp32_accurate", lambda: config2(c, "fp32", args.batch, 2, 1)))
        if args.config != 3:
            todo.append(("config3", lambda: config3(c, precision, None, 2, 1)))
        if args.config != 4:
            todo.append(("config4", lambda: config4(c, precision, None, 2, 1)))
        if args.config == 2:
            todo.append(("batch_sweep", lambda: batch_sweep(c, precision)))
        for name, fn in todo:
            # every rank must take the same branch (the extras synchronise across ranks): agree on the time guard and on
            # failures collectively
            if max_over_ranks(1.0 if time.time() - T_START > 240 else 0.0) > 0:
                extra[name] = {"skipped": "time guard (240 s)"}
                continue
            try:
                r = fn()
                r.pop("rooflines", None)
                extra[name] = r
            except Exception as ex:   # an extra must never take the headline line down
                extra[name] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
                if world > 1:         # a rank that failed inside a collective region cannot rejoin safely: stop the extras
                    break
            torch.cuda.empty_cache()
        if world == 1:
            try:
                extra["gpu_eager_baseline"] = gpu_eager_baseline(c, args.batch)
            except Exception as ex:
                extra["gpu_eager_baseline"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    if rank == 0:
        line["extra"] = extra
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            # in its own process: the reference's bare module names (attr_functions, utils, ...) are the drop-in package's too
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                                   capture_output=True, text=True, timeout=300)
                cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception as ex:
                cpu = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def pass_result(c, name, B, D, K, ms_dev, ms_e2e, launches, h2d, d2h, cfg, flops_per_img_step=None, how_e2e=""):
    world = c.world
    out = {"workload": name, "value": world * B * D * K / (ms_dev * 1e-3), "unit": UNIT, "batch_per_gpu": B,
           "denoising_steps_per_pass": D, "passes": K, "ms_per_pass": ms_dev / K, "ms_per_denoising_step": ms_dev / (K * D),
           "timed_region_s": ms_dev * 1e-3, "launches": launches, "config": cfg,
           "e2e": {"value": world * B * D * K / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "ms_per_step": ms_e2e / K, "how": how_e2e}}
    if flops_per_img_step:
        out["tflops_per_img_step_as_executed"] = flops_per_img_step / 1e12
        out["achieved_tflops_per_gpu"] = flops_per_img_step * B * D * K / (ms_dev * 1e-3) / 1e12
    return out


def dump_outputs(out, out_dir, max_elems=4 << 20):
    """Writes the EditorOutput of the last timed pass as out_dir/<field>.npy in float32: ``imgs`` and the per-step histories
    ``pred_original_samples`` / ``model_outputs`` stacked to (steps, ...).  An array of more than max_elems elements (16 MB)
    is replaced by a fixed sample: the same seeded element positions of every step, shape (steps, n) ((1, n) for ``imgs``),
    so that two builds compare element for element and the three files stay under 48 MB together."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        a = (v if torch.is_tensor(v) else torch.stack(list(v))).detach().float()
        if a.numel() > max_elems:
            rows = a.reshape(a.shape[0] if not torch.is_tensor(v) else 1, -1)
            pick = torch.randperm(rows.shape[1], generator=torch.Generator().manual_seed(0))[:max_elems // rows.shape[0]]
            a = rows[:, pick.sort().values.to(rows.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


# ----- BASELINE configs[1]: the headline
def config2(c, precision, B, K, W, headline=False):
    from attr_functions import SingleColorAttrFunc
    from models import create_diffusion_model
    from SegDiffEditPipeline import SegDiffEditPipeline
    args, dev, world, rank = c.args, c.dev, c.world, c.rank
    D = args.denoise_steps
    wrapper = create_diffusion_model("ddpm", sample_clipping=False, max_batch=B, seed=0, precision=precision)
    sch = wrapper.scheduler
    sch.set_timesteps(max(T_INFER, D))
    if os.environ.get("B2E_BENCH_GRAPH_HEADLINE") == "1":      # experiment knob (profiles/README.md): no gain at batch 8
        wrapper.unet.enable_cuda_graph()
    pipe = SegDiffEditPipeline(wrapper, None)
    f = SingleColorAttrFunc(target=TARGET, color_idx=CHANNEL, loss_scale=LOSS_SCALE, t1=0, t2=10 ** 9, per_sample=True)
    gen = torch.Generator().manual_seed(1000 + rank)        # per-rank shard of the global batch
    S = 256
    # host (pinned) copies of the inputs: x_T shard and the noise maps of every step ((C,H,W) per step, broadcast over the
    # batch like the reference's zs[step_idx]); pinned buffers for the results
    x_host = torch.randn(B, 3, S, S, generator=gen).pin_memory()
    zs_host = torch.randn(D, 3, S, S, generator=gen).pin_memory()
    out_host = torch.empty(B, 3, S, S).pin_memory()
    x0_host = torch.empty(D, B, 3, S, S).pin_memory()
    x_dev, zs_dev = x_host.to(dev), zs_host.to(dev)

    def run(from_host):
        """One pass = one public pipeline call.  from_host: H2D of x_T / z inside, D2H of the results inside."""
        if from_host:
            x = x_host.to(dev, non_blocking=True)
            zs = zs_host.to(dev, non_blocking=True)
        else:
            x, zs = x_dev, zs_dev
        # host leg: the x0-prediction history streams to pinned host memory step by step on the pipeline's copy stream
        # (overlapped with the next step's UNet forward, joined before the call returns); the final images follow
        out = pipe.edit_image(xt=x, eta=ETA, zs=zs, attr_func=f, inversion_method="ddpm", Tskip=0, xts=None,
                              prog_bar=False, output_type="tensor", x0_history_out=x0_host if from_host else None)
        if from_host:
            out_host.copy_(out.imgs, non_blocking=True)
        if world > 1:
            c.gather(out.imgs, world * B)     # the path's only collective: final result gather (NCCL)
        return out

    for _ in range(W):      # W untimed passes of each shape (plans, function attributes, allocator growth, lazy NCCL setup)
        run(False)
    run(True)
    ms_dev, launches, _ = c.timed(lambda: run(False), K)
    ms_e2e, _, last = c.timed(lambda: run(True), K)
    h2d = (x_host.numel() + zs_host.numel()) * 4
    d2h = (out_host.numel() + x0_host.numel()) * 4
    res = pass_result(c, "BASELINE configs[1]", B, D, K, ms_dev, ms_e2e, launches, h2d, d2h, workload_config(args, B, D),
                      wrapper.unet.flops_per_sample,
                      "SegDiffEditPipeline.edit_image from pinned host x_T / z maps; the x0-prediction history (copied step by "
                      "step on a side stream, overlapped with the next UNet forward, joined before the end event) and the final "
                      "images land in pinned host memory inside the timed region; bytes are per bench step (pass)")
    res["precision"] = precision
    if headline and c.args.dump_outputs:
        res["last_output"] = last
    if headline and rank == 0:
        res["rooflines"] = rooflines(c, wrapper, sch, x_dev, precision)
    del pipe, wrapper
    return res


def rooflines(c, wrapper, sch, x_dev, precision):
    """Tensor roofline of the tcgen05 convolution kernel over ALL its launches of one forward (FLOP-weighted; ALGORITHMIC
    FLOPs: identity-residual K segments are executed but counted as bytes), per-variant figures, the GroupNorm / other
    shares, and HBM rooflines of the fused step kernels at a batch that exceeds L2."""
    args, ops, dev = c.args, c.ops, c.dev
    pk = peaks()
    prof = wrapper.unet.profile(x_dev, int(sch.timesteps[-1]))
    if args.profile_out:
        with open(args.profile_out, "w") as fo:
            json.dump(prof, fo)
    conv = [p for p in prof if p["kind"] == "conv_igemm"]
    tot_ms = sum(p["ms"] for p in prof)
    by_kind = {}
    for p in prof:
        d = by_kind.setdefault(p["kind"], {"ms": 0.0, "launch_groups": 0})
        d["ms"] += p["ms"]
        d["launch_groups"] += 1
    try:
        with open(os.path.join(REPO, "profiles", "ncu_traffic.json")) as f:
            ncu = json.load(f)
    except Exception:
        ncu = {}

    def tensor_roofline(launches, kernel):
        ms = sum(p["ms"] for p in launches)
        fl = sum(p["flops"] for p in launches)
        ach = fl / (ms * 1e-3) / 1e12
        return {"bound": "tensor", "kernel": kernel, "achieved": ach, "peak": pk["tf_burst"], "unit": "TFLOP/s",
                "frac": ach / pk["tf_burst"], "frac_of_sustained": ach / pk["tf_sust"],
                "peak_source": pk["src"] + ", burst bf16 (each launch is event-timed alone; fp16 operands run at the same "
                               "UTCHMMA rate)", "launches": len(launches),
                "flops_per_launch": fl / max(1, len(launches)), "us_per_launch": ms * 1e3 / max(1, len(launches)),
                "share_of_unet_time": ms / tot_ms,
                "how": "ALGORITHMIC FLOPs (2*M*N*K of the convolution / linear / attention GEMM; identity-residual K segments "
                       "excluded, counted as bytes; the two large upsampler convolutions are counted as the four 2x2-tap "
                       "sub-pixel phase convolutions actually executed - 2.25x fewer FLOPs than nearest-upsample + 3x3, "
                       "-4 % on the forward) / CUDA-event duration per launch, one instrumented forward (events on the "
                       "launching stream)"}

    roof = tensor_roofline(conv, "conv_igemm_kernel, all variants (every conv / linear / attention GEMM launch of the UNet forward)")
    roof["traffic"] = ncu.get("conv", {}).get("dram_bytes_per_launch")
    roof["traffic_source"] = ncu.get("conv", {}).get("source")
    roof["tensor_pipe_active_pct_ncu"] = ncu.get("conv", {}).get("tensor_pipe_active_pct_time_weighted")
    roof.update({"flops_per_forward": sum(p["flops"] for p in conv), "unet_ms_instrumented": tot_ms,
                 "by_kind_ms": {k: round(v["ms"], 4) for k, v in by_kind.items()}})
    variants = {}
    for key, tag in (("halo2_256x256", "halo2"), ("halo1", "halo1"), ("pair", " pair"), ("splitK", "splitK")):
        sel = [p for p in conv if tag in p["desc"]]
        if sel:
            variants[key] = {k: v for k, v in tensor_roofline(sel, tag.strip()).items()
                             if k in ("achieved", "frac", "frac_of_sustained", "launches", "us_per_launch", "share_of_unet_time")}
    # ---- HBM rooflines of the fused step kernels at a batch that exceeds L2 (algorithmic bytes per element, DESIGN.md section 4)
    Bs, S = args.step_kernel_batch, 256
    xs = torch.randn(Bs, 3, S, S, device=dev)
    es = torch.randn(Bs, 3, S, S, device=dev)
    x0r = torch.randn(Bs, 3, S, S, device=dev)
    zsb = torch.randn(3, S, S, device=dev)
    mask = (torch.rand(1, 3, S, S, device=dev) > 0.5).float()
    coef = sch.coeffs(int(sch.timesteps[-5]), ETA, "ddpm")

    def hbm(fn, bytes_per_elem, name, reps=10):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        by = bytes_per_elem * xs.numel()
        gbs = by / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": name, "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                "peak_source": pk["src"], "batch": Bs, "bytes_per_elem": bytes_per_elem, "bytes_per_launch": by,
                "ms_per_launch": ms}

    kw = dict(noise=zsb, targets=[TARGET, None, None], loss_scale=LOSS_SCALE, n_mean=S * S)
    step = hbm(lambda: ops.guided_step(xs, es, coef, **kw), 16.0,
               "guided_step_vec4 (fused x0 + DDPM step + sigma*z + colour guidance): read x_t, eps; write x_prev, x0")
    step["traffic"] = ncu.get("step", {}).get("dram_bytes_per_launch")
    step["traffic_source"] = ncu.get("step", {}).get("source")
    step["how"] = "16 B/elem algorithmic bytes / CUDA-event time, working set 4x%.0f MB > L2" % (xs.numel() * 4 / 1e6)
    others = {}
    try:
        others["guided_step_l2reg (two passes, masked + L2-regularised guidance)"] = hbm(
            lambda: ops.guided_step_l2reg(xs, es, coef, noise=zsb, targets=[TARGET, None, None], loss_scale=LOSS_SCALE, mask=mask,
                                          x_ref=x0r, lambda_=0.1), 36.0, "l2reg_pass1 + l2reg_pass2")
    except Exception as ex:
        others["guided_step_l2reg"] = {"error": str(ex)[:200]}
    try:
        zout = torch.empty_like(xs)
        xm = x0r.clone()
        others["extract_noise (z_t extraction, in-place correction)"] = hbm(
            lambda: ops.extract_noise(xs, es, xm, zout, coef), 20.0, "extract_noise_kernel")
    except Exception as ex:
        others["extract_noise"] = {"error": str(ex)[:200]}
    try:
        others["pred_x0 (map2)"] = hbm(lambda: ops.pred_x0(xs, es, float(coef.sqrt_a_t), float(coef.sqrt_b_t)), 12.0, "map2_kernel<pred_x0>")
        others["apply_mask"] = hbm(lambda: ops.apply_mask(mask, xs, es), 12.0, "apply_mask_kernel")
        others["to_uint8"] = hbm(lambda: ops.to_uint8(xs), 5.0, "to_uint8_kernel")
    except Exception as ex:
        others["map2/apply_mask/to_uint8"] = {"error": str(ex)[:200]}
    del xs, es, x0r
    torch.cuda.empty_cache()
    return {"roofline": roof, "roofline_conv_variants": variants, "roofline_step_kernel": step, "roofline_step_kernels": others,
            "unet_tflops_per_img_as_executed": wrapper.unet.flops_per_sample / 1e12,
            "unet_tflops_per_img_algorithmic": sum(p["flops"] for p in conv) / x_dev.shape[0] / 1e12}


# ----- BASELINE configs[0] on the GPU: DDIM eta = 0, clip_sample, batch 1 (the reference's native batch)
def config1(c, precision, B, K, W, headline=False):
    from attr_functions import SingleColorAttrFunc
    from models import create_diffusion_model
    from SegDiffEditPipeline import SegDiffEditPipeline
    B = B or 1
    D = c.args.denoise_steps
    w = create_diffusion_model("ddpm", sample_clipping=True, max_batch=B, seed=0, precision=precision)
    w.scheduler.set_timesteps(max(T_INFER, D))
    if os.environ.get("B2E_BENCH_GRAPH", "1") != "0":
        w.unet.enable_cuda_graph()     # batch 1 is launch-bound: replay the forward as one CUDA graph
    pipe = SegDiffEditPipeline(w, None)
    f = SingleColorAttrFunc(target=0.8, color_idx=0, loss_scale=100.0, t1=0, t2=10 ** 9, per_sample=True)
    x_host = torch.randn(B, 3, 256, 256, generator=torch.Generator().manual_seed(1234)).pin_memory()
    out_host = torch.empty(B, 3, 256, 256).pin_memory()
    x0_host = torch.empty(max(T_INFER, D), B, 3, 256, 256).pin_memory()
    x_dev = x_host.to(c.dev)

    def run(from_host):
        x = x_host.to(c.dev, non_blocking=True) if from_host else x_dev
        out = pipe.edit_image(xt=x, eta=0.0, attr_func=f, prog_bar=False, output_type="tensor",
                              x0_history_out=x0_host if from_host else None)
        if from_host:
            out_host.copy_(out.imgs, non_blocking=True)
        return out
    for _ in range(W):
        run(False)
    run(True)
    D = max(T_INFER, D)    # eta = 0 walks the whole schedule
    ms_dev, launches, _ = c.timed(lambda: run(False), K)
    ms_e2e, _, last = c.timed(lambda: run(True), K)
    cfg = {"workload": f"BASELINE configs[0] on the GPU: DDPM-256, colour-guided DDIM (eta=0, clip_sample) {D} steps, batch {B}",
           "batch_per_gpu": B, "guidance": "SingleColorAttrFunc(target=0.8,color_idx=0,loss_scale=100)"}
    res = pass_result(c, "BASELINE configs[0] (GPU)", B, D, K, ms_dev, ms_e2e, launches, x_host.numel() * 4,
                      (out_host.numel() + x0_host.numel()) * 4, cfg, w.unet.flops_per_sample, "as the headline")
    res["metric"] = "guided img-steps/s (DDPM-256, colour-guided DDIM-50, batch 1)"
    res["precision"] = precision
    if headline and c.args.dump_outputs:
        res["last_output"] = last
    res["cuda_graph"] = bool(w.unet._graph_on)
    del pipe, w
    return res


# ----- BASELINE configs[4]: colour-guided DDIM throughput over the batch size (per GPU of this run)
def batch_sweep(c, precision, batches=(2, 4, 16, 32, 64, 128, 256), D=4, K=2):
    """img-steps/s of the colour-guided DDIM step (configs[0]'s workload) at each batch size, HBM-resident inputs, a D-step
    schedule (the per-step work does not depend on the schedule length), K passes after one warm-up pass."""
    from attr_functions import SingleColorAttrFunc
    from models import create_diffusion_model
    from SegDiffEditPipeline import SegDiffEditPipeline
    f = SingleColorAttrFunc(target=0.8, color_idx=0, loss_scale=100.0, t1=0, t2=10 ** 9, per_sample=True)
    points = []
    for B in batches:
        w = create_diffusion_model("ddpm", sample_clipping=True, max_batch=B, seed=0, precision=precision)
        w.scheduler.set_timesteps(D)
        pipe = SegDiffEditPipeline(w, None)
        x = torch.randn(B, 3, 256, 256, generator=torch.Generator().manual_seed(77 + c.rank)).to(c.dev)
        run = lambda: pipe.edit_image(xt=x, eta=0.0, attr_func=f, prog_bar=False, output_type="tensor")   # noqa: E731
        run()
        ms, _, _ = c.timed(run, K)
        points.append({"batch_per_gpu": B, "value": c.world * B * D * K / (ms * 1e-3), "ms_per_denoising_step": ms / (K * D),
                       "achieved_tflops_per_gpu": B * w.unet.flops_per_sample / (ms / (K * D) * 1e-3) / 1e12})
        del pipe, w, x
        torch.cuda.empty_cache()
    return {"workload": "BASELINE configs[4]: colour-guided DDIM on DDPM-256 over the batch size (batch 1: extra.batch1, batch 8: "
                        "the headline)", "unit": UNIT, "denoising_steps_per_pass": D, "passes": K, "precision": precision,
            "n_gpus": c.world, "points": points}


# ----- BASELINE configs[2]: LDM, segmentation-mask colour guidance THROUGH the VQ decoder
def config3(c, precision, B, K, W, headline=False):
    from attr_functions import SingleColorAttrFunc
    from models import create_diffusion_model
    from SegDiffEditPipeline import SegDiffEditPipeline
    B = B or 32
    D = 4 if not headline else min(c.args.denoise_steps, 10)
    w = create_diffusion_model("ldm", sample_clipping=False, max_batch=B, seed=0, precision=precision)
    w.scheduler.set_timesteps(D)
    pipe = SegDiffEditPipeline(w, None)
    g = torch.Generator().manual_seed(2)
    x_host = torch.randn(B, 3, 64, 64, generator=g).pin_memory()
    # hair-like blob mask at latent resolution (the parsing-map fixtures live in the reference tree, absent on the GPU box)
    yy, xx = torch.meshgrid(torch.arange(64.0), torch.arange(64.0), indexing="ij")
    mask = (((yy - 20) / 18) ** 2 + ((xx - 32) / 24) ** 2 <= 1).float().expand(1, 3, 64, 64).contiguous().to(c.dev)
    f = SingleColorAttrFunc(target=0.8, color_idx=0, loss_scale=50.0, t1=0, t2=10 ** 9, use_mask=True, mask_attr_grad=True)
    out_host = torch.empty(B, 3, 256, 256).pin_memory()
    x_dev = x_host.to(c.dev)

    def run(from_host):
        x = x_host.to(c.dev, non_blocking=True) if from_host else x_dev
        out = pipe.edit_image(xt=x, attr_func=f, prog_bar=False, output_type="tensor", mask=mask)
        if from_host:
            out_host.copy_(out.imgs, non_blocking=True)
        return out
    for _ in range(W):
        run(False)
    run(True)
    ms_dev, launches, _ = c.timed(lambda: run(False), K)
    ms_e2e, _, last = c.timed(lambda: run(True), K)
    fl = w.unet.flops_per_sample + w.vqvae.flops_per_sample   # gradient mode: the decoder figure counts forward + backward
    cfg = {"workload": f"BASELINE configs[2]: LDM-CelebAHQ layout (64x64x3 latent, random-init), masked colour guidance through the "
                       f"native VQ decoder (forward + latent gradient), batch {B}, {D} DDIM steps per pass + one final decode",
           "batch_per_gpu": B, "guidance": "SingleColorAttrFunc(use_mask, mask_attr_grad), decode inside the guidance graph"}
    res = pass_result(c, "BASELINE configs[2]", B, D, K, ms_dev, ms_e2e, launches, x_host.numel() * 4, out_host.numel() * 4, cfg, fl,
                      "edit_image from a pinned host latent batch; decoded images copied to pinned host memory")
    res["metric"] = "guided img-steps/s (LDM 64x64x3 latent, mask guidance through the VQ decoder)"
    res["precision"] = precision
    if headline and c.args.dump_outputs:
        res["last_output"] = last
    res["max_memory_gb"] = torch.cuda.max_memory_allocated() / 1e9
    del pipe, w
    return res


# ----- BASELINE configs[3]: SD 1.x, CFG + classifier guidance through the KL decoder and the ResNet-50 predictor
def config4(c, precision, B, K, W, headline=False):
    from attr_functions import ClassifierAttrFunc
    from models import create_diffusion_model, get_pretrained_anyGAN
    from SegDiffEditPipeline import SegDiffEditPipeline
    B = B or 8
    D = 3 if not headline else min(c.args.denoise_steps, 6)
    pprec = os.environ.get("B2E_BENCH_PREDICTOR_PRECISION", "fp32")    # get_pretrained_anyGAN's default: fp32-accurate forward
    predictor = get_pretrained_anyGAN(input_size=512, max_batch=B, precision=pprec)
    w = create_diffusion_model("sd", sample_clipping=False, max_batch=B, seed=0, precision=precision, with_encoder=False)
    w.scheduler.set_timesteps(D)
    pipe = SegDiffEditPipeline(w, None)
    x_host = torch.randn(B, 4, 64, 64, generator=torch.Generator().manual_seed(4 + c.rank)).pin_memory()
    text_emb = torch.randn(2, 77, 768, generator=torch.Generator().manual_seed(3)).to(c.dev)   # no tokenizer files offline
    w.additional_prep = lambda model, prompt: text_emb
    f = ClassifierAttrFunc(predictor, idx_for_class=31, idx_of_interest=0, loss_scale=50.0, t1=0, t2=10 ** 9)
    out_host = torch.empty(B, 3, 512, 512).pin_memory()
    x_dev = x_host.to(c.dev)

    def run(from_host):
        x = x_host.to(c.dev, non_blocking=True) if from_host else x_dev
        out = pipe.edit_image(xt=x, attr_func=f, prompt="a photo of a face", cfg_scale=7.5, prog_bar=False, output_type="tensor")
        if from_host:
            out_host.copy_(out.imgs, non_blocking=True)
        if c.world > 1:
            c.gather(out.imgs, c.world * B)
        return out
    for _ in range(W):
        run(False)
    run(True)
    ms_dev, launches, _ = c.timed(lambda: run(False), K)
    ms_e2e, _, last = c.timed(lambda: run(True), K)
    fl = 2 * w.unet.flops_per_sample + w.vae.flops_per_sample
    cfg = {"workload": f"BASELINE configs[3]: Stable Diffusion 1.x layout (64x64x4 latent, random-init), CFG 7.5 (doubled latent batch, "
                       f"precomputed (2,77,768) text embedding) + classifier guidance through the native KL decoder and ResNet-50 "
                       f"predictor (forward + gradient), batch {B} per GPU, {D} DDIM steps per pass + one final decode",
           "batch_per_gpu": B, "global_batch": B * c.world, "guidance": "ClassifierAttrFunc(idx_for_class=31, idx_of_interest=0)",
           "predictor_precision": pprec}
    res = pass_result(c, "BASELINE configs[3]", B, D, K, ms_dev, ms_e2e, launches, x_host.numel() * 4, out_host.numel() * 4, cfg, fl,
                      "edit_image from a pinned host latent batch; decoded 512x512 images copied to pinned host memory")
    res["metric"] = "guided img-steps/s (SD-1.x 64x64x4 latent, CFG + classifier guidance)"
    res["precision"] = precision
    if headline and c.args.dump_outputs:
        res["last_output"] = last
    res["max_memory_gb"] = torch.cuda.max_memory_allocated() / 1e9
    del pipe, w, predictor
    return res


# ----- the informative GPU baseline: what a diffusers + PyTorch user gets on this B200 (torch eager, cuDNN)
def gpu_eager_baseline(c, B):
    """The headline step with the oracle restatement of diffusers' UNet2DModel run by torch eager (cuDNN / cuBLAS) on the
    same GPU, and the reference's step math as torch element-wise ops (oracle.step_math: the ~40 ATen launches per step the
    fused kernel replaces).  Checker code used as a BASELINE only; fp16 (what the native headline computes in), bf16 and fp32."""
    if REPO not in sys.path:
        sys.path.append(REPO)
    from oracle import step_math as sm
    from oracle.ddim_scheduler import DDIMScheduler
    from oracle.unet2d import DDPM256_CONFIG, UNet2DModel
    dev = c.dev
    sch = DDIMScheduler.from_preset("ddpm", clip_sample=False)
    sch.set_timesteps(T_INFER)
    ts = [int(t) for t in sch.timesteps]
    out = {}
    g = torch.Generator().manual_seed(1000)
    x0 = torch.randn(B, 3, 256, 256, generator=g).to(dev)
    zs = torch.randn(8, 3, 256, 256, generator=g).to(dev)
    for name, dt, tf32 in (("fp16", torch.float16, False), ("bf16", torch.bfloat16, False), ("fp32_tf32_off", torch.float32, False),
                           ("fp32_tf32_on", torch.float32, True)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
        torch.manual_seed(0)
        unet = UNet2DModel(**DDPM256_CONFIG).eval().to(dev).to(dt)

        def steps(n, x):
            for i in range(n):
                t = ts[-8 + (i % 8)]
                with torch.no_grad():
                    eps = unet(x.to(dt), torch.tensor(t, device=dev))["sample"].float()
                cf = sm.step_coeffs(sch, t)
                xp, _ = sm.ddpm_reverse_step(x, eps, cf, ETA, zs[i % 8])
                x, _ = sm.color_guidance_update(xp, eps, cf, [TARGET, None, None], [1, 1, 1], LOSS_SCALE)
            return x
        steps(2, x0)
        torch.cuda.synchronize()
        n = 6
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        steps(n, x0)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        out[name] = {"value": B / ms * 1e3, "unit": UNIT, "ms_per_denoising_step": ms, "batch": B}
        del unet
        torch.cuda.empty_cache()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    out["what"] = ("oracle restatement of diffusers' UNet2DModel (DDPM-256 layout) in torch eager on this GPU (cuDNN / cuBLAS) + the "
                   "reference's step math as torch element-wise ops, same batch and step as the headline, device-resident inputs; "
                   "not the reference arm (that is the CPU path) - the number a diffusers + PyTorch user would see on this box")
    return out


if __name__ == "__main__":
    main()
