"""Cost of the differentiable DeepLabV3+ against the fused loss-head plan at the C3 segmentor geometry (ResNet-50, output
stride 16, batch 32, 256x512; the flagship workload's random-init weights, seed 42, and synthetic 8x8 block labels, SURVEY 8d).

Times, with CUDA events and after warm-up, the median of --iters calls of
  1. fused:     DeepLabV3.infer(x, gt) - forward, CE(ignore 255) and the input gradient in one plan;
  2. autograd:  logits = seg(x.requires_grad_()), torch per-image CE, backward;
  3. one eager GSG translation step (UNet + SRGAN + guidance, bench.py's C3 workload) with a custom criterion (per-image CE
     through torch autograd) against the default step, eager and replayed from a CUDA graph.
The arms of 1-2 and of 3 alternate call by call.  Reports library launches per call, the torch allocator's peak per arm, and
the card name and power limit from the same run.  Writes one JSON line.
usage: python tools/bench_seg_autograd.py [--iters 20] [--warmup 3] [--out PATH]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.nn.functional as F


def power_limit_w(index):
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetEnforcedPowerLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out)
    except Exception:
        return None


def per_image_ce(logits, gt):
    ce = F.cross_entropy(logits, gt, ignore_index=255, reduction="none")
    n = (gt != 255).flatten(1).sum(1).clamp_min(1)
    return ce.flatten(1).sum(1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "seg_autograd_c3.json"))
    a = ap.parse_args()
    if a.iters < 20:
        raise SystemExit("--iters must be at least 20")
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from bench import WORKLOADS, GpuWorkload, block_labels
    from weatherconverter_b200 import ops
    from weatherconverter_b200.sgg.sgg import apply_gsg_batch

    dev = torch.device("cuda")
    spec = dict(WORKLOADS["c3"])
    wl = GpuWorkload(spec, dev, 0)                       # UNet, SRGAN and DeepLabV3+-R50 (seed 42) of the C3 workload
    B, H, W = spec["batch"], 4 * spec["h"], 4 * spec["w"]
    seg = wl.seg.shared_replica()                        # own plan binding: the graphed step keeps wl.seg's
    gt = block_labels(torch.Generator().manual_seed(1234), B, H, W).to(dev)
    x = torch.randn(B, 3, H, W, generator=torch.Generator().manual_seed(1234)).to(dev)

    def timed(fn):
        torch.cuda.synchronize()
        n0 = ops.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1), ops.launch_count() - n0, out

    def fused():
        return seg.infer(x, gt)["grad"]

    def autograd():
        xg = x.clone().requires_grad_(True)
        per_image_ce(seg(xg), gt).sum().backward()
        return xg.grad

    def run_arms(arms, warmup, iters):
        ms = {k: [] for k in arms}
        launches, peak = {}, {}
        for _ in range(warmup):
            for fn in arms.values():
                fn()
        for it in range(iters):
            for k, fn in arms.items():
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                base = torch.cuda.memory_allocated()
                t, n, _ = timed(fn)
                ms[k].append(t)
                launches[k] = n
                peak[k] = max(peak.get(k, 0), torch.cuda.max_memory_allocated() - base)
        return ms, launches, peak

    seg_ms, seg_launches, seg_peak = run_arms({"fused": fused, "autograd": autograd}, a.warmup, a.iters)
    g_f, g_a = fused(), autograd()
    grad_rel = float((g_a - g_f).norm() / g_f.norm())
    del g_f, g_a

    # ---- one GSG translation step
    wl.capture()
    gen = torch.Generator(device=dev).manual_seed(5)
    z = torch.randn(wl.x0.shape, device=dev, generator=gen)
    state = {"k": 0}

    def eager_default():
        state["k"] += 1
        return wl.step(wl.x0, state["k"], z)

    def graphed_default():
        state["k"] += 1
        wl.sg.load(wl.x0)
        return wl.graph_step(state["k"], z)

    def eager_custom():
        state["k"] += 1
        i = wl.timestep(state["k"])
        wl.unet(wl.x0, wl.t_tensor(i), out=wl.eps)
        mu, sigma, _ = wl.sched.sample_prev_timestep(wl.x0, wl.eps, i, z=z)
        return apply_gsg_batch(wl.seg, mu, sigma, wl.srgan(wl.x0), wl.gt, 60.0, criterion=per_image_ce)

    step_ms, step_launches, step_peak = run_arms(
        {"eager_default": eager_default, "graphed_default": graphed_default, "eager_custom_criterion": eager_custom},
        a.warmup, a.iters)

    med = {k: statistics.median(v) for k, v in {**seg_ms, **step_ms}.items()}
    rec = {
        "metric": "differentiable DeepLabV3+ vs the fused loss-head plan (C3: R50 os16, batch %d, %dx%d)" % (B, H, W),
        "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev.index or 0),
        "iters": a.iters, "warmup": a.warmup, "timing": "CUDA events per call, median; arms alternated call by call",
        "seg_fused_infer_grad_ms": med["fused"], "seg_autograd_ce_backward_ms": med["autograd"],
        "seg_autograd_over_fused": med["autograd"] / med["fused"],
        "seg_fused_launches": seg_launches["fused"], "seg_autograd_library_launches": seg_launches["autograd"],
        "seg_fused_peak_extra_gib": seg_peak["fused"] / 2 ** 30, "seg_autograd_peak_extra_gib": seg_peak["autograd"] / 2 ** 30,
        "seg_autograd_vs_fused_grad_rms_rel": grad_rel,
        "gsg_step_eager_default_ms": med["eager_default"], "gsg_step_graphed_default_ms": med["graphed_default"],
        "gsg_step_eager_custom_criterion_ms": med["eager_custom_criterion"],
        "gsg_step_custom_over_eager_default": med["eager_custom_criterion"] / med["eager_default"],
        "gsg_step_custom_over_graphed_default": med["eager_custom_criterion"] / med["graphed_default"],
        "gsg_step_library_launches": {k: step_launches[k] for k in step_launches},
        "gsg_step_peak_extra_gib": {k: v / 2 ** 30 for k, v in step_peak.items()},
        "peak_note": "torch allocator peak during one call above what was allocated before it (plan workspaces allocated "
                     "during warm-up are not included); library launches count kernels of libwc_b200 only, not torch's CE",
        "seg_fused_workspace_gib": seg._infer.plan.ws.numel() / 2 ** 30,
        "seg_autograd_workspace_gib": sum(p.ws.numel() for ps in seg._grad_plans.values() for p in ps) / 2 ** 30,
        "hbm_gib_resident_end": torch.cuda.memory_allocated() / 2 ** 30,
        "ms_all": {k: v for k, v in {**seg_ms, **step_ms}.items()},
    }
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
