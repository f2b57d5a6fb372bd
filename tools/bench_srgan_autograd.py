"""Cost of the differentiable SRGAN generator at the C3 geometry (batch 32, 64x128 latent -> 256x512; bench.py's C3 workload
weights) and of guidance through it.

Times, with CUDA events and after warm-up, the median of --iters calls of
  1. the no-grad forward (wc_srgan_forward, the inference plan);
  2. the saved forward (wc_srgan_forward_saved, the with-grad plan) and the seeded backward (wc_srgan_backward_seeded);
  3. the backward's per-op breakdown from the library's per-launch CUDA-event profile (one backward, eager);
  4. one eager GSG translation step with the pooled stand-in avg_pool2d(dL/d sr, 4) (bench.py's step) against one step guided
     through the generator (sgg.apply_gsg_through_srgan).
The arms of 1-2 and of 4 alternate call by call.  Reports the with-grad plan's workspace and the card name and power limit
read in the same run.  Writes one JSON line.
usage: python tools/bench_srgan_autograd.py [--iters 20] [--warmup 3] [--out PATH]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch


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


def backward_op_labels(num_blocks, n_up):
    """Library launches of wc_srgan_backward_seeded in plan order (csrc/srgan.cu)."""
    labels = ["final: tanh derivative", "final: 3->64 9x9 data gradient (CUDA cores)"]
    for u in reversed(range(n_up)):
        labels += [f"upsampler {u}: PixelShuffle + PReLU backward", f"upsampler {u}: 256->64 3x3 data gradient"]
    labels.append("convblock: 3x3 data gradient")
    for i in reversed(range(num_blocks)):
        labels += [f"block {i}: block2 data gradient", f"block {i}: PReLU backward", f"block {i}: block1 data gradient"]
    labels += ["initial: PReLU backward", "initial: 64->3 9x9 data gradient (CUDA cores)"]
    return labels


def group_of(label):
    if label.startswith("final"):
        return "final_layer"
    if label.startswith("upsampler"):
        return "upsamplers"
    if label.startswith("initial"):
        return "initial_layer"
    return "prelu_elementwise" if "PReLU" in label else "trunk_dgrad_igemm"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "r3_srgan_autograd_c3.json"))
    a = ap.parse_args()
    if a.iters < 20:
        raise SystemExit("--iters must be at least 20")
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from bench import WORKLOADS, GpuWorkload
    from weatherconverter_b200 import _lib, ops
    from weatherconverter_b200._lib import check, ptr, stream_ptr
    from weatherconverter_b200.sgg.sgg import apply_gsg_through_srgan

    lib = _lib.lib()
    dev = torch.device("cuda")
    spec = dict(WORKLOADS["c3"])
    wl = GpuWorkload(spec, dev, 0)
    G = wl.srgan
    B, h, w = spec["batch"], spec["h"], spec["w"]
    x = torch.rand(B, 3, h, w, generator=torch.Generator().manual_seed(1234)).to(dev) * 2 - 1
    y = torch.empty(B, 3, 4 * h, 4 * w, device=dev)
    dy = torch.randn(B, 3, 4 * h, 4 * w, generator=torch.Generator().manual_seed(1235)).to(dev) * 1e-3
    dx = torch.empty_like(x)
    plan = G._grad_plan(B, h, w, x.device)

    def timed(fn):
        torch.cuda.synchronize()
        n0 = ops.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1), ops.launch_count() - n0, out

    def nograd():
        with torch.no_grad():
            return G(x, out=y)

    def saved():
        check(lib.wc_srgan_forward_saved(plan.handle, ptr(x), ptr(y), B, h, w, ptr(plan.ws), plan.ws.numel(), stream_ptr()))

    def backward():
        check(lib.wc_srgan_backward_seeded(plan.handle, ptr(dy), ptr(dx), stream_ptr()))

    ms = {"nograd_forward": [], "saved_forward": [], "seeded_backward": []}
    launches = {}
    for _ in range(a.warmup):
        nograd(); saved(); backward()
    for _ in range(a.iters):
        for k, fn in (("nograd_forward", nograd), ("saved_forward", saved), ("seeded_backward", backward)):
            t, n, _ = timed(fn)
            ms[k].append(t)
            launches[k] = n

    # ---- per-op breakdown of one backward (CUDA events around every library launch, eager)
    saved()
    torch.cuda.synchronize()
    lib.wc_profile_begin()
    backward()
    torch.cuda.synchronize()
    cap = 4096
    c_cls, c_ms, c_work, c_info = (C.c_int * cap)(), (C.c_double * cap)(), (C.c_double * cap)(), (C.c_int * (6 * cap))()
    nrec = min(cap, lib.wc_profile_detail(cap, c_cls, c_ms, c_work, c_info))
    ms_c, cnt_c, work_c = (C.c_double * 8)(), (C.c_longlong * 8)(), (C.c_double * 8)()
    check(lib.wc_profile_end(ms_c, cnt_c, work_c))
    op_ms = [c_ms[i] for i in range(nrec)]
    labels = backward_op_labels(G.num_blocks, G.upscale_factor // 2)
    breakdown, groups = None, {}
    if len(labels) == nrec:
        breakdown = [{"op": lb, "ms": t} for lb, t in zip(labels, op_ms)]
        for lb, t in zip(labels, op_ms):
            groups[group_of(lb)] = groups.get(group_of(lb), 0.0) + t
    else:
        breakdown = [{"op": f"launch {i} (class {c_cls[i]})", "ms": op_ms[i]} for i in range(nrec)]

    # ---- one GSG translation step: pooled stand-in vs through the generator
    gen = torch.Generator(device=dev).manual_seed(5)
    z = torch.randn(wl.x0.shape, device=dev, generator=gen)
    state = {"k": 0}

    def step_pooled():
        state["k"] += 1
        return wl.step(wl.x0, state["k"], z)

    def step_through():
        state["k"] += 1
        i = wl.timestep(state["k"])
        wl.unet(wl.x0, wl.t_tensor(i), out=wl.eps)
        mu, sigma, _ = wl.sched.sample_prev_timestep(wl.x0, wl.eps, i, z=z)
        return apply_gsg_through_srgan(wl.seg, G, mu, sigma, wl.x0, wl.gt, 60.0)

    step_ms = {"gsg_step_pooled": [], "gsg_step_through_srgan": []}
    step_launches = {}
    for _ in range(a.warmup):
        step_pooled(); step_through()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    for _ in range(a.iters):
        for k, fn in (("gsg_step_pooled", step_pooled), ("gsg_step_through_srgan", step_through)):
            t, n, _ = timed(fn)
            step_ms[k].append(t)
            step_launches[k] = n

    med = {k: statistics.median(v) for k, v in {**ms, **step_ms}.items()}
    grad_ws = sum(p.ws.numel() for ps in G._grad_plans.values() for p in ps)
    rec = {
        "metric": "differentiable SRGAN generator (C3: batch %d, %dx%d -> %dx%d)" % (B, h, w, 4 * h, 4 * w),
        "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev.index or 0),
        "iters": a.iters, "warmup": a.warmup, "timing": "CUDA events per call, median; arms alternated call by call",
        "nograd_forward_ms": med["nograd_forward"], "saved_forward_ms": med["saved_forward"],
        "seeded_backward_ms": med["seeded_backward"],
        "saved_over_nograd_forward": med["saved_forward"] / med["nograd_forward"],
        "launches": launches,
        "backward_breakdown_ms_by_group": groups, "backward_breakdown": breakdown,
        "backward_breakdown_note": "one eager backward with a CUDA event pair around every library launch",
        "gsg_step_pooled_ms": med["gsg_step_pooled"], "gsg_step_through_srgan_ms": med["gsg_step_through_srgan"],
        "gsg_step_through_over_pooled": med["gsg_step_through_srgan"] / med["gsg_step_pooled"],
        "gsg_step_library_launches": step_launches,
        "nograd_workspace_gib": G._infer.plan.ws.numel() / 2 ** 30,
        "grad_plan_workspace_gib": grad_ws / 2 ** 30,
        "grad_plans": sum(len(ps) for ps in G._grad_plans.values()),
        "hbm_gib_resident_end": torch.cuda.memory_allocated() / 2 ** 30,
        "ms_all": {k: v for k, v in {**ms, **step_ms}.items()},
    }
    plan.busy = False
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
