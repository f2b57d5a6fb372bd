"""Cost of the DDIM sampler against the full DDPM chain, at bench.py's C2 (UNet sampling 128x256, batch 16) and C3 (guided
translation, latent 64x128 -> 256x512, batch 32) workloads and weights.

For each workload, in one process, with CUDA events:
  1. ms per graphed reverse step, DDIM (a 50-step eta = 1 schedule; the table-indexed step kernel) against DDPM
     (ddpm_step_kernel<2>): one StepGraph each, the two arms alternated block by block (--rounds blocks of --steps replays);
  2. the step kernel alone, ddim_step_kernel<2> against ddpm_step_kernel<2>, on 24 x 3 x 128 x 256 fp32 tensors (9.4 MB each):
     --launches launches per arm captured in one CUDA graph, rotating over 8 buffer sets (302 MB, more than the 126 MB L2)
     so every launch reads from HBM; arms alternated;
  3. wall time per batch (host clock around a whole call that ends in a device synchronise, StepGraph capture included) and
     images/s: C2 sample_tensor(use_graph=True) with DDIM K in {50, 100, 250} (eta = 0) against the 1000-step DDPM chain;
     C3 sample_with_sgg(use_graph=True) with DDIM K = 50, eta = 1 against the 500-step DDPM chain.
Writes one JSON line per workload to <out-dir>/r3_ddim_c2.json and r3_ddim_c3.json, with the card name and power limit read
in the same run.
usage: python tools/bench_ddim.py [--which c2,c3] [--rounds 5] [--steps 10] [--launches 200] [--out-dir profiles]"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch

from bench_srgan_autograd import power_limit_w


def events_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def graphed_step_ms(wl, ddim, rounds, steps):
    """Median ms per replay of the DDPM and the DDIM step graphs, alternated block by block."""
    from weatherconverter_b200.graphs import StepGraph

    def ddim_fn(xt, t_dev, z):
        eps = wl.unet(xt, t_dev)
        if wl.spec["kind"] == "ddpm":
            return ddim.step_indexed(xt, eps, t_dev, z)
        from weatherconverter_b200.sgg.sgg import apply_gsg_batch
        mu, sigma, _ = ddim.sample_prev_timestep_indexed(xt, eps, t_dev, z)
        return apply_gsg_batch(wl.seg, mu, sigma, wl.srgan(xt), wl.gt, 60.0)

    graphs = {"ddpm": StepGraph(wl.step_fn, wl.x0.shape, wl.dev), "ddim": StepGraph(ddim_fn, wl.x0.shape, wl.dev)}
    ts = {"ddpm": list(range(wl.T - 1, 0, -1)), "ddim": ddim.timesteps[:-1]}
    z = torch.randn(wl.x0.shape, device=wl.dev, generator=torch.Generator(device=wl.dev).manual_seed(5))
    ms = {"ddpm": [], "ddim": []}
    for r in range(rounds + 1):                     # round 0 is warm-up
        for arm, g in graphs.items():
            g.load(wl.x0)
            seq = [ts[arm][(r * steps + k) % len(ts[arm])] for k in range(steps)]

            def run():
                for i in seq:
                    g.replay(wl.t_all[i:i + 1], z)
            t = events_ms(run) / steps
            if r:
                ms[arm].append(t)
    return ms


def kernel_ms(ddpm_sched, ddim, launches, dev):
    """ms per launch of ddpm_step_kernel<2> and ddim_step_kernel<2> (graph of `launches` launches, HBM-resident buffers)."""
    from weatherconverter_b200._lib import check, lib, ptr, stream_ptr
    shape, sets = (24, 3, 128, 256), 8
    gen = torch.Generator(device=dev).manual_seed(9)
    bufs = [[torch.randn(shape, device=dev, generator=gen) for _ in range(4)] for _ in range(sets)]
    n_per, B = bufs[0][0][0].numel(), shape[0]
    t_dev = torch.tensor([ddim.timesteps[1]], device=dev)
    tabs = {"ddpm": ddpm_sched._tables_on(dev), "ddim": ddim._tables_on(dev)}
    fns = {"ddpm": lib().wc_ddpm_step_indexed, "ddim": lib().wc_ddim_step_indexed}
    graphs = {}
    for arm in ("ddpm", "ddim"):
        def body():
            for k in range(launches):
                x, e, z, o = bufs[k % sets]
                check(fns[arm](ptr(x), ptr(e), ptr(z), ptr(o), None, None, n_per, B, ptr(tabs[arm]), ptr(t_dev),
                               ddim.num_timesteps if arm == "ddim" else ddpm_sched.num_timesteps, stream_ptr()))
        body()                                      # eager warm-up
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            body()
        graphs[arm] = g
    ms = {"ddpm": [], "ddim": []}
    for r in range(6):
        for arm, g in graphs.items():
            t = events_ms(g.replay) / launches
            if r:
                ms[arm].append(t)
    nbytes = 4 * 4 * n_per * B                      # read x, eps, z; write out
    return ms, nbytes, shape


def wall_s(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--which", default="c2,c3")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--out-dir", default="profiles")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from bench import WORKLOADS, GpuWorkload
    from weatherconverter_b200.diffusion_model.sample_ddpm import sample_tensor
    from weatherconverter_b200.translation import sample_with_sgg
    dev = torch.device("cuda")
    torch.backends.cudnn.benchmark = False
    for which in a.which.split(","):
        spec = dict(WORKLOADS[which])
        wl = GpuWorkload(spec, dev, 0)
        B = spec["batch"]
        ddim50 = wl.sched.ddim(50, eta=1.0, num_timesteps=wl.T)
        step = graphed_step_ms(wl, ddim50, a.rounds, a.steps)
        kms, nbytes, kshape = kernel_ms(wl.sched, ddim50, a.launches, dev)
        gen = torch.Generator(device=dev).manual_seed(11)
        runs = {}
        if spec["kind"] == "ddpm":
            shape = tuple(wl.x0.shape)

            def sample(sampler):
                return lambda: sample_tensor(wl.unet, wl.sched, xT=wl.x0, num_timesteps=wl.T, device_noise=True,
                                             generator=gen, use_graph=True, sampler=sampler)
            wall_s(sample(wl.sched.ddim(4, eta=0.0)))       # warm-up: plans bound, modules loaded
            for name, sampler in ((f"ddpm_{wl.T}", None), ("ddim_50", wl.sched.ddim(50)), ("ddim_100", wl.sched.ddim(100)),
                                  ("ddim_250", wl.sched.ddim(250))):
                runs[name] = wall_s(sample(sampler))
        else:
            x_in = torch.rand(wl.x0.shape, generator=torch.Generator().manual_seed(12)).to(dev) * 2 - 1
            t_fwd = torch.full((B,), wl.T - 1, dtype=torch.int64)

            def translate(sampler):
                return lambda: sample_with_sgg(x_in, wl.unet, wl.sched, wl.seg, wl.gt, wl.srgan, n_steps=wl.T, t_forward=t_fwd,
                                               device_noise=True, generator=gen, use_graph=True, sampler=sampler)
            wall_s(translate(wl.sched.ddim(4, eta=1.0, num_timesteps=wl.T)))
            for name, sampler in ((f"ddpm_{wl.T}", None), ("ddim_50_eta1", ddim50)):
                runs[name] = wall_s(translate(sampler))
        med = {k: statistics.median(v) for k, v in step.items()}
        kmed = {k: statistics.median(v) for k, v in kms.items()}
        rec = {
            "metric": f"DDIM vs DDPM ({which}: {spec['desc']})",
            "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev.index or 0),
            "batch": B, "latent": [spec["h"], spec["w"]], "ddpm_steps": wl.T,
            "graphed_step_ms": {"ddpm": med["ddpm"], "ddim_50_eta1": med["ddim"], "ddim_over_ddpm": med["ddim"] / med["ddpm"],
                                "spread_ms": {k: [min(v), max(v)] for k, v in step.items()},
                                "timing": f"{a.rounds} alternated blocks of {a.steps} graph replays per arm, CUDA events, "
                                          "median of the per-block ms/step"},
            "step_kernel": {"ddpm_us": 1e3 * kmed["ddpm"], "ddim_us": 1e3 * kmed["ddim"],
                            "ddim_over_ddpm": kmed["ddim"] / kmed["ddpm"], "shape": list(kshape), "bytes_per_launch": nbytes,
                            "ddpm_gbs": nbytes / kmed["ddpm"] / 1e6, "ddim_gbs": nbytes / kmed["ddim"] / 1e6,
                            "spread_us": {k: [1e3 * min(v), 1e3 * max(v)] for k, v in kms.items()},
                            "timing": f"one CUDA graph of {a.launches} launches per arm over 8 rotating buffer sets (302 MB, "
                                      "beyond L2), 5 alternated replays, CUDA events"},
            "per_batch": {k: {"wall_s": v, "images_per_s": B / v} for k, v in runs.items()},
            "per_batch_timing": "host clock around one whole call ending in a device synchronise; includes the StepGraph "
                                "capture (2 eager warm-up steps + capture) of that call; one call per arm",
        }
        line = json.dumps(rec)
        print(line, flush=True)
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, f"r3_ddim_{which}.json"), "w") as f:
            f.write(line + "\n")
        del wl
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
