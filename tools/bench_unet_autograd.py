"""Cost of the differentiable Unet against the fused training step at the C5 geometry (default config, batch 64, 128x256).

Two models with the same weights: one trained by DenoisingTrainer.step (fused MSE + Adam), one by the reference's step body
on the differentiable Unet (zero_grad, add_noise, model, an MSE lambda, backward, torch.optim.Adam.step).  The two arms
alternate step by step in one process and every step is timed with CUDA events.  Then the backward alone is timed, and its
library launches counted, in full mode (parameters and x need gradients) and in data-only mode (only x does), again
alternated.  Writes one JSON line.  usage: python tools/bench_unet_autograd.py [--steps 20] [--warmup 3] [--out PATH]"""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F


def power_limit_w(index):
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetEnforcedPowerLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=os.path.join("profiles", "unet_autograd_c5.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from oracle.unet import DEFAULT_MODEL_CONFIG
    from oracle.weights import synth_state_dict
    from weatherconverter_b200 import ops
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet, param_spec
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    from weatherconverter_b200.diffusion_model.train_ddpm import DenoisingTrainer

    dev = torch.device("cuda")
    cfg = dict(DEFAULT_MODEL_CONFIG)
    B, H, W = a.batch, 128, 256
    sd = synth_state_dict({k: (v, torch.float32) for k, v in param_spec(cfg).items()}, 3455)
    sched = LinearNoiseScheduler(1000, 1e-4, 0.02)
    model_f, model_g = Unet(cfg).to(dev), Unet(cfg).to(dev)
    model_f.load_state_dict(sd)
    model_g.load_state_dict(sd)
    model_g.differentiable = True
    trainer = DenoisingTrainer(model_f, sched, lr=1e-4, seed=0)
    optimizer = torch.optim.Adam(model_g.parameters(), lr=1e-4)
    criterion = lambda pred, target: F.mse_loss(pred, target)   # noqa: E731
    gen_cpu, gen_dev = torch.Generator().manual_seed(0), torch.Generator(device=dev).manual_seed(0)
    images = (torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(1)) * 2 - 1).to(dev)

    def fused_step():
        return trainer.step(images)

    def generic_step():
        optimizer.zero_grad()
        noise = torch.randn(images.shape, device=dev, generator=gen_dev)
        t = torch.randint(0, sched.num_timesteps, (B,), generator=gen_cpu).to(dev)
        noisy = sched.add_noise(images, noise, t)
        loss = criterion(model_g(noisy, t), noise)
        loss.backward()
        optimizer.step()
        return loss

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1), out

    for _ in range(a.warmup):
        fused_step()
        generic_step()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ms_f, ms_g, loss_f, loss_g = [], [], None, None
    for _ in range(a.steps):
        m, loss_f = timed(fused_step)
        ms_f.append(m)
        m, loss_g = timed(generic_step)
        ms_g.append(m)
    peak = torch.cuda.max_memory_allocated()

    # backward alone: full (parameters + x) and data-only (x); the forward is outside the timed window
    x = sched.add_noise(images, torch.randn(images.shape, device=dev, generator=gen_dev),
                        torch.randint(0, 1000, (B,), generator=gen_cpu).to(dev))
    t = torch.randint(0, 1000, (B,), generator=gen_cpu).to(dev)
    w = torch.randn(images.shape, device=dev, generator=gen_dev)

    def backward(full):
        model_g.requires_grad_(full)
        model_g.zero_grad(set_to_none=True)
        xr = x.clone().requires_grad_()
        loss = (model_g(xr, t) * w).mean()
        torch.cuda.synchronize()
        n0 = ops.launch_count()
        ms, _ = timed(loss.backward)
        return ms, ops.launch_count() - n0

    bwd = {True: [], False: []}
    launches = {}
    for _ in range(a.warmup):
        backward(True)
        backward(False)
    for _ in range(max(10, a.steps // 2)):
        for full in (True, False):
            ms, n = backward(full)
            bwd[full].append(ms)
            launches[full] = n
    model_g.requires_grad_(True)

    med_f, med_g = statistics.median(ms_f), statistics.median(ms_g)
    bf, bd = statistics.median(bwd[True]), statistics.median(bwd[False])
    rec = {
        "metric": "differentiable Unet vs fused training step (C5: default config, batch %d, 128x256)" % B,
        "device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(dev.index or 0),
        "steps": a.steps, "warmup": a.warmup, "timing": "CUDA events per step, arms alternated step by step",
        "fused_ms_per_step": med_f, "generic_ms_per_step": med_g, "generic_over_fused": med_g / med_f,
        "fused_ms_all": ms_f, "generic_ms_all": ms_g,
        "backward_full_ms": bf, "backward_data_only_ms": bd, "data_only_saving": 1.0 - bd / bf,
        "backward_full_launches": launches[True], "backward_data_only_launches": launches[False],
        "peak_hbm_gib": peak / 2 ** 30,
        "peak_hbm_note": "torch allocator peak over the timed steps, both arms resident (two 128x256 batch-64 training plans)",
        "final_loss_fused": loss_f.item(), "final_loss_generic": loss_g.item(),
    }
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
