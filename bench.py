#!/usr/bin/env python
"""bench.py — headline benchmark of the WeatherConverter hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c3|c2|c1|c5|ref] [--graph 0|1]
                    [--dump-outputs DIR]

Default workload (every N, weak scaling) = the configuration BASELINE.json's metric is quoted on:
  c3  SGG-guided translation at 256x512 (BASELINE.json configs[2]/[3]), batch 32 per GPU, N = 500 reverse steps,
      geometry A of SURVEY.md 8d (reference-faithful): latent 64x128 (UNet config.yaml with im_size 64) -> SRGAN x4 ->
      DeepLabV3+-ResNet-50 (os16, 19 classes) forward + CE + input gradient at 256x512 -> avg-pool 4 -> guidance
      update (lambda = 60), GSG on every step (the repaired driver of SURVEY.md 8c).
  c2  UNet DDPM sampling at 128x256, batch 16 per GPU, 1000-step schedule (BASELINE.json configs[1]).
  c5  denoising-loss TRAINING step at 128x256, batch 64 per GPU, NCCL gradient all-reduce at N > 1 (BASELINE.json
      configs[4]; metric = trained images/s; step = add_noise + forward + MSE + backward + all-reduce + Adam).
  ref the reference's OWN driver geometry (translation.py:100-146): batch 1, latent 128x128 (im_size 128), SRGAN x4,
      DeepLabV3+-ResNet-101 at 512x512, 500 steps - the launch-bound regime (one image, ~700 launches per step).
By default every step of the b200 arm is ONE cudaGraphLaunch of the captured reverse step (weatherconverter_b200/graphs.py; the
public drivers' use_graph=True path); `eager` in the line is the same loop launched kernel by kernel.
A "step" is ONE reverse-diffusion step over the batch; per-step cost does not depend on t, so
    images/s = (N_gpus * batch) / (schedule_steps * seconds_per_step).
`value` times the steps with inputs resident in HBM; `e2e` times the same steps through the public Python API with
the per-step noise coming from pinned HOST memory (the reference draws z on the CPU every step,
linear_noise_scheduler.py:110) and x_{t-1} read back to the host, copies inside the timed region.
`--impl reference` times the reference algorithm's CPU implementation (the oracle port — the reference is a Python
source tree that cannot travel to the GPU box) on all host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "guided translation images/sec (256x512, T steps) at 1/2/4/8 B200 vs host CPU"
UNIT = "images/s"

WORKLOADS = {
    "c3": dict(kind="sgg", im_size=64, batch=32, h=64, w=128, T=500,
               desc="C3/C4: SGG-guided translation 256x512 (latent 64x128, SRGAN x4, DeepLabV3+-R50 gradient guidance every "
                    "step, lambda 60), batch 32/GPU, 500 reverse steps (BASELINE.json configs[2]/[3], geometry A)"),
    "c2": dict(kind="ddpm", im_size=128, batch=16, h=128, w=256, T=1000,
               desc="C2: UNet DDPM sampling 128x256, batch 16/GPU, 1000-step schedule (BASELINE.json configs[1])"),
    "c5": dict(kind="train", im_size=128, batch=64, h=128, w=256, T=1000,
               desc="C5: denoising-loss training step 128x256, batch 64/GPU, Adam, NCCL gradient all-reduce across GPUs "
                    "(BASELINE.json configs[4])"),
    "c1": dict(kind="ddpm", im_size=64, batch=4, h=64, w=64, T=50,
               desc="C1: UNet DDPM sampling 64x64, batch 4, 50 steps (BASELINE.json configs[0])"),
    "ref": dict(kind="sgg", im_size=128, batch=1, h=128, w=128, T=500, backbone="resnet101",
                desc="reference driver geometry (translation.py:100-146): batch 1, latent 128x128 (im_size 128), SRGAN x4, "
                     "DeepLabV3+-ResNet-101 gradient guidance at 512x512 every step, lambda 60, 500 reverse steps"),
}


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d.get("hbm_gbs", 6650.0), tf_burst=d.get("bf16_tflops", 1590.0),
                    tf_sustained=d.get("bf16_tflops_sustained", 1400.0), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU via NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.05)

    def finish(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes each array as <out_dir>/<name>.npy in float32.  An array over its share of DUMP_BYTES is written
    as a fixed sample of its flattened elements (indices drawn with seed 0, ascending), so that two builds run with the same
    arguments can be compared value for value."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // 4 // len(arrays)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > cap:
            idx = torch.randint(0, t.numel(), (cap,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def block_labels(gen, B, H, W, blk=8):
    """Cityscapes-shaped synthetic masks: 8x8 blocks of uniform class in 0..18, 5 % of the blocks = 255 (SURVEY 8d)."""
    import torch
    lab = torch.randint(0, 19, (B, H // blk, W // blk), generator=gen)
    lab[torch.rand(B, H // blk, W // blk, generator=gen) < 0.05] = 255
    return lab.repeat_interleave(blk, 1).repeat_interleave(blk, 2)


# ------------------------------------------------------------------------------------------------ GPU workloads
class GpuWorkload:
    def __init__(self, spec, dev, rank):
        import torch
        from weatherconverter_b200.diffusion_model.config.models import ModelConfig
        from weatherconverter_b200.diffusion_model.models.unet_base import Unet
        from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
        from weatherconverter_b200.sharding import initial_noise
        self.spec, self.dev = spec, dev
        B, h, w = spec["batch"], spec["h"], spec["w"]
        torch.manual_seed(3455)   # diffusion config.yaml:32
        self.unet = Unet(ModelConfig(im_size=spec["im_size"])).to(dev).eval()
        self.sched = LinearNoiseScheduler(spec["T"] if spec["kind"] == "ddpm" else 1000, 1e-4, 0.02)
        self.x0 = initial_noise((3, h, w), rank * B, (rank + 1) * B).to(dev)   # RNG keyed by the global image index
        self.eps = torch.empty_like(self.x0)
        self.T = spec["T"]
        if spec["kind"] == "sgg":
            from weatherconverter_b200.seg_model.network import modeling
            from weatherconverter_b200.srgan_model.models import Generator
            torch.manual_seed(42)   # seg config.yaml:3
            self.backbone = spec.get("backbone", "resnet50")
            self.seg = getattr(modeling, "deeplabv3plus_" + self.backbone)(num_classes=19, output_stride=16, pretrained_backbone=False)
            g = torch.Generator().manual_seed(7)
            for n, b in self.seg.named_buffers():   # non-degenerate eval BatchNorm statistics (SURVEY 8c)
                if n.endswith("running_mean"):
                    b.copy_(0.1 * torch.randn(b.shape, generator=g))
                elif n.endswith("running_var"):
                    b.copy_(0.5 + torch.rand(b.shape, generator=g))
            self.seg = self.seg.to(dev).eval()
            torch.manual_seed(0)
            self.srgan = Generator(upscale_factor=4)
            for n, b in self.srgan.named_buffers():
                if n.endswith("running_mean"):
                    b.copy_(0.1 * torch.randn(b.shape, generator=g))
                elif n.endswith("running_var"):
                    b.copy_(0.5 + torch.rand(b.shape, generator=g))
            self.srgan = self.srgan.to(dev).eval()
            self.gt = block_labels(torch.Generator().manual_seed(1234 + rank), B, 4 * h, 4 * w).to(dev)
        self.t_dev = {}
        self.t_all = torch.arange(1000, device=dev, dtype=torch.int64)
        self.sg = None
        self.launches_per_step = None

    def step_fn(self, xt, t_dev, z):
        """The reverse step in its CUDA-graph-capturable form: the timestep is read from device memory (what
        sample_with_sgg / sample_tensor capture with use_graph=True)."""
        eps = self.unet(xt, t_dev)
        if self.spec["kind"] == "ddpm":
            return self.sched.step_indexed(xt, eps, t_dev, z)
        from weatherconverter_b200.sgg.sgg import apply_gsg_batch
        mu, sigma, _ = self.sched.sample_prev_timestep_indexed(xt, eps, t_dev, z)
        return apply_gsg_batch(self.seg, mu, sigma, self.srgan(xt), self.gt, 60.0)

    def capture(self):
        from weatherconverter_b200 import ops
        from weatherconverter_b200.graphs import StepGraph
        self.sg = StepGraph(self.step_fn, self.x0.shape, self.dev, warmup=2)
        before = ops.launch_count()     # kernels of ONE eager step == nodes of the captured graph
        self.step_fn(self.sg.xt, self.sg.t, self.sg.z)
        self.launches_per_step = ops.launch_count() - before

    def timestep(self, k):
        return self.T - 1 - (k % (self.T - 1))

    def graph_step(self, k, z):
        """One cudaGraphLaunch: x_t <- reverse step at timestep(k), in place on the graph's static buffer."""
        i = self.timestep(k)
        return self.sg.replay(self.t_all[i:i + 1], z)

    def t_tensor(self, i):
        import torch
        if i not in self.t_dev:
            self.t_dev[i] = torch.tensor([i], device=self.dev)
        return self.t_dev[i]

    def step(self, xt, k, z):
        """One reverse step at timestep i = T-1-(k mod (T-1)) (never 0: the timed steps all inject noise)."""
        i = self.T - 1 - (k % (self.T - 1))
        self.unet(xt, self.t_tensor(i), out=self.eps)
        if self.spec["kind"] == "ddpm":
            return self.sched.step(xt, self.eps, i, z=z)
        from weatherconverter_b200.sgg.sgg import apply_gsg_batch
        mu, sigma, _ = self.sched.sample_prev_timestep(xt, self.eps, i, z=z)
        sr = self.srgan(xt)
        return apply_gsg_batch(self.seg, mu, sigma, sr, self.gt, 60.0)

    def flops_per_step(self):
        f = self.unet.flops_per_forward()
        parts = {"unet": f}
        if self.spec["kind"] == "sgg":
            sf, sb = self.seg.flops()
            parts.update(srgan=self.srgan.flops(), seg_fwd=sf, seg_dgrad=sb)
        return sum(parts.values()), parts


# ------------------------------------------------------------------------------------------------ CPU reference
def cpu_reference_rate(spec, steps, warmup, batch=1, shared=None):
    """Oracle port (plain PyTorch fp32, all host threads) on a bounded sample: `batch` images, `steps` timed reverse steps.
    Returns (images/s extrapolated linearly to the schedule, seconds/step/image, cores, first_step) where first_step =
    (x_{t-1}, mu + sigma z) of the very first step (used for the parity key).  `shared` = dict(unet=, seg=, srgan= state
    dicts, xt=, gt=, z=, i=) makes the oracle run on the GPU arm's own weights and inputs."""
    import torch
    from oracle import deeplab, sgg, srgan
    from oracle.scheduler import OracleScheduler
    from oracle.unet import DEFAULT_MODEL_CONFIG, unet_forward, unet_param_spec
    from oracle.weights import synth_state_dict
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = spec["im_size"]
    T, h, w = spec["T"], spec["h"], spec["w"]
    backbone = spec.get("backbone", "resnet50")
    sched = OracleScheduler(T if spec["kind"] == "ddpm" else 1000, 1e-4, 0.02)
    g = torch.Generator().manual_seed(1234)
    if shared is not None:
        sd, xt = shared["unet"], shared["xt"].clone()
        batch = xt.shape[0]
        if spec["kind"] == "sgg":
            seg_sd, gan_sd, gt = shared["seg"], shared["srgan"], shared["gt"]
    else:
        sd = synth_state_dict(unet_param_spec(cfg), 3455)
        xt = torch.randn(batch, 3, h, w, generator=g)
        if spec["kind"] == "sgg":
            seg_sd = synth_state_dict(deeplab.deeplab_param_spec(backbone), 42)
            gan_sd = synth_state_dict(srgan.srgan_param_spec(), 0)
            gt = block_labels(g, batch, 4 * h, 4 * w)
    times, first = [], None
    with torch.no_grad():
        for k in range(warmup + steps):
            i = shared["i"] if (shared is not None and k == 0) else T - 1 - k
            t0 = time.perf_counter()
            eps = unet_forward(sd, cfg, xt, torch.tensor([i]))
            z = shared["z"] if (shared is not None and k == 0) else torch.randn(xt.shape, generator=g)
            mean, sz, _ = sched.sample_prev_timestep(xt, eps, i, z=z)
            if spec["kind"] == "sgg":
                sr = srgan.generator_forward(gan_sd, xt)
                with torch.enable_grad():
                    xt, _, _ = sgg.apply_gsg(seg_sd, mean, sz, sr, gt, 60.0, backbone)
            else:
                xt = mean + sz
            dt = time.perf_counter() - t0
            if first is None:
                first = (xt.clone(), mean + sz)
            if k >= warmup:
                times.append(dt)
    sec = sum(times) / len(times) / batch
    return 1.0 / (T * sec), sec, cores, first


TRAIN_METRIC = "denoising-loss training images/sec (128x256, batch 64/GPU, Adam, NCCL gradient all-reduce)"


def cpu_train_rate(spec, steps, warmup):
    """Oracle port of the training step (PyTorch fp32 autograd + Adam, all host threads) on ONE image."""
    import torch
    from oracle.scheduler import OracleScheduler
    from oracle.train import train_step
    from oracle.unet import DEFAULT_MODEL_CONFIG, unet_param_spec
    from oracle.weights import synth_state_dict
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = spec["im_size"]
    sd = synth_state_dict(unet_param_spec(cfg), 3455)
    sched = OracleScheduler(1000, 1e-4, 0.02)
    g = torch.Generator().manual_seed(1234)
    x = torch.rand(1, 3, spec["h"], spec["w"], generator=g) * 2 - 1
    times = []
    for k in range(warmup + steps):
        noise = torch.randn(x.shape, generator=g)
        t = torch.randint(0, 1000, (1,), generator=g)
        t0 = time.perf_counter()
        _, _, sd = train_step(sd, cfg, x, noise, t, sched, step=k + 1)
        dt = time.perf_counter() - t0
        if k >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return 1.0 / sec, sec, cores


def run_train(args):
    """C5: training step.  value = images trained per second over all ranks (inputs resident in HBM); e2e = the same
    step with the image batch coming from pinned host memory and the loss read back every step."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from weatherconverter_b200 import _lib, ops
    from weatherconverter_b200.diffusion_model.config.models import ModelConfig
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    from weatherconverter_b200.diffusion_model.train_ddpm import DenoisingTrainer
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # rank 0 prints ONE JSON line on stdout: NCCL's banner / debug output (NCCL_DEBUG from the environment or from
        # /etc/nccl.conf) goes to stderr instead
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    spec = dict(WORKLOADS["c5"])
    if args.batch:
        spec["batch"] = args.batch
    B, h, w = spec["batch"], spec["h"], spec["w"]
    W_, K = max(args.warmup, 3), args.steps
    peaks = read_peaks()
    torch.manual_seed(3455)                       # same initial replica on every rank (config.yaml:32)
    model = Unet(ModelConfig(im_size=spec["im_size"])).to(dev)
    sched = LinearNoiseScheduler(1000, 1e-4, 0.02)
    trainer = DenoisingTrainer(model, sched, lr=1e-4)
    g = torch.Generator().manual_seed(1234 + rank)   # every rank trains on its own shard of the global batch
    imgs_host = [(torch.rand(B, 3, h, w, generator=g) * 2 - 1).pin_memory() for _ in range(2)]
    imgs = [x.to(dev) for x in imgs_host]
    ts = [torch.randint(0, 1000, (B,), generator=g) for _ in range(4)]
    gz = torch.Generator(device=dev).manual_seed(99 + rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one(k, x):
        noise = torch.randn(x.shape, device=dev, generator=gz)
        return trainer.step(x, noise=noise, t=ts[k % 4])

    for k in range(W_):
        one(k, imgs[k % 2])
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(W_, W_ + K):
        loss = one(k, imgs[k % 2])
    e1.record()
    barrier()
    clocks = sampler.finish()
    launches = ops.launch_count() - l0
    ms_total = e0.elapsed_time(e1)
    loss_val = float(loss)
    if args.dump_outputs and rank == 0:   # the last timed step's loss and the weights it left, before the e2e leg moves them
        dump_outputs(args.dump_outputs, {"loss": loss, "params": trainer.flat_params[:trainer.used]})
    # e2e: batch from pinned host memory, loss read back each step (as the reference's loss.item(), train_ddpm.py:116)
    x_dev = torch.empty_like(imgs[0])
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for k in range(K):
        x_dev.copy_(imgs_host[k % 2], non_blocking=True)
        loss_val = float(one(k, x_dev))
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    classes, roofline = {}, None
    flops_step = trainer.flops_per_step
    if not args.no_profile and not args.resident_only:
        lib = _lib.lib()
        KP = 1
        lib.wc_profile_begin()
        one(0, imgs[0])
        ms_c, cnt_c, work_c = (C.c_double * 8)(), (C.c_longlong * 8)(), (C.c_double * 8)()
        _lib.check(lib.wc_profile_end(ms_c, cnt_c, work_c))
        names = ["igemm_wgrad_tcgen05", "flash_attention_fwd_bwd_tcgen05", "groupnorm_fwd_bwd", "boundary_conv", "elementwise_adam_mse", "other"]
        for i, n in enumerate(names):
            if cnt_c[i]:
                classes[n] = {"ms_per_step": ms_c[i] / KP, "launches_per_step": cnt_c[i] / KP, "work_per_step": work_c[i] / KP}
        prof_total = sum(v["ms_per_step"] for v in classes.values())
        for n, v in classes.items():
            if "tcgen05" in n:
                v["tflops"] = v["work_per_step"] / (v["ms_per_step"] * 1e-3) / 1e12
            elif v["work_per_step"] > 0:
                v["gbs"] = v["work_per_step"] / (v["ms_per_step"] * 1e-3) / 1e9
            v["share_of_step"] = v["ms_per_step"] / prof_total
        dom = max(("igemm_wgrad_tcgen05", "flash_attention_fwd_bwd_tcgen05"), key=lambda n: classes.get(n, {}).get("ms_per_step", 0))
        achieved = classes[dom]["tflops"]
        roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                    "frac": achieved / peaks["tf_sustained"], "traffic": None,
                    "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                    "share_of_step": classes[dom]["share_of_step"],
                    "flops_per_launch": classes[dom]["work_per_step"] / classes[dom]["launches_per_step"],
                    "avg_launch_ms": classes[dom]["ms_per_step"] / classes[dom]["launches_per_step"],
                    "launches_per_step": classes[dom]["launches_per_step"]}
    if world > 1:
        tt = torch.tensor([ms_total, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = float(tt[0]), float(tt[1])
    ms_step = ms_total / K
    value = world * B / (ms_step * 1e-3)
    e2e_value = world * B / (ms_e2e / K * 1e-3)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, sec, cores = cpu_train_rate(spec, 1, 1)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sec_per_step_per_image": sec,
                        "sample": f"oracle port (PyTorch fp32 autograd + Adam, {cores} threads): batch of 1 image, 1 timed step after 1 warm-up"}
    if rank == 0:
        line = {
            "metric": TRAIN_METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W_,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": spec["desc"], "batch_per_gpu": B, "image": [h, w],
                       "step": "add_noise + UNet forward + MSE + full backward (data + weight gradients) + bucketed NCCL all-reduce + fused Adam",
                       "l2": "per-step working set (tens of GB of saved activations) exceeds the 126 MB L2; no explicit flush",
                       "weights": "random init (seed 3455), fp32 master weights, bf16 activations / GEMM operands, fp32 accumulation"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * 3 * h * w * 4, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / K},
            "gpu_launches": int(launches), "launches_per_step": launches / K, "clocks": clocks, "roofline": roofline,
            "kernel_classes": classes, "step_gflop_per_image": flops_step / B / 1e9,
            "step_tflops": flops_step / (ms_step * 1e-3) / 1e12,
            "step_frac_of_tensor_peak": flops_step / (ms_step * 1e-3) / 1e12 / peaks["tf_sustained"],
            "cpu_baseline": cpu_baseline, "final_loss": loss_val, "finite": loss_val == loss_val,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    """Reference arm: rank 0 only; CPU implementation of the same step on a bounded sample."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    spec = WORKLOADS[args.workload]
    if spec["kind"] == "train":
        steps, warm = min(args.steps, 2), 1
        value, sec, cores = cpu_train_rate(spec, steps, warm)
        sample = (f"oracle port (PyTorch fp32 autograd + Adam, {cores} threads): batch of 1 image, {steps} timed training steps "
                  f"after {warm} warm-up")
        print(json.dumps({
            "impl": "reference", "metric": TRAIN_METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": spec["desc"], "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)
        return
    # --steps / --warmup are honoured up to a cap that keeps the run within a few minutes on the host cores (one reverse step
    # of one image costs 0.8 - 3 s there); the sample is a batch of 2 images (per-image guidance = per-image loop, as the
    # reference's B = 1 contract demands), throughput extrapolated linearly to the schedule (per-step cost is t-independent)
    cap_steps, cap_warm, nb = (10, 3, 2) if args.workload != "ref" else (4, 1, 1)
    steps, warm = max(1, min(args.steps, cap_steps)), max(0, min(args.warmup, cap_warm))
    nb = min(nb, spec["batch"])
    value, sec, cores, _ = cpu_reference_rate(spec, steps, warm, batch=nb)
    sample = (f"oracle port (PyTorch fp32, {cores} threads): batch of {nb} image(s), {steps} timed reverse steps after {warm} "
              f"warm-up (--steps {args.steps} / --warmup {args.warmup} honoured up to the caps {cap_steps} / {cap_warm}), "
              f"extrapolated linearly to {spec['T']} steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": sec * nb * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": spec["desc"], "batch_per_gpu": spec["batch"], "latent": [spec["h"], spec["w"]],
                   "schedule_steps": spec["T"], "sample": sample, "sample_batch": nb},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _dram_traffic_per_launch(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per igemm launch (bytes), averaged over the launches of one step, from the
    NEWEST committed ncu launch list of the same command (profiles/r<round>_dram_traffic_<workload>.json, made by
    tools/launch_traffic.py); returns (bytes or None, source file or None).  DRAM counters need ncu, so this cannot be measured
    inside the timed run; the file name (round / build tag) is reported next to the number so a stale capture is visible."""
    import glob
    import re
    pdir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles")
    best = None
    for path in glob.glob(os.path.join(pdir, f"r*_dram_traffic_{workload}.json")):
        m = re.match(r"r(\d+)_", os.path.basename(path))
        if m and (best is None or int(m.group(1)) > best[0]):
            best = (int(m.group(1)), path)
    if best is None:
        return None, None
    try:
        with open(best[1]) as f:
            return float(json.load(f)["dram_bytes_per_launch"]), os.path.basename(best[1])
    except (OSError, KeyError, ValueError):
        return None, None


# exponentials per clock per SM with the MUFU pipe (16 / clk / SM) and the FMA-pipe polynomial (15.3 / clk / SM) both saturated,
# each measured alone on this pool's B200 (tools/micro/pipe_rate.cu, profiles/r2_pipe_rate.txt)
EXP_PER_CLK_PER_SM = 31.3


def class_floors(records, peaks, sm_mhz, sms=148):
    """Per kernel class: which resource bounds it and the time that resource alone would take (`floor_ms`), summed over the
    launches of the profiling window, next to the measured time.  records: (cls, ms, work, info[6]) per launch.
      igemm      max(FLOPs / sustained bf16 peak, algorithmic bytes / HBM peak) per launch; bytes = activations in (M x Cin) +
                 packed weights (N x K) + outputs (M x N), 2 B each
      attention  max(FLOPs / peak, N^2 exponentials per head / (EXP_PER_CLK_PER_SM x SMs x SM clock))
      GroupNorm, boundary convs, scheduler: algorithmic bytes / HBM peak"""
    names = ["igemm_tcgen05", "flash_attention_tcgen05", "groupnorm_silu", "boundary_conv", "scheduler", "other"]
    tf, hbm = peaks["tf_sustained"] * 1e12, peaks["hbm"] * 1e9
    exp_rate = EXP_PER_CLK_PER_SM * sms * (sm_mhz or 1965.0) * 1e6
    out = {}
    for cls, ms, work, info in records:
        n = names[cls] if cls < len(names) else "other"
        d = out.setdefault(n, {"measured_ms": 0.0, "floor_ms": 0.0, "tensor_ms": 0.0, "hbm_ms": 0.0, "exp_ms": 0.0, "launches": 0})
        d["measured_ms"] += ms
        d["launches"] += 1
        if cls == 0:
            M, N, K, taps = info[0], info[1], info[2], max(1, info[4] % 100)   # info[4] also carries epilogue flags in its thousands
            t_t, t_h = work / tf * 1e3, 2.0 * (M * (K / taps) + N * K + M * N) / hbm * 1e3
            d["tensor_ms"] += t_t; d["hbm_ms"] += t_h; d["floor_ms"] += max(t_t, t_h)
        elif cls == 1:
            BH, ntok = info[0], info[1]
            t_t, t_e = work / tf * 1e3, float(BH) * ntok * ntok / exp_rate * 1e3
            d["tensor_ms"] += t_t; d["exp_ms"] += t_e; d["floor_ms"] += max(t_t, t_e)
        elif work > 0:
            t_h = work / hbm * 1e3
            d["hbm_ms"] += t_h; d["floor_ms"] += t_h
    for n, d in out.items():
        parts = {"tensor": d.pop("tensor_ms"), "hbm": d.pop("hbm_ms"), "exp": d.pop("exp_ms")}
        d["bound"] = max(parts, key=parts.get) if d["floor_ms"] > 0 else None
        d["floor_parts_ms"] = {k: v for k, v in parts.items() if v > 0}
        d["frac"] = d["floor_ms"] / d["measured_ms"] if d["measured_ms"] > 0 and d["floor_ms"] > 0 else None
    return out


def secondary_training(dev, rank, world, peaks, steps=3, warmup=3, batch=64):
    """Short C5 run (training step with the NCCL gradient all-reduce) appended to the N > 1 line, so the one collective of the
    hot path has a record in the scaling run: images/s over all ranks, all-reduce bytes per step, and how much of the
    stand-alone all-reduce time the overlap with the backward plan hides."""
    import torch
    import torch.distributed as dist
    from weatherconverter_b200.diffusion_model.config.models import ModelConfig
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    from weatherconverter_b200.diffusion_model.train_ddpm import DenoisingTrainer
    spec = WORKLOADS["c5"]
    h, w = spec["h"], spec["w"]
    torch.manual_seed(3455)
    model = Unet(ModelConfig(im_size=spec["im_size"])).to(dev)
    trainer = DenoisingTrainer(model, LinearNoiseScheduler(1000, 1e-4, 0.02), lr=1e-4)
    g = torch.Generator().manual_seed(1234 + rank)
    imgs = (torch.rand(batch, 3, h, w, generator=g) * 2 - 1).to(dev)
    ts = [torch.randint(0, 1000, (batch,), generator=g) for _ in range(4)]
    gz = torch.Generator(device=dev).manual_seed(99 + rank)

    def timed(n):
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(n):
            loss = trainer.step(imgs, noise=torch.randn(imgs.shape, device=dev, generator=gz), t=ts[k % 4])
        e1.record()
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n, float(loss)

    timed(warmup)
    ms_full, loss = timed(steps)
    # stand-alone all-reduce of the flat gradient buffer, and the step without any communication
    torch.cuda.synchronize(); dist.barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(3):
        dist.all_reduce(trainer.flat_grads[:trainer.used])
    a1.record()
    torch.cuda.synchronize()
    ms_ar = a0.elapsed_time(a1) / 3
    real_world, trainer.world = trainer.world, 1
    ms_nocomm, _ = timed(steps)
    trainer.world = real_world
    tt = torch.tensor([ms_full, ms_ar, ms_nocomm], device=dev, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_full, ms_ar, ms_nocomm = (float(v) for v in tt)
    exposed = max(0.0, ms_full - ms_nocomm)
    return {"workload": spec["desc"], "metric": TRAIN_METRIC, "value": world * batch / (ms_full * 1e-3), "unit": UNIT,
            "steps": steps, "warmup": warmup, "ms_per_step": ms_full, "ms_per_step_without_allreduce": ms_nocomm,
            "allreduce_bytes_per_step": int(trainer.used) * 4, "allreduce_alone_ms": ms_ar,
            "allreduce_alone_busbw_gbs": 2.0 * (world - 1) / world * trainer.used * 4 / (ms_ar * 1e-3) / 1e9,
            "allreduce_exposed_ms": exposed,
            "allreduce_hidden_frac": min(1.0, max(0.0, 1.0 - exposed / ms_ar)) if ms_ar > 0 else None,
            "buckets": len(trainer._buckets), "step_tflops_per_gpu": trainer.flops_per_step / (ms_full * 1e-3) / 1e12,
            "final_loss": loss, "finite": loss == loss}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch (C4: 128 / 64 / 32 at 2 / 4 / 8 GPUs)")
    ap.add_argument("--graph", type=int, default=1, help="1: one cudaGraphLaunch per step (default); 0: eager launches only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short C5 (NCCL) record at N > 1")
    ap.add_argument("--resident-only", action="store_true", help="eager resident leg only (ncu launch lists)")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last timed step as "
                    "DIR/<name>.npy (float32, 64 MB at most; rank 0's shard at N > 1): x_prev, or loss and params for c5")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU arm's outputs")
    if args.impl == "reference":
        return run_reference(args)
    if WORKLOADS[args.workload]["kind"] == "train":
        return run_train(args)

    import ctypes as C
    import torch
    import torch.distributed as dist
    from weatherconverter_b200 import _lib, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # rank 0 prints ONE JSON line on stdout: NCCL's banner / communicator lines go to stderr and stay visible there
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        dist.init_process_group("nccl", device_id=dev)
    W_ = max(args.warmup, 3)
    K = args.steps
    spec = dict(WORKLOADS[args.workload])
    if args.batch:
        spec["batch"] = args.batch
    B, T = spec["batch"], spec["T"]
    peaks = read_peaks()
    wl = GpuWorkload(spec, dev, rank)
    x0 = wl.x0
    gz = torch.Generator(device=dev).manual_seed(99 + rank)
    use_graph = bool(args.graph) and not args.resident_only

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(W_, W_ + n):
            fn(k)
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    zs = [torch.randn(x0.shape, device=dev, generator=gz) for _ in range(4)]
    z_host = [torch.randn(x0.shape).pin_memory() for _ in range(4)]
    x_host = torch.empty(x0.shape).pin_memory()
    bytes_io = x0.numel() * 4

    # ---------------- eager loop (kernel-by-kernel launches): warm-up, then K timed steps ----------------
    state = {"xt": x0.clone()}

    def eager_step(k):
        state["xt"] = wl.step(state["xt"], k, zs[k % 4])

    for k in range(W_):
        eager_step(k)
    l0 = ops.launch_count()
    ms_eager = timed(eager_step, K)
    eager_launches = ops.launch_count() - l0
    finite = bool(torch.isfinite(state["xt"]).all())

    # ---------------- graph loop: ONE cudaGraphLaunch per step, z resident in HBM (`value`) ----------------
    clocks = None
    if use_graph:
        wl.capture()
        wl.sg.load(x0)
        for k in range(W_):
            wl.graph_step(k, zs[k % 4])
        # warm the end-to-end path too (pinned buffers, copy engines) BEFORE either timed leg, so that the two legs are ordered
        # by the work they do and not by which ran first
        for k in range(W_):
            wl.graph_step(k, z_host[k % 4])
            x_host.copy_(wl.sg.xt, non_blocking=True)
        sampler = ClockSampler(local_rank)
        sampler.start()
        ms_total = timed(lambda k: wl.graph_step(k, zs[k % 4]), K)
        clocks = sampler.finish()
        if args.dump_outputs and rank == 0:   # x_{t-1} of the last timed step, before the e2e leg steps on from it
            dump_outputs(args.dump_outputs, {"x_prev": wl.sg.xt})
        finite = finite and bool(torch.isfinite(wl.sg.xt).all())
        launches = wl.launches_per_step * K
        # ---------------- end-to-end leg: z from pinned host memory, x_{t-1} read back each step ----------------

        def e2e_step(k):
            wl.graph_step(k, z_host[k % 4])                 # H2D copy of this step's noise into the graph's static buffer
            x_host.copy_(wl.sg.xt, non_blocking=True)       # D2H read-back of x_{t-1}
        ms_e2e = timed(e2e_step, K)
    else:
        sampler = ClockSampler(local_rank)
        sampler.start()
        ms_total = timed(eager_step, K)
        clocks = sampler.finish()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"x_prev": state["xt"]})
        launches = eager_launches
        z_dev = torch.empty_like(x0)

        def e2e_step(k):
            z_dev.copy_(z_host[k % 4], non_blocking=True)
            state["xt"] = wl.step(state["xt"], k, z_dev)
            x_host.copy_(state["xt"], non_blocking=True)
        if args.resident_only:
            ms_e2e = ms_total
        else:
            for k in range(W_):
                e2e_step(k)
            ms_e2e = timed(e2e_step, K)
    if args.resident_only:
        args.no_profile = True

    # ---------------- per-kernel-class timing (CUDA events around every launch, eager), roofline per class
    classes, roofline, by_class = {}, None, {}
    flops_step, flop_parts = wl.flops_per_step()
    if not args.no_profile:
        lib = _lib.lib()
        KP = min(K, 3)
        lib.wc_profile_begin()
        xt = x0.clone()
        for k in range(KP):
            xt = wl.step(xt, k, zs[k % 4])
        cap = 4096 * KP
        c_cls, c_ms, c_work, c_info = (C.c_int * cap)(), (C.c_double * cap)(), (C.c_double * cap)(), (C.c_int * (6 * cap))()
        nrec = min(cap, lib.wc_profile_detail(cap, c_cls, c_ms, c_work, c_info))
        records = [(c_cls[i], c_ms[i], c_work[i], [c_info[6 * i + j] for j in range(6)]) for i in range(nrec)]
        ms_c, cnt_c, work_c = (C.c_double * 8)(), (C.c_longlong * 8)(), (C.c_double * 8)()
        _lib.check(lib.wc_profile_end(ms_c, cnt_c, work_c))
        names = ["igemm_tcgen05", "flash_attention_tcgen05", "groupnorm_silu", "boundary_conv", "scheduler", "other"]
        for i, n in enumerate(names):
            if cnt_c[i]:
                classes[n] = {"ms_per_step": ms_c[i] / KP, "launches_per_step": cnt_c[i] / KP, "work_per_step": work_c[i] / KP}
        prof_total = sum(v["ms_per_step"] for v in classes.values())
        for n, v in classes.items():
            if n in ("igemm_tcgen05", "flash_attention_tcgen05"):
                v["tflops"] = v["work_per_step"] / (v["ms_per_step"] * 1e-3) / 1e12
            elif v["work_per_step"] > 0:
                v["gbs"] = v["work_per_step"] / (v["ms_per_step"] * 1e-3) / 1e9
            v["share_of_step"] = v["ms_per_step"] / prof_total
        by_class = class_floors(records, peaks, (clocks or {}).get("sm_mhz"))
        for d in by_class.values():
            d["measured_ms"] /= KP; d["floor_ms"] /= KP; d["launches"] /= KP
            d["floor_parts_ms"] = {k: v / KP for k, v in d["floor_parts_ms"].items()}
        dom = "igemm_tcgen05"
        achieved = classes[dom]["tflops"]
        traffic, traffic_src = _dram_traffic_per_launch(args.workload)
        roofline = {"bound": "tensor", "kernel": "igemm_kernel (csrc/igemm.cu)", "achieved": achieved,
                    "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": achieved / peaks["tf_sustained"],
                    "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                    "share_of_step": classes[dom]["share_of_step"],
                    "flops_per_launch": classes[dom]["work_per_step"] / classes[dom]["launches_per_step"],
                    "avg_launch_ms": classes[dom]["ms_per_step"] / classes[dom]["launches_per_step"],
                    "launches_per_step": classes[dom]["launches_per_step"],
                    "by_class": by_class,
                    "step_floor_ms": sum(d["floor_ms"] for d in by_class.values()),
                    "step_measured_ms_eager_events": prof_total,
                    "exp_peak": f"{EXP_PER_CLK_PER_SM} exponentials/clk/SM (MUFU 16 + FMA-pipe polynomial 15.3, profiles/r2_pipe_rate.txt)"}

    # ---------------- reduce over ranks (max time), assemble the line ----------------
    if world > 1:
        tt = torch.tensor([ms_total, ms_e2e, ms_eager], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e, ms_eager = float(tt[0]), float(tt[1]), float(tt[2])
    ms_step = ms_total / K
    value = world * B / (T * ms_step * 1e-3)
    e2e_value = world * B / (T * (ms_e2e / K) * 1e-3)

    cpu_baseline, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the oracle runs on the GPU arm's own weights and on image 0 of its batch, so its first step doubles as a parity check
        i0 = T - 1
        shared = dict(unet={k: v.detach().cpu() for k, v in wl.unet.state_dict().items()}, xt=x0[0:1].cpu(), z=zs[0][0:1].cpu(), i=i0)
        if spec["kind"] == "sgg":
            shared.update(seg={k: v.detach().cpu() for k, v in wl.seg.state_dict().items()},
                          srgan={k: v.detach().cpu() for k, v in wl.srgan.state_dict().items()}, gt=wl.gt[0:1].cpu())
        v, sec, cores, first = cpu_reference_rate(WORKLOADS[args.workload], args.cpu_steps, 1, shared=shared)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sec_per_step_per_image": sec,
                        "sample": f"oracle port (PyTorch fp32, {cores} threads): image 0 of the batch, {args.cpu_steps} timed reverse steps "
                                  f"after 1 warm-up, extrapolated linearly to {T} steps"}
        # parity of the measured path (outside every timed region): the same first step on the GPU, full batch, image 0 compared
        eps = wl.unet(x0, wl.t_tensor(i0))
        mu, sigma, _ = wl.sched.sample_prev_timestep(x0, eps, i0, z=zs[0])
        base_gpu = (mu + sigma)[0:1].cpu()
        got = wl.step(x0, 0, zs[0])[0:1].cpu() if wl.timestep(0) == i0 else None
        ref_x, ref_base = first
        import math
        err = (got - ref_x).double()
        parity = {"what": f"x_(t-1) of image 0 after one reverse step at t = {i0}: GPU batch of {B} vs the fp32 oracle on the same weights / inputs",
                  "max_abs": float(err.abs().max()), "rms_rel": float(err.norm() / ref_x.double().norm()),
                  "psnr_db": 10 * math.log10(float(ref_x.abs().max()) ** 2 / max(float((err ** 2).mean()), 1e-30))}
        if spec["kind"] == "sgg":
            d_ref, d_gpu = (ref_x.double() - ref_base.double()), (got.double() - base_gpu.double())
            parity["guidance_term_rms_rel"] = float((d_gpu - d_ref).norm() / d_ref.norm())
            parity["guidance_term_cosine"] = float((d_gpu * d_ref).sum() / (d_gpu.norm() * d_ref.norm() + 1e-300))
    secondary = None
    if world > 1 and not args.no_secondary:
        del wl
        torch.cuda.empty_cache()
        secondary = secondary_training(dev, rank, world, peaks)
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W_,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": spec["desc"], "batch_per_gpu": B, "latent": [spec["h"], spec["w"]], "schedule_steps": T,
                       "step": "one reverse-diffusion step over the batch (UNet forward + posterior"
                               + (" + SRGAN x4 + DeepLabV3+ forward/CE/input-gradient + guidance update)" if spec["kind"] == "sgg" else " update)"),
                       "launch": "one cudaGraphLaunch per step (captured reverse step, timestep and noise in static device buffers)" if use_graph
                                 else "eager: one host launch per kernel",
                       "l2": "per-step working set (GBs of activations) exceeds the 126 MB L2; no explicit flush",
                       "weights": "random init (UNet seed 3455, seg 42, SRGAN 0), BatchNorm statistics randomised"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": bytes_io, "d2h_bytes_per_step": bytes_io,
                    "ms_per_step": ms_e2e / K},
            "gpu_launches": int(launches), "launches_per_step": launches / K,
            "graph_launches": K if use_graph else 0,
            "eager": {"ms_per_step": ms_eager / K, "value": world * B / (T * (ms_eager / K) * 1e-3), "host_launches_per_step": eager_launches / K},
            "clocks": clocks,
            "roofline": roofline,
            "kernel_classes": classes,
            "step_gflop_per_image": flops_step / B / 1e9,
            "step_gflop_parts_per_image": {k: v / B / 1e9 for k, v in flop_parts.items()},
            "step_tflops": flops_step / (ms_step * 1e-3) / 1e12,
            "step_frac_of_tensor_peak": flops_step / (ms_step * 1e-3) / 1e12 / peaks["tf_sustained"],
            "cpu_baseline": cpu_baseline,
            "parity": parity,
            "secondary": secondary,
            "peak_hbm_gb": torch.cuda.max_memory_allocated(dev) / 1e9,
            "finite": finite,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
