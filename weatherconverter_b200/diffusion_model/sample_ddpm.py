"""Unconditional DDPM sampling with the reference's entry points (diffusion_model/sample_ddpm.py:17-87).

``sample`` keeps the reference signature and side effect (writes a PNG grid).  ``sample_tensor`` is the
same reverse loop returning the final tensor, with the knobs parity tests and benchmarks need: injected
``x_T`` / per-step noise, non-square sizes, on-device noise, per-step recording.
"""
import os
from datetime import datetime

import torch
import yaml

from .config.models import Config, DiffusionConfig, ModelConfig, TrainingConfig
from .models.unet_base import Unet
from .scheduler.linear_noise_scheduler import LinearNoiseScheduler

device = torch.device('cuda' if torch.cuda.is_available() else 'cpu')


def load_config(config_path: str) -> Config:
    with open(config_path, 'r') as file:
        return Config(**yaml.safe_load(file))


@torch.no_grad()
def sample_tensor(model, scheduler, shape=None, num_timesteps=None, xT=None, noise=None, device_noise=False,
                  generator=None, record=None, use_graph=False, sampler=None):
    """Reverse loop of sample_ddpm.py:35-44.  noise: optional [T, *shape] tensor (or callable i -> tensor), noise[i]
    is the z drawn at step i.  device_noise=True draws z with the CUDA generator instead of the reference's CPU
    generator (throughput runs).  sampler: a DDIMSchedule (``scheduler.ddim(...)``); the loop then walks
    ``sampler.timesteps`` instead of every timestep, and noise[t] / noise(t) is the z of the step that starts at t.
    ``record`` gets one entry per executed step.  Returns x_0 (un-clamped, as the loop leaves it)."""
    T = num_timesteps if num_timesteps is not None else scheduler.num_timesteps
    steps = list(reversed(range(T))) if sampler is None else sampler.timesteps
    if sampler is not None and max(steps) >= T:
        raise ValueError(f"the DDIM schedule has timestep {max(steps)}, beyond this {T}-step chain")
    sched = scheduler if sampler is None else sampler
    noisy = sampler is None or sampler.eta > 0                     # eta == 0: DDIM draws no noise
    if xT is None:
        xT = torch.randn(shape).to(device)                         # reference :35 (CPU generator, then H2D)
    xt = xT.to(device).float().contiguous()
    if use_graph and len(steps) > 1:
        # every step but the last replays ONE captured CUDA graph (UNet forward + fused posterior update with the timestep
        # read on the device): one cudaGraphLaunch per step instead of ~330 kernel launches; bit-identical to the eager loop
        from ..graphs import StepGraph

        def step(x, t_dev, z):
            return sched.step_indexed(x, model(x, t_dev), t_dev, z)
        sg = StepGraph(step, xt.shape, xt.device)
        sg.load(xt)
        t_all = torch.arange(T, device=xt.device, dtype=torch.int64)
        for i in steps[:-1]:
            if noise is not None:
                z = (noise(i) if callable(noise) else noise[i]).to(xt.device)
            elif not noisy:
                z = None
            elif device_noise:
                z = torch.randn(xt.shape, device=xt.device, generator=generator)
            else:
                z = scheduler._draw(xt)
            sg.replay(t_all[i:i + 1], z)
            if record is not None:
                record.append(sg.xt.clone())
        xt = sched.step(sg.xt, model(sg.xt, t_all[steps[-1]:steps[-1] + 1]), steps[-1])
        if record is not None:
            record.append(xt.clone())
        return xt
    eps = torch.empty_like(xt)
    for i in steps:
        t = torch.as_tensor(i).unsqueeze(0).to(xt.device)          # reference :39
        model(xt, t, out=eps)
        if i == steps[-1]:
            z = None
        elif noise is not None:
            z = noise(i) if callable(noise) else noise[i]
            z = z.to(xt.device)
        elif device_noise and noisy:
            z = torch.randn(xt.shape, device=xt.device, generator=generator)
        else:
            z = None                                               # scheduler draws from the CPU generator (:110)
        xt = sched.step(xt, eps, i, z=z)                           # fused mean + sigma*z (reference :42-44)
        if record is not None:
            record.append(xt.clone())
    return xt


def sample(model, scheduler: LinearNoiseScheduler, train_config: TrainingConfig, model_config: ModelConfig,
           diffusion_config: DiffusionConfig, save_path: str = 'diffusion_model_v2/outputs/samples'):
    r"""Sample stepwise by going backward one timestep at a time and save the x0 grid (reference :23-53)."""
    xt = sample_tensor(model, scheduler,
                       (train_config.sample_size, model_config.im_channels, model_config.im_size, model_config.im_size),
                       num_timesteps=diffusion_config.num_timesteps)
    # reference :47-51 (clamp, (x+1)/2, make_grid, ToPILImage) as one byte-exact kernel; only the uint8 grid crosses PCIe
    from PIL import Image
    from ..image_io import ddpm_grid_uint8
    img = Image.fromarray(ddpm_grid_uint8(xt, train_config.num_grid_rows).cpu().numpy())
    os.makedirs(save_path, exist_ok=True)
    now = datetime.now()
    img.save(os.path.join(save_path, f'x_410{now.hour}{now.minute}{now.second}.png'))
    img.close()


def load_model(model_path: str, model_config: ModelConfig) -> torch.nn.Module:
    model = Unet(model_config).to(device)
    checkpoint = torch.load(model_path, map_location=device)
    model.load_state_dict(checkpoint['model_state_dict'])
    model.eval()
    return model


def load_scheduler(diffusion_config: DiffusionConfig) -> LinearNoiseScheduler:
    return LinearNoiseScheduler(num_timesteps=diffusion_config.num_timesteps, beta_start=diffusion_config.beta_start,
                                beta_end=diffusion_config.beta_end)


def infer(config: Config):
    epoch = 410
    checkpoint_path = os.path.join(config.folders.checkpoints, f'{epoch}-checkpoint.ckpt')
    model = load_model(checkpoint_path, config.model)
    scheduler = load_scheduler(config.diffusion)
    with torch.no_grad():
        sample(model, scheduler, config.training, config.model, config.diffusion, config.folders.samples)


if __name__ == '__main__':
    infer(load_config('diffusion_model/config/config.yaml'))
