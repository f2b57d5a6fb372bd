"""SGG-guided translation driver with the reference's entry point (translation.py:46-97).

``sample_with_sgg(input_tensor, diff_model, diff_scheduler, seg_model, gt, srgan_model)`` keeps the reference's
signature and constants (LAMBDA = 60, N = 500).  The driver as shipped cannot finish (SURVEY.md 3.3: D1 the guided x_t
is overwritten, D2 ``mu + None`` at i = 0, D3 LCG shape error on the 2nd iteration, D7 float64 promotion, D8 autograd
graph kept across steps), so the default here is the REPAIRED loop of SURVEY.md 8c: no autograd graph, global
guidance (GSG) on every step i > 0, ``x_t = mu`` at i = 0, guided x_t kept (fp32).  ``mode="alternate"`` restores the
shipped schedule of translation.py:84-87 - local class guidance (LCG, repaired final sum) on even steps, GSG on odd steps.
``reference_quirks=True`` reproduces D1 verbatim (guidance computed, then discarded) for step-level comparison with the
shipped code.
Batches are independent chains: image b is guided by its own loss/gradient (vmap of the reference's B = 1 call).
"""
import torch

from .sgg.sgg import apply_gsg_batch, apply_gsg_through_srgan, apply_lcg
from .srgan_model.inference import inference as srgan_inference

device = torch.device('cuda' if torch.cuda.is_available() else 'cpu')

LAMBDA = 60.0
N_STEPS = 500


def load_input_image(path: str, image_size: int = 128) -> torch.Tensor:
    """translation.py:131,138-145: open the RGB image (host, PIL decode) and run Resize(BILINEAR) + CenterCrop + ToTensor +
    x*2-1 on the GPU, bit-identical to the reference's torchvision/PIL transform (weatherconverter_b200/image_io.py)."""
    import numpy as np
    from PIL import Image
    from . import image_io
    img = torch.from_numpy(np.array(Image.open(path).convert("RGB"))).to(device)
    return image_io.diffusion_input(img, image_size)


def _sample_with_sgg_graphed(xt, diff_model, diff_scheduler, sched, steps, seg_model, gt, srgan_model, n_steps, lam,
                             step_noise, device_noise, generator, mode, record):
    """The loop of sample_with_sgg with every guided step (all but the last) replayed from a captured CUDA graph.  One graph
    per guidance kind in use (GSG and / or LCG); the timestep and the noise are fed through static device buffers."""
    from .graphs import StepGraph
    dev = xt.device
    # GSG runs the segmentor on B images, LCG on 19 B masked images: two plan bindings that must both stay alive
    seg_for = {"gsg": seg_model, "lcg": seg_model.shared_replica() if mode == "alternate" else seg_model}

    def make(kind):
        def step(x, t_dev, z):
            eps = diff_model(x, t_dev)                                                      # reference :74
            mu, sigma, _ = sched.sample_prev_timestep_indexed(x, eps, t_dev, z)             # reference :78
            sr_xt = srgan_inference(srgan_model, x)                                         # reference :81
            if kind == "lcg":
                return apply_lcg(seg_for["lcg"], mu, sigma, sr_xt, gt, lam)                 # reference :84-85
            return apply_gsg_batch(seg_for["gsg"], mu, sigma, sr_xt, gt, lam)               # reference :86-87
        return StepGraph(step, xt.shape, dev)

    kinds = {"gsg": ("gsg",), "lcg": ("lcg",), "alternate": ("gsg", "lcg")}[mode]
    graphs = {k: make(k) for k in kinds} if len(steps) > 1 else {}
    t_all = torch.arange(n_steps, device=dev, dtype=torch.int64)
    cur = xt
    last = len(steps) - 1
    for k, i in enumerate(steps):
        if k == last:
            eps = diff_model(cur, t_all[i:i + 1])
            cur = sched.step(cur, eps, i)                                                   # repair of D2: x_0 = mu
        else:
            if step_noise is not None:
                z = (step_noise(i) if callable(step_noise) else step_noise[i]).to(dev)
            elif device_noise:
                z = torch.randn(cur.shape, device=dev, generator=generator)
            else:
                z = diff_scheduler._draw(cur)                                               # reference scheduler.py:110
            g = graphs["lcg" if (mode == "lcg" or (mode == "alternate" and (last - k) % 2 == 0)) else "gsg"]
            if cur is not g.xt:
                g.load(cur)
            cur = g.replay(t_all[i:i + 1], z)
        if record is not None:
            record.append(cur.clone())
    return srgan_inference(srgan_model, cur)                                                # reference :95-97


@torch.no_grad()
def sample_with_sgg(input_tensor, diff_model, diff_scheduler, seg_model, gt, srgan_model, *, n_steps=N_STEPS,
                    lam=LAMBDA, noise=None, t_forward=None, step_noise=None, device_noise=False, generator=None,
                    guidance=True, mode="gsg", reference_quirks=False, record=None, record_base=None, use_graph=False,
                    criterion=None, grad_through_srgan=False, sampler=None):
    """input_tensor [B,3,h,w] in [-1,1]; gt [B,4h,4w] int64 trainIds (255 = ignore).  Returns sr_x0 [B,3,4h,4w].
    Injection points for parity runs: ``t_forward`` [B] (reference :63 draws randint(0, N)), ``noise`` like the input
    (:64), ``step_noise`` [N, B,3,h,w] or callable i -> z (scheduler.py:110); ``record`` / ``record_base`` collect x_t and
    the unguided mu + sigma of every step.  ``mode``: "gsg" (global guidance on every
    step, the repaired default), "alternate" (reference :84-87: LCG when i is even, GSG when i is odd) or "lcg".
    ``use_graph=True`` captures the guided reverse step once per guidance kind as a CUDA graph (weatherconverter_b200/graphs.py)
    and replays it: one cudaGraphLaunch per step instead of ~440 kernel launches, bit-identical to the eager loop.
    ``criterion``: callable (logits [B,19,H,W], gt [B,H,W]) -> per-image losses [B] that replaces the fused CE(ignore 255) of
    every GSG step (sgg/sgg.py: apply_gsg_batch); eager loop and mode="gsg" only.
    ``grad_through_srgan=True``: every GSG step is guided by the exact d loss / d x_t through the SRGAN generator
    (sgg/sgg.py: apply_gsg_through_srgan) instead of avg_pool2d(d loss / d sr_xt, 4); the SR image is computed once per step.
    The guidance magnitude differs in scale from the pooled stand-in, so ``lam`` may need retuning.  Eager loop, mode="gsg"
    and reference_quirks=False only.
    ``sampler``: a DDIMSchedule (``diff_scheduler.ddim(..., num_timesteps=n_steps)``); the loop walks ``sampler.timesteps``
    instead of all n_steps timesteps, guidance runs on every step but the last with mu = the DDIM mean and sigma = its
    sigma * z, and "alternate" runs LCG on the steps whose position from the end is even.  Choosing ``lam`` for a strided
    schedule is the caller's job: a DDIM step's sigma is larger than a DDPM step's, and nothing is rescaled."""
    if not isinstance(grad_through_srgan, bool):
        raise TypeError("grad_through_srgan must be a bool")
    if grad_through_srgan:
        if use_graph:
            raise ValueError("grad_through_srgan: the step runs torch autograd through the generator, which the step graph "
                             "cannot capture; use use_graph=False")
        if mode != "gsg":
            raise ValueError("grad_through_srgan applies to global guidance (mode='gsg') only")
        if reference_quirks:
            raise ValueError("grad_through_srgan has no reference counterpart; reference_quirks=True cannot be combined with it")
    if mode not in ("gsg", "alternate", "lcg"):
        raise ValueError("mode must be 'gsg', 'alternate' or 'lcg'")
    if criterion is not None:
        if use_graph:
            raise ValueError("criterion: a custom guidance loss runs torch autograd, which the step graph cannot capture; "
                             "use use_graph=False")
        if mode != "gsg":
            raise ValueError("criterion applies to global guidance (mode='gsg') only; local class guidance uses the fused CE")
    if sampler is not None:
        if max(sampler.timesteps) >= n_steps:
            raise ValueError(f"the DDIM schedule has timestep {max(sampler.timesteps)}, beyond this {n_steps}-step chain")
        if reference_quirks:
            raise ValueError("the reference has no DDIM sampler; reference_quirks=True cannot be combined with sampler")
        if guidance and sampler.eta == 0:
            raise ValueError("guidance scales its term by the step's sigma * z, which is 0 for a DDIM schedule with eta == 0: "
                             "guidance would silently do nothing; use eta > 0 or guidance=False")
    sched = diff_scheduler if sampler is None else sampler
    steps = list(reversed(range(n_steps))) if sampler is None else sampler.timesteps
    noisy = sampler is None or sampler.eta > 0                                             # eta == 0: DDIM draws no noise
    x0 = input_tensor.to(device).float().contiguous()
    gt = gt.to(device)
    B = x0.shape[0]
    t = t_forward if t_forward is not None else torch.randint(0, n_steps, (B,))            # reference :63
    noise = noise if noise is not None else torch.randn_like(x0)                            # reference :64
    xt = diff_scheduler.add_noise2(x0, noise.to(device), t.to(device))                      # reference :65
    if use_graph and guidance and not reference_quirks and record_base is None:
        return _sample_with_sgg_graphed(xt, diff_model, diff_scheduler, sched, steps, seg_model, gt, srgan_model, n_steps,
                                        lam, step_noise, device_noise, generator, mode, record)
    eps = torch.empty_like(xt)
    last = len(steps) - 1
    for k, i in enumerate(steps):                                                           # reference :70
        diff_model(xt, torch.as_tensor(i).unsqueeze(0).to(device), out=eps)                # reference :74
        if k == last:
            xt = sched.step(xt, eps, i)                                                     # repair of D2: x_0 = mu
            if record_base is not None:
                record_base.append(xt.clone())
        else:
            if step_noise is not None:
                z = (step_noise(i) if callable(step_noise) else step_noise[i]).to(device)
            elif device_noise and noisy:
                z = torch.randn(xt.shape, device=xt.device, generator=generator)
            else:
                z = None
            mu, sigma, _ = sched.sample_prev_timestep(xt, eps, i, z=z)                      # reference :78
            if record_base is not None:              # the unguided update: x_t - this = the guidance term alone
                record_base.append(mu if sigma is None else mu + sigma)                     # sigma None: DDIM, eta == 0
            if guidance and grad_through_srgan:
                xt = apply_gsg_through_srgan(seg_model, srgan_model, mu, sigma, xt, gt, lam, criterion=criterion)
            elif guidance:
                sr_xt = srgan_inference(srgan_model, xt)                                    # reference :81
                if mode == "lcg" or (mode == "alternate" and (last - k) % 2 == 0):
                    guided = apply_lcg(seg_model, mu, sigma, sr_xt, gt, lam)                # reference :84-85
                else:
                    guided = apply_gsg_batch(seg_model, mu, sigma, sr_xt, gt, lam, criterion=criterion)  # reference :86-87
                xt = (mu + sigma) if reference_quirks else guided                           # reference :90 (D1)
            else:
                xt = mu if sigma is None else mu + sigma
        if record is not None:
            record.append(xt.clone())
    return srgan_inference(srgan_model, xt)                                                 # reference :95-97
