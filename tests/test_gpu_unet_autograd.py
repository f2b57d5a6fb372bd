"""GPU tests of the differentiable Unet (Unet.differentiable = True): torch autograd through the sm_100a training plan,
against torch autograd through the fp32 oracle (itself pinned to the reference's gradients by train_step.pt), against the
fused DenoisingTrainer step, and the plan pool's lifetime rules."""
import zlib

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda")


def _build(cfg, seed, dev):
    from oracle.weights import synth_state_dict
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet, param_spec
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    sd = synth_state_dict({k: (v, torch.float32) for k, v in param_spec(cfg).items()}, seed)
    model = Unet(cfg).to(dev)
    model.load_state_dict(sd)
    return sd, model, LinearNoiseScheduler(1000, 1e-4, 0.02)


def _small_cfg(im_size):
    from oracle.unet import DEFAULT_MODEL_CONFIG
    cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = im_size
    return cfg


def _rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-20))


def _cos(a, b):
    return float((a * b).sum() / (a.norm() * b.norm() + 1e-20))


def _grads(model):
    return {n: p.grad.detach().clone() for n, p in model.named_parameters()}


def test_weighted_smooth_l1_gradients_vs_oracle():
    """An arbitrary loss (per-pixel weighted smooth L1), ragged t, x.requires_grad_(): all parameter gradients and dL/dx
    against torch autograd through oracle.unet.unet_forward in fp32 on the host."""
    from oracle.unet import unet_forward
    dev = _dev()
    cfg = _small_cfg(64)
    sd, model, _ = _build(cfg, 99, dev)
    model.differentiable = True
    g = torch.Generator().manual_seed(21)
    x = torch.randn(3, 3, 32, 64, generator=g)
    target = torch.randn(3, 3, 32, 64, generator=g)
    weight = torch.rand(3, 3, 32, 64, generator=g) * 2
    t = torch.tensor([5, 420, 999])

    def loss_fn(pred, target, weight):
        return (weight * F.smooth_l1_loss(pred, target, reduction="none", beta=0.5)).mean()

    xd = x.to(dev).requires_grad_()
    loss = loss_fn(model(xd, t.to(dev)), target.to(dev), weight.to(dev))
    loss.backward()
    torch.cuda.synchronize()

    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xr = x.clone().requires_grad_()
    loss_ref = loss_fn(unet_forward(params, cfg, xr, t), target, weight)
    loss_ref.backward()
    loss, loss_ref = loss.item(), loss_ref.item()

    assert abs(loss - loss_ref) < 3e-3 * abs(loss_ref), (loss, loss_ref)
    mine = dict(model.named_parameters())
    assert set(params) == set(mine)
    num = den = 0.0
    worst, worst_name, cos_min = 0.0, "", 1.0
    for k, p_ref in params.items():
        g_ref, gg = p_ref.grad, mine[k].grad.detach().cpu()
        assert gg.shape == g_ref.shape and torch.isfinite(gg).all(), k
        a, b = float((gg - g_ref).norm()), float(g_ref.norm())
        num += a * a
        den += b * b
        if a / (b + 1e-12) > worst:
            worst, worst_name = a / (b + 1e-12), k
        cos_min = min(cos_min, _cos(gg, g_ref))
    dx, dx_ref = xd.grad.cpu(), xr.grad
    dx_rel, dx_cos = _rel(dx, dx_ref), _cos(dx, dx_ref)
    print(f"weighted smooth-L1: loss {loss:.6f} vs {loss_ref:.6f}; parameter gradients rms-rel "
          f"{(num / den) ** 0.5:.3e}, worst {worst_name} {worst:.3e}, min cosine {cos_min:.5f}; "
          f"dL/dx rms-rel {dx_rel:.3e}, cosine {dx_cos:.6f}")
    assert (num / den) ** 0.5 < 3e-2
    assert worst < 1.5e-1, (worst_name, worst)
    assert cos_min > 0.995, cos_min
    assert dx_rel < 3e-2, dx_rel
    assert dx_cos > 0.995, dx_cos


def test_generic_mse_equals_fused_step_at_c5():
    """Default config, batch 64, 128x256: MSE through the differentiable Unet and DenoisingTrainer.forward_backward on the
    same weights and inputs.  Only dpred differs, by the rounding of torch's mse_loss backward against the fused kernel."""
    from oracle.unet import DEFAULT_MODEL_CONFIG
    from weatherconverter_b200.diffusion_model.train_ddpm import DenoisingTrainer
    dev = _dev()
    _, model, sched = _build(dict(DEFAULT_MODEL_CONFIG), 3455, dev)
    g = torch.Generator().manual_seed(8)
    images = (torch.rand(64, 3, 128, 256, generator=g) * 2 - 1).to(dev)
    noise = torch.randn(64, 3, 128, 256, generator=g).to(dev)
    t = torch.randint(0, 1000, (64,), generator=g).to(dev)
    noisy = sched.add_noise(images, noise, t)

    model.differentiable = True
    loss_g = F.mse_loss(model(noisy, t), noise)
    loss_g.backward()
    grads_g = _grads(model)
    loss_g = loss_g.item()
    model.differentiable = False
    model.zero_grad(set_to_none=True)
    model._train_plans.clear()          # give the 41 GB workspace back before the trainer binds its own

    trainer = DenoisingTrainer(model, sched, lr=1e-4)
    loss_f = float(trainer.forward_backward(noisy, t, noise))
    torch.cuda.synchronize()
    num = den = 0.0
    for n, p in model.named_parameters():
        a, b = float((p.grad - grads_g[n]).norm()), float(p.grad.norm())
        num += a * a
        den += b * b
    rel = (num / den) ** 0.5
    print(f"C5 generic vs fused: loss {loss_g:.8f} vs {loss_f:.8f} (rel {abs(loss_g - loss_f) / loss_f:.2e}), "
          f"gradient rms-rel {rel:.3e}")
    assert abs(loss_g - loss_f) <= 1e-6 * abs(loss_f)
    assert rel <= 1e-3


def test_data_only_backward():
    """Every parameter frozen: dL/dx equals the full backward's bit for bit, with strictly fewer launches, and no
    parameter gets a .grad."""
    from weatherconverter_b200 import ops
    dev = _dev()
    _, model, _ = _build(_small_cfg(32), 7, dev)
    model.differentiable = True
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 3, 32, 64, generator=g).to(dev)
    w = torch.randn(2, 3, 32, 64, generator=g).to(dev)
    t = torch.tensor([3, 700], device=dev)

    def run():
        xr = x.clone().requires_grad_()
        loss = (model(xr, t) * w).sum()
        torch.cuda.synchronize()
        before = ops.launch_count()
        loss.backward()
        torch.cuda.synchronize()
        return xr.grad, ops.launch_count() - before

    dx_full, n_full = run()
    model.zero_grad(set_to_none=True)
    model.requires_grad_(False)
    dx_data, n_data = run()
    print(f"backward launches: full {n_full}, data-only {n_data}")
    assert torch.equal(dx_full, dx_data)
    assert n_data < n_full
    assert all(p.grad is None for p in model.parameters())


def test_gradient_accumulation_and_two_live_graphs():
    dev = _dev()
    _, model, _ = _build(_small_cfg(32), 11, dev)
    model.differentiable = True
    g = torch.Generator().manual_seed(6)
    x1, x2 = (torch.randn(2, 3, 32, 32, generator=g).to(dev) for _ in range(2))
    t1, t2 = torch.tensor([10, 500], device=dev), torch.tensor([900, 1], device=dev)

    def loss(x, t):
        return model(x, t).square().mean()

    loss(x1, t1).backward()
    g1 = _grads(model)
    model.zero_grad(set_to_none=True)
    loss(x2, t2).backward()
    g2 = _grads(model)
    # two backward calls without zero_grad accumulate
    model.zero_grad(set_to_none=True)
    loss(x1, t1).backward()
    loss(x2, t2).backward()
    for n, p in model.named_parameters():
        assert torch.equal(p.grad, g1[n] + g2[n]), n
    # two live graphs (the second forward leases a second plan), one backward of the summed losses
    model.zero_grad(set_to_none=True)
    total = loss(x1, t1) + loss(x2, t2)
    assert len(model._train_plans[(2, 32, 32)]) == 2
    total.backward()
    for n, p in model.named_parameters():
        assert torch.equal(p.grad, g1[n] + g2[n]), n


def test_reference_loop_l1_adamw_clip_vs_oracle():
    """The reference's step body, unmodified, with nn.L1Loss, AdamW(weight_decay=1e-2) and clip_grad_norm_(..., 1.0), three
    steps on the GPU and the same three steps on the oracle's parameters on the host."""
    from oracle.scheduler import OracleScheduler
    from oracle.unet import unet_forward
    dev = _dev()
    cfg = _small_cfg(32)
    sd, model, sched = _build(cfg, 5, dev)
    model.differentiable = True
    lr = 1e-4
    g = torch.Generator().manual_seed(17)
    images = torch.rand(2, 3, 32, 64, generator=g) * 2 - 1
    noises = [torch.randn(2, 3, 32, 64, generator=g) for _ in range(3)]
    ts = [torch.randint(0, 1000, (2,), generator=g) for _ in range(3)]

    criterion = nn.L1Loss()
    optimizer = torch.optim.AdamW(model.parameters(), lr=lr, weight_decay=1e-2)
    ref_params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref_opt = torch.optim.AdamW(list(ref_params.values()), lr=lr, weight_decay=1e-2)
    osched = OracleScheduler(1000, 1e-4, 0.02)
    for step in range(3):
        im, noise, t = images.to(dev), noises[step].to(dev), ts[step].to(dev)
        optimizer.zero_grad()
        noisy = sched.add_noise(im, noise, t)
        noise_pred = model(noisy, t)
        loss = criterion(noise_pred, noise)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        optimizer.step()

        ref_opt.zero_grad()
        loss_ref = criterion(unet_forward(ref_params, cfg, osched.add_noise(images, noises[step], ts[step]), ts[step]),
                             noises[step])
        loss_ref.backward()
        torch.nn.utils.clip_grad_norm_(list(ref_params.values()), 1.0)
        ref_opt.step()
        loss, loss_ref = loss.item(), loss_ref.item()
        print(f"step {step}: loss {loss:.6f} vs oracle {loss_ref:.6f}")
        assert abs(loss - loss_ref) < 3e-3 * abs(loss_ref), (step, loss, loss_ref)
    bad = n_s = 0
    mine = dict(model.named_parameters())
    for k, ref in ref_params.items():
        p, r = mine[k].detach().cpu().flatten(), ref.detach().flatten()
        idx = torch.randint(0, p.numel(), (min(32, p.numel()),),
                            generator=torch.Generator().manual_seed(zlib.crc32(k.encode()) & 0x7FFFFFFF))
        bad += int(((p[idx] - r[idx]).abs() > 0.5 * lr * 3).sum())
        n_s += idx.numel()
    print(f"after 3 AdamW steps: {bad} of {n_s} sampled weights differ by more than 0.5*lr per step")
    assert bad <= 0.05 * n_s


def test_pool_lifetime_memory_and_errors():
    dev = _dev()
    cfg = _small_cfg(32)
    _, model, sched = _build(cfg, 13, dev)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(2, 3, 32, 32, generator=g).to(dev)
    t = torch.tensor([250], device=dev)          # one timestep for the batch: broadcast to [B]

    with torch.no_grad():
        ref = model(x, t)
    y = model(x, t)                               # differentiable = False: the inference plan, grad mode or not
    assert y.grad_fn is None and torch.equal(y, ref)
    model.differentiable = True
    with torch.no_grad():
        y = model(x, t)
    assert y.grad_fn is None and torch.equal(y, ref)

    for _ in range(10):                           # graphs freed without a backward give their plan back
        model(x, t)
    assert len(model._train_plans[(2, 32, 32)]) == 1

    with pytest.raises(RuntimeError, match="out="):
        model(x, t, out=torch.empty_like(x))

    loss = model(x, t).square().mean()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already been backpropagated"):
        loss.backward()
    del loss

    # steady state of the reference loop: nothing grows after the optimizer state exists
    optimizer = torch.optim.AdamW(model.parameters(), lr=1e-4)
    images = torch.rand(2, 3, 32, 32, generator=g).to(dev) * 2 - 1
    mem = []
    for step in range(5):
        optimizer.zero_grad()
        noise = torch.randn(images.shape, generator=g).to(dev)
        tt = torch.randint(0, 1000, (2,), generator=g).to(dev)
        loss = F.mse_loss(model(sched.add_noise(images, noise, tt), tt), noise)
        loss.backward()
        optimizer.step()
        torch.cuda.synchronize()
        mem.append(torch.cuda.memory_allocated())
    print(f"memory_allocated after steps 1..5: {mem}")
    assert mem[4] == mem[1]
    assert len(model._train_plans[(2, 32, 32)]) == 1


def test_train_runs_l1_loss_on_the_generic_path():
    from weatherconverter_b200.diffusion_model.train_ddpm import train
    dev = _dev()
    _, model, sched = _build(_small_cfg(32), 7, dev)
    g = torch.Generator().manual_seed(9)
    images = torch.rand(4, 3, 32, 32, generator=g) * 2 - 1
    noise = torch.randn(4, 3, 32, 32, generator=g).to(dev)
    t = torch.tensor([50, 300, 600, 900], device=dev)
    criterion = nn.L1Loss()

    def fixed_batch_loss():
        with torch.no_grad():
            return float(criterion(model(sched.add_noise(images.to(dev), noise, t), t), noise))

    before = fixed_batch_loss()
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-3)
    logged = []
    losses = train([images] * 4, model, optimizer, criterion, sched, epochs=1, log_interval=2, seed=1,
                   on_log=lambda ep, it, v: logged.append((ep, it)))
    after = fixed_batch_loss()
    print(f"train() with L1Loss: step losses {losses}, fixed-batch loss {before:.5f} -> {after:.5f}")
    assert len(losses) == 4 and all(torch.isfinite(torch.tensor(losses)))
    assert logged == [(1, 2), (1, 4)]
    assert model.differentiable is False
    assert after < before
    assert len(optimizer.state) == len(list(model.parameters()))
