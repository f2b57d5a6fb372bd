"""GPU parity of the legacy UNet (diffusion_model/models/old_modules.py) and the sample_integrated loop against golden
tensors produced by the reference's own modules (tests/golden/make_golden.py:g_legacy)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda")


def _psnr(a, b):
    mse = float(((a - b) ** 2).mean())
    peak = float(b.abs().max())
    return 10 * math.log10(peak * peak / max(mse, 1e-30))


def _model(d, dev):
    from oracle.legacy_unet import legacy_param_spec
    from oracle.weights import synth_state_dict
    from weatherconverter_b200.diffusion_model.models.old_modules import UNet
    m = UNet().to(dev).eval()
    m.load_state_dict(synth_state_dict(legacy_param_spec(), d["seed"]))
    return m


def test_legacy_unet_forward(golden):
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    dev = _dev()
    d = golden("legacy_unet.pt")
    m = _model(d, dev)
    s = LinearNoiseScheduler(1000, 1e-4, 0.02)
    t = s.one_minus_cum_prod.to(dev)[d["t_idx"].to(dev)].view(-1, 1, 1, 1)
    y = m(d["x"].to(dev), t).cpu()
    rel = float((y - d["y"]).norm() / d["y"].norm())
    print(f"legacy UNet forward: rms-rel {rel:.3e}, PSNR {_psnr(y, d['y']):.1f} dB, {m.launches_per_forward()} launches")
    assert rel < 2.5e-2, rel        # bf16 storage / fp32 accumulation vs the fp32 reference


def test_sample_integrated_trajectory(golden):
    from weatherconverter_b200.diffusion_model.sample_integrated import postprocess, sample_tensor
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    dev = _dev()
    d = golden("legacy_unet.pt")
    m = _model(d, dev)
    s = LinearNoiseScheduler(1000, 1e-4, 0.02)
    rec = []
    xt = sample_tensor(m, s, num_timesteps=3, xT=d["xT"], noise=d["zs"], record=rec)
    for k in range(3):    # the golden keeps each step at a fixed sample of its elements, traj_idx
        p = _psnr(rec[k].cpu().flatten()[d["traj_idx"]], d["traj"][k])
        print(f"step {k}: PSNR {p:.1f} dB")
        assert p > 45.0, (k, p)
    img = postprocess(xt)
    assert img.dtype == torch.uint8 and img.shape == (2, 3, 128, 128)
