"""CPU tests of the DDIM sampler's host side: schedule construction and rejections, the coefficient table against the float64
formulas, its reduction to the DDPM posterior at stride 1 and eta = 1, and the translation driver's argument checks."""
import math

import pytest
import torch


def _sched(T=1000):
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    return LinearNoiseScheduler(T, 1e-4, 0.02)


def test_default_timesteps_are_the_rounded_linspace_descending():
    s = _sched()
    d = s.ddim(50, eta=0.5)
    assert d.timesteps == [round(x) for x in torch.linspace(0, 999, 50, dtype=torch.float64).tolist()][::-1]
    assert d.timesteps[0] == 999 and d.timesteps[-1] == 0 and len(d.timesteps) == 50 and d.eta == 0.5
    assert s.ddim(1000, eta=1).timesteps == list(range(999, -1, -1))
    assert s.ddim(4, num_timesteps=12).timesteps == [11, 7, 4, 0]
    assert s.ddim(3, num_timesteps=500).timesteps == [499, 250, 0]
    assert s.ddim(1, num_timesteps=1).timesteps == [0]
    assert s.ddim(timesteps=[900, 400, 7], eta=0.2).timesteps == [900, 400, 7]
    assert s.ddim(timesteps=torch.tensor([5, 3]), num_timesteps=6).timesteps == [5, 3]


@pytest.mark.parametrize("kw", [
    dict(timesteps=[]),
    dict(timesteps=[5, 5, 1]),
    dict(timesteps=[5, 3, 3]),
    dict(timesteps=[1000, 3]),
    dict(timesteps=[7, -1]),
    dict(timesteps=[3, 5]),
    dict(timesteps=[5.5, 1]),
    dict(timesteps=[11, 0], num_timesteps=10),
    dict(num_steps=10, eta=-0.1),
    dict(num_steps=10, eta=1.5),
    dict(num_steps=10, eta=float("nan")),
    dict(num_steps=1001),
    dict(num_steps=13, num_timesteps=12),
    dict(num_steps=0),
    dict(num_steps=1),
    dict(num_steps=10, num_timesteps=1001),
    dict(num_steps=10, timesteps=[5, 0]),
    dict(),
])
def test_ddim_rejects(kw):
    with pytest.raises(ValueError):
        _sched().ddim(**kw)


def _formula(acp, t, tp, eta):
    """float64 coefficients of the step t -> tp (tp None: the final step to x0)."""
    a = float(acp[t])
    if tp is None:
        return [math.sqrt(a), math.sqrt(1 - a), 1.0, 0.0, 0.0]
    ap = float(acp[tp])
    sigma = eta * math.sqrt((1 - ap) / (1 - a) * (1 - a / ap))
    return [math.sqrt(a), math.sqrt(1 - a), math.sqrt(ap), math.sqrt(max(0.0, 1 - ap - sigma * sigma)), sigma]


@pytest.mark.parametrize("kw", [dict(num_steps=50, eta=0.0), dict(num_steps=17, eta=0.5, num_timesteps=500),
                                dict(timesteps=[999, 600, 3], eta=1.0), dict(num_steps=12, eta=1.0, num_timesteps=12)])
def test_coefficient_table_matches_the_float64_formulas(kw):
    s = _sched()
    d = s.ddim(**kw)
    n = d.num_timesteps
    assert d.coef_table.dtype == torch.float32 and tuple(d.coef_table.shape) == (5, n)
    acp = s._host["alpha_cum_prod"].double()
    ts = d.timesteps
    for k, t in enumerate(ts):
        want = torch.tensor(_formula(acp, t, ts[k + 1] if k + 1 < len(ts) else None, d.eta), dtype=torch.float64)
        # each coefficient is rounded to fp32 exactly once
        assert torch.equal(d.coef_table[:, t], want.float()), t
    others = [t for t in range(n) if t not in set(ts)]
    assert torch.equal(d.coef_table[:, others], torch.tensor([1.0, 0.0, 1.0, 0.0, 0.0]).unsqueeze(1).expand(5, len(others)))


@pytest.mark.parametrize("T", [12, 1000])
def test_stride_one_eta_one_reduces_to_ddpm(T):
    """A stride-1, eta = 1 DDIM step is the DDPM posterior: mean = x / sqrt(alpha_t) - beta_t / (s_t sqrt(alpha_t)) eps with
    sigma_t^2 = (1 - acp_{t-1}) / (1 - acp_t) beta_t.  DDIM derives alpha_t and beta_t from the fp32 acp table
    (acp_t / acp_{t-1}); the DDPM tables use the fp32 betas, and fp32 cumprod makes the two agree only to 2^-24 in absolute
    terms.  So the x-coefficient agrees to a few fp32 ulps, and the eps-coefficient and sigma, which carry beta_t, agree to
    a few 2^-24 / beta_t relative (measured: x 1.9 ulp; eps 3.4 and sigma 1.0 in units of 2^-24 / beta_t at T = 1000)."""
    s = _sched(T)
    d = s.ddim(T, eta=1.0)
    tab = d.coef_table.double()
    beta, alpha = s._host["betas"].double(), s._host["alphas"].double()
    s_t, sig = torch.tensor(s._coef["s"], dtype=torch.float64), torch.tensor(s._coef["sigma"], dtype=torch.float64)
    t = torch.arange(1, T)
    u = 2.0 ** -24
    x_coef, x_ref = tab[2, t] / tab[0, t], 1 / alpha[t].sqrt()
    assert float(((x_coef - x_ref) / x_ref).abs().max()) < 4 * u
    e_coef, e_ref = tab[3, t] - tab[2, t] * tab[1, t] / tab[0, t], -beta[t] / (s_t[t] * alpha[t].sqrt())
    assert bool((((e_coef - e_ref) / e_ref).abs() < 4 * u / beta[t]).all())
    assert bool((((tab[4, t] - sig[t]) / sig[t]).abs() < 2 * u / beta[t]).all())
    # the final step (t = 0) is the DDPM t == 0 mean: (x - s_0 eps) / sqrt(acp_0), no noise
    assert tab[2, 0] == 1.0 and tab[3, 0] == 0.0 and tab[4, 0] == 0.0
    assert torch.equal(d.coef_table[1, 0], torch.tensor(s._coef["s"][0]))


def test_eta_zero_has_no_noise_and_eta_scales_sigma():
    s = _sched()
    d0, d1, dh = s.ddim(20, eta=0.0), s.ddim(20, eta=1.0), s.ddim(20, eta=0.5)
    assert float(d0.coef_table[4].abs().max()) == 0.0
    ts = d1.timesteps[:-1]
    assert torch.allclose(dh.coef_table[4, ts].double(), 0.5 * d1.coef_table[4, ts].double(), rtol=1e-6, atol=0)
    # eta = 0: d = sqrt(1 - acp_prev), the deterministic DDIM direction
    acp = s._host["alpha_cum_prod"].double()
    for k, t in enumerate(ts):
        assert float(d0.coef_table[3, t]) == float(torch.tensor(math.sqrt(1 - float(acp[d0.timesteps[k + 1]]))).float())


def _inputs():
    return torch.zeros(1, 3, 16, 32), torch.zeros(1, 64, 128, dtype=torch.long)


def test_sample_with_sgg_rejects_bad_ddim_use_before_device_work():
    from weatherconverter_b200.translation import sample_with_sgg
    x, gt = _inputs()
    s = _sched()
    with pytest.raises(ValueError, match="beyond"):
        sample_with_sgg(x, None, None, None, gt, None, n_steps=500, sampler=s.ddim(50, eta=1.0))
    with pytest.raises(ValueError, match="reference_quirks"):
        sample_with_sgg(x, None, None, None, gt, None, n_steps=500, sampler=s.ddim(50, eta=1.0, num_timesteps=500),
                        reference_quirks=True)
    for mode in ("gsg", "alternate", "lcg"):
        with pytest.raises(ValueError, match="silently do nothing"):
            sample_with_sgg(x, None, None, None, gt, None, n_steps=500, sampler=s.ddim(50, num_timesteps=500), mode=mode)


def test_sample_tensor_rejects_a_schedule_beyond_the_chain():
    from weatherconverter_b200.diffusion_model.sample_ddpm import sample_tensor
    s = _sched()
    with pytest.raises(ValueError, match="beyond"):
        sample_tensor(None, s, (1, 3, 8, 8), num_timesteps=12, sampler=s.ddim(10))
