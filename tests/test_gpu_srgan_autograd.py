"""GPU tests of the differentiable SRGAN generator (torch autograd through wc_srgan_forward_saved / wc_srgan_backward_seeded):
forward bits identical to inference, dL/dx against torch autograd through the fp32 oracle (tensor-core and CUDA-core final
layers, positive and sign-mixed PReLU slopes), the seg(G(x)) chain, the plan pool's lifetime rules, and guidance through the
generator."""
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda")


def _rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-20))


def _cos(a, b):
    return float(F.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0))


def _srgan_sd(seed, upscale=4, signed_slopes=False, conditioned=True):
    """Synthetic generator weights.  conditioned: the final pointwise layer scaled by 0.03 and every block2 BatchNorm gain
    halved, so that a gradient error measures the backward's wiring rather than the fixture's sensitivity to bf16 storage:
    - The synthetic weights put the pre-tanh output at a standard deviation near 6, so about 70 % of the pixels saturate, and
      there the tanh derivative 2y(1-y) turns the forward's bf16 rounding into an unbounded relative error of the gradient (a
      CPU emulation of bf16 storage alone then gives cosine 0.89 against fp32).  Scaled, the pre-tanh has a standard
      deviation near 0.3 and no pixel saturates.
    - With full-gain residual branches the 16-block trunk amplifies bf16 rounding: the same emulation gives cosine 0.993 and
      rms-rel 0.11; with halved block2 gains, 0.998-0.999 and 0.04-0.06.
    signed_slopes: every PReLU gets about a third of its slopes negated and some exactly 0, which the synthetic slopes
    (0.25 +- 0.05, all positive) never exercise."""
    from oracle.srgan import srgan_param_spec
    from oracle.weights import synth_state_dict
    sd = synth_state_dict(srgan_param_spec(upscale_factor=upscale), seed)
    if conditioned:
        for k in list(sd):
            if k in ("final_conv.pointwise.weight", "final_conv.pointwise.bias"):
                sd[k] = sd[k] * 0.03
            elif k.endswith("block2.bn.weight"):
                sd[k] = sd[k] * 0.5
    if signed_slopes:
        for k in sd:
            if k.endswith(".act.weight"):
                a = sd[k].clone()
                c = torch.arange(a.numel())
                a[c % 3 == 0] = -a[c % 3 == 0]
                a[c % 8 == 5] = 0.0
                sd[k] = a
    return sd


def _srgan(sd, dev, upscale=4):
    from weatherconverter_b200.srgan_model.models import Generator
    G = Generator(upscale_factor=upscale)
    G.load_state_dict(sd)
    return G.to(dev).eval()


def _seg_conditioned(golden, dev):
    """DeepLabV3+-R50 of the conditioned segmentor fixture (seg_conditioned.pt: the last BN gain of every bottleneck scaled),
    whose input gradient is stable under bf16 storage; the plain random-init segmentor's is chaotic (DESIGN.md section 4)
    and would hide the generator's part of the chain."""
    from oracle.weights import synth_state_dict
    from weatherconverter_b200.seg_model.network import modeling
    dc = golden("seg_conditioned.pt")
    seg = modeling.deeplabv3plus_resnet50(19, 16, False)
    ssd = synth_state_dict(seg.state_dict(), dc["seed"])
    for k in ssd:
        if k.endswith("bn3.weight"):
            ssd[k] = ssd[k] * dc["bn3_gain"]
    seg.load_state_dict(ssd)
    return ssd, seg.to(dev).eval()


def sr_loss(y):
    """Column-weighted L1 distance to a black image on a strided slice plus a squared term over the whole SR output, per
    image: [B].  (An L1 target inside the output range would put kinks where the forward's bf16 rounding flips the sign.)"""
    s = y[:, :, 1::3, ::2]
    wgt = torch.linspace(0.5, 2.0, s.shape[-1], device=y.device, dtype=y.dtype)
    return (wgt * s.abs()).mean((1, 2, 3)) + 0.5 * y.pow(2).mean((1, 2, 3))


def per_image_ce(logits, gt):
    ce = F.cross_entropy(logits, gt, ignore_index=255, reduction="none")
    n = (gt != 255).flatten(1).sum(1).clamp_min(1)
    return ce.flatten(1).sum(1) / n


def _grad_case(upscale, B, h, w, signed_slopes, seed=0):
    """(cosine, rms-rel) of the CUDA dL/dx against torch autograd through the fp32 oracle for sr_loss."""
    from oracle.srgan import generator_forward
    dev = _dev()
    sd = _srgan_sd(seed, upscale, signed_slopes)
    G = _srgan(sd, dev, upscale)
    x = torch.rand(B, 3, h, w, generator=torch.Generator().manual_seed(seed + 7)) * 2 - 1
    xg = x.to(dev).requires_grad_(True)
    sr_loss(G(xg)).sum().backward()
    xr = x.clone().requires_grad_(True)
    sr_loss(generator_forward(sd, xr, upscale_factor=upscale)).sum().backward()
    got = xg.grad.cpu()
    assert torch.isfinite(got).all()
    return _cos(got, xr.grad), _rel(got, xr.grad)


def test_autograd_forward_is_the_inference_bits(golden):
    """The srgan.pt golden input and the C3 shape (B = 32, 64 x 128): the autograd forward == the no-grad forward, bit for bit."""
    dev = _dev()
    d = golden("srgan.pt")
    G = _srgan(_srgan_sd(d["seed"], conditioned=False), dev)
    c3 = torch.rand(32, 3, 64, 128, generator=torch.Generator().manual_seed(3)) * 2 - 1
    for tag, x in (("srgan.pt", d["x"]), ("c3", c3)):
        x = x.to(dev)
        with torch.no_grad():
            plain = G(x)
        xg = x.clone().requires_grad_(True)
        y = G(xg)
        assert y.grad_fn is not None and plain.grad_fn is None
        assert torch.equal(y.detach(), plain), tag
        assert torch.equal(G(x), plain), tag             # x without requires_grad: no graph, same bits
        del y, xg


# Thresholds: 1.25x the rms-rel first measured on a B200 (1000 W), cosine >= 0.99 on every case.  Measured (synthetic /
# signed slopes): x4_tc_final cosine 0.99848 / 0.99810, rms-rel 5.51e-2 / 6.17e-2; x2_cuda_core_final cosine 0.99681 /
# 0.99624, rms-rel 8.03e-2 / 8.67e-2.  A CPU emulation of bf16 storage alone on these weights gives cosine 0.998-0.999.
_MAX_REL = {("x4_tc_final", False): 0.069, ("x4_tc_final", True): 0.077,
            ("x2_cuda_core_final", False): 0.100, ("x2_cuda_core_final", True): 0.108}
_CASES = {
    # (upscale, B, h, w): upscale 4 takes the tensor-core final layer; upscale 2 at an odd latent width (output width 66, not a
    # multiple of 4) takes the CUDA-core final layer
    "x4_tc_final": (4, 2, 32, 64),
    "x2_cuda_core_final": (2, 2, 16, 33),
}


@pytest.mark.parametrize("signed_slopes", [False, True], ids=["synthetic_slopes", "signed_slopes"])
@pytest.mark.parametrize("case", list(_CASES))
def test_input_gradient_vs_oracle_autograd(case, signed_slopes):
    """bf16 activations and gradients over 35 convolutions against fp32 autograd.  A wrong PReLU mask or PixelShuffle index
    shows as a cosine far below 0.99."""
    upscale, B, h, w = _CASES[case]
    cos, rel = _grad_case(upscale, B, h, w, signed_slopes)
    print(f"{case} signed_slopes={signed_slopes}: dL/dx vs fp32 oracle autograd: cosine {cos:.5f} rms-rel {rel:.3e}")
    assert cos >= 0.99, (case, signed_slopes, cos)
    assert rel <= _MAX_REL[case, signed_slopes], (case, signed_slopes, rel)


def test_seg_of_srgan_chain_vs_oracle(golden):
    """seg(G(x)) with per-image CE, x.requires_grad, through the two autograd Functions, against the oracle's chain rule
    (dL/d sr from oracle.deeplab.infer, then autograd through oracle.srgan.generator_forward).  R50 at 128 x 256.
    Measured on a B200 (1000 W): chain cosine 0.91486 / 0.90665, rms-rel 0.416 / 0.431 for the two images, while the
    segmentor's own dL/d sr at the same images is at cosine 0.909 / 0.903, rms-rel 0.425 / 0.442: the error is the
    segmentor's bf16 sensitivity at this low-contrast input, and the generator adds none.  The wiring itself is checked
    against the generator's backward seeded with the fused segmentor gradient (measured rms-rel 7.8e-3).  Thresholds: 1.25x
    the measured error."""
    from oracle import deeplab
    from oracle.srgan import generator_forward
    dev = _dev()
    sd = _srgan_sd(0)
    G = _srgan(sd, dev)
    ssd, seg = _seg_conditioned(golden, dev)
    gen = torch.Generator().manual_seed(11)
    x = torch.rand(2, 3, 32, 64, generator=gen) * 2 - 1
    gt = torch.randint(0, 19, (2, 16, 32), generator=gen).repeat_interleave(8, 1).repeat_interleave(8, 2)   # 8x8 label blocks
    gt[:, :16] = 255
    xg = x.to(dev).requires_grad_(True)
    per_image_ce(seg(G(xg)), gt.to(dev)).sum().backward()
    got = xg.grad.cpu()
    # wiring: the chain equals the generator's backward seeded with the fused plan's gradient at the same SR image
    xw = x.to(dev).requires_grad_(True)
    sr_w = G(xw)
    g_sr_cuda = seg.infer(sr_w.detach(), gt.to(dev))["grad"]
    wired, = torch.autograd.grad(sr_w, xw, g_sr_cuda)
    wrel = _rel(got, wired.cpu())
    print(f"seg(G(x)) vs G backward seeded with the fused segmentor gradient: rms-rel {wrel:.3e}")
    assert wrel <= 1e-2
    for b in range(2):
        xr = x[b:b + 1].clone().requires_grad_(True)
        sr = generator_forward(sd, xr)
        _, g_sr, _ = deeplab.infer(ssd, sr.detach(), gt[b:b + 1])
        ref = torch.autograd.grad(sr, xr, g_sr)[0][0]
        cos, rel = _cos(got[b], ref), _rel(got[b], ref)
        scos, srel = _cos(g_sr_cuda[b].cpu(), g_sr[0]), _rel(g_sr_cuda[b].cpu(), g_sr[0])
        print(f"seg(G(x)) per-image CE, image {b}: dL/dx vs oracle chain rule: cosine {cos:.5f} rms-rel {rel:.3e} "
              f"(segmentor part alone, dL/d sr: cosine {scos:.5f} rms-rel {srel:.3e})")
        assert cos >= 0.88 and rel <= 0.54, (b, cos, rel)
    assert all(p.grad is None for p in list(G.parameters()) + list(seg.parameters()))


def test_graph_hygiene():
    from weatherconverter_b200._lib import lib, ptr, stream_ptr
    dev = _dev()
    G = _srgan(_srgan_sd(0), dev)
    gen = torch.Generator().manual_seed(5)
    x1 = (torch.rand(2, 3, 16, 32, generator=gen) * 2 - 1).to(dev)
    x2 = x1.flip(-1).contiguous()
    key = (2, 16, 32)

    def grad_of(x):
        xg = x.clone().requires_grad_(True)
        sr_loss(G(xg)).sum().backward()
        return xg.grad

    alone1, alone2 = grad_of(x1), grad_of(x2)
    # two live graphs, backpropagated in reverse order
    a, b = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    la, lb = sr_loss(G(a)).sum(), sr_loss(G(b)).sum()
    assert len(G._grad_plans[key]) == 2
    lb.backward()
    la.backward()
    assert torch.equal(a.grad, alone1) and torch.equal(b.grad, alone2)
    # torch.autograd.grad
    xg = x1.clone().requires_grad_(True)
    gx, = torch.autograd.grad(sr_loss(G(xg)).sum(), xg)
    assert torch.equal(gx, alone1)
    # a non-contiguous incoming gradient gives the bits of its contiguous copy
    seed = torch.randn(2, 3, 128, 64, device=dev).transpose(2, 3)
    assert not seed.is_contiguous()
    xa, xb = x1.clone().requires_grad_(True), x1.clone().requires_grad_(True)
    G(xa).backward(seed)
    G(xb).backward(seed.contiguous())
    assert torch.equal(xa.grad, xb.grad)
    # a second backward through the same graph raises
    xg = x1.clone().requires_grad_(True)
    loss = sr_loss(G(xg)).sum()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already been backpropagated"):
        loss.backward()
    # out= is rejected on the autograd path
    with pytest.raises(RuntimeError, match="out="):
        G(x1.clone().requires_grad_(True), out=torch.empty(2, 3, 64, 128, device=dev))
    # the backward without a saved forward returns its error
    plan = G._grad_plans[key][0]
    dx = torch.empty(2, 3, 16, 32, device=dev)
    assert lib().wc_srgan_backward_seeded(plan.handle, ptr(seed.contiguous()), ptr(dx), stream_ptr()) != 0
    assert b"no saved forward" in lib().wc_last_error()
    # the parameters are constants
    assert all(p.grad is None for p in G.parameters())
    # the pool does not grow, and memory is constant across iterations
    del a, b, la, lb, xa, xb, xg, loss
    mem = []
    for _ in range(5):
        grad_of(x1)
        torch.cuda.synchronize()
        mem.append(torch.cuda.memory_allocated())
        assert len(G._grad_plans[key]) == 2
    assert len(set(mem)) == 1, mem


def test_inplace_weight_change_rebuilds_the_pool():
    """load_state_dict copies into the same storage: the autograd path must see the new weights, and the gradient changes."""
    dev = _dev()
    G = _srgan(_srgan_sd(0), dev)
    x = (torch.rand(2, 3, 16, 32, generator=torch.Generator().manual_seed(9)) * 2 - 1).to(dev)

    def run():
        xg = x.clone().requires_grad_(True)
        y = G(xg)
        sr_loss(y).sum().backward()
        return y.detach(), xg.grad

    y0, g0 = run()
    ptrs = [p.data_ptr() for p in G.parameters()]
    G.load_state_dict(_srgan_sd(1))
    assert ptrs == [p.data_ptr() for p in G.parameters()]
    y1, g1 = run()
    with torch.no_grad():
        ref = G(x)
    assert not torch.equal(y1, y0) and not torch.equal(g1, g0)
    assert torch.equal(y1, ref)


def _guidance_setup(golden, dev):
    d = golden("sgg.pt")["gsg"]
    ssd, seg = _seg_conditioned(golden, dev)
    sd = _srgan_sd(0)
    xt = torch.rand(d["mu"].shape, generator=torch.Generator().manual_seed(21)) * 2 - 1
    return d, ssd, seg, sd, _srgan(sd, dev), xt


def test_gsg_through_srgan_vs_oracle(golden):
    """One apply_gsg_through_srgan step against a per-image oracle (chain-rule gradient -> compute_gradient_magnitude ->
    update), compared on the guidance term alone x_t - (mu + sigma); criterion=per-image CE equals the fused call; the ratio of
    the through-SRGAN guidance magnitude to the pooled stand-in's is printed.  Measured on a B200 (1000 W): guidance term
    cosine 0.96389, rms-rel 0.267 (thresholds at 1.25x the error); criterion vs fused: rms-rel 0; magnitude ratio 0.270."""
    from oracle import deeplab
    from oracle.sgg import compute_gradient_magnitude
    from oracle.srgan import generator_forward
    from weatherconverter_b200.sgg.sgg import apply_gsg_batch, apply_gsg_through_srgan
    from weatherconverter_b200.srgan_model.inference import inference as srgan_inference
    dev = _dev()
    d, ssd, seg, sd, G, xt = _guidance_setup(golden, dev)
    mu, sigma, gt, lam = d["mu"], d["sigma"], d["gt"], d["lam"]
    got, aux = apply_gsg_through_srgan(seg, G, mu.to(dev), sigma.to(dev), xt.to(dev), gt.to(dev), lam, return_aux=True)
    with torch.no_grad():
        assert torch.equal(aux["sr"], srgan_inference(G, xt.to(dev)))
    refs = []
    for b in range(mu.shape[0]):
        xr = xt[b:b + 1].clone().requires_grad_(True)
        sr = generator_forward(sd, xr)
        _, g_sr, _ = deeplab.infer(ssd, sr.detach(), gt[b:b + 1])
        g_x, = torch.autograd.grad(sr, xr, g_sr)
        mag = compute_gradient_magnitude(g_x)
        refs.append((mu[b:b + 1].double() + lam * sigma[b:b + 1].double() * mag + sigma[b:b + 1].double()).float())
    ref = torch.cat(refs)
    base = mu + sigma
    term, term_ref = (got.cpu() - base).double(), (ref - base).double()
    cos, rel = _cos(term, term_ref), _rel(term, term_ref)
    print(f"apply_gsg_through_srgan vs oracle chain rule: guidance term cosine {cos:.5f} rms-rel {rel:.3e}")
    assert cos >= 0.955 and rel <= 0.334, (cos, rel)
    crit = apply_gsg_through_srgan(seg, G, mu.to(dev), sigma.to(dev), xt.to(dev), gt.to(dev), lam, criterion=per_image_ce)
    crel = _rel((crit.cpu() - base).double(), term)
    print(f"apply_gsg_through_srgan(criterion=per-image CE) vs fused: guidance-term rms-rel {crel:.3e}")
    assert crel <= 1e-2
    pooled = apply_gsg_batch(seg, mu.to(dev), sigma.to(dev), srgan_inference(G, xt.to(dev)), gt.to(dev), lam)
    pterm = (pooled.cpu() - base).double()
    ratio = float(term.norm() / pterm.norm())
    print(f"guidance magnitude, through-SRGAN / pooled stand-in: {ratio:.4f} "
          f"(mean |term| {float(term.abs().mean()):.3e} vs {float(pterm.abs().mean()):.3e})")
    assert 0 < ratio < float("inf")


def test_sample_with_sgg_grad_through_srgan(golden):
    from oracle.weights import synth_state_dict
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet, param_spec
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    from weatherconverter_b200.seg_model.network import modeling
    from weatherconverter_b200.translation import sample_with_sgg
    dev = _dev()
    d = golden("sgg.pt")["driver"]
    unet = Unet(d["cfg"]).to(dev).eval()
    unet.load_state_dict(synth_state_dict({k: (v, torch.float32) for k, v in param_spec(d["cfg"]).items()}, d["unet_seed"]))
    seg = modeling.deeplabv3plus_resnet50(19, 16, False)
    seg.load_state_dict(synth_state_dict(seg.state_dict(), d["seg_seed"]))
    seg = seg.to(dev).eval()
    G = _srgan(_srgan_sd(d["srgan_seed"]), dev)
    sched = LinearNoiseScheduler(1000, 1e-4, 0.02)
    kw = dict(n_steps=3, noise=d["noise"], t_forward=d["t_fwd"], step_noise=d["zs"])
    rec, base = [], []
    out = sample_with_sgg(d["x0"], unet, sched, seg, d["gt"], G, grad_through_srgan=True, record=rec, record_base=base, **kw)
    assert torch.isfinite(out).all()
    assert len(rec) == len(base) == 3
    for k in range(2):   # i = 2, 1: guided steps
        term = rec[k] - base[k]
        assert torch.isfinite(term).all() and float(term.abs().max()) > 0, k
    assert torch.equal(rec[2], base[2])   # i = 0: x_0 = mu, no guidance
    assert all(p.grad is None for p in G.parameters())
