"""GPU tests of the differentiable DeepLabV3+ (torch autograd through wc_seg_forward / wc_seg_backward_seeded): logits
bit-identical to the fused plan, CE through autograd against the fused infer gradient, an arbitrary loss against torch
autograd through the fp32 oracle, both output strides and both backbones, the plan pool's lifetime rules, and guidance
with a custom criterion."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda")


def _seg(backbone, seed, dev, output_stride=16, bn3_gain=None):
    from oracle.weights import synth_state_dict
    from weatherconverter_b200.seg_model.network import modeling
    m = getattr(modeling, "deeplabv3plus_" + backbone)(num_classes=19, output_stride=output_stride, pretrained_backbone=False)
    sd = synth_state_dict(m.state_dict(), seed)
    if bn3_gain is not None:
        for k in sd:
            if k.endswith("bn3.weight"):
                sd[k] = sd[k] * bn3_gain
    m.load_state_dict(sd)
    return sd, m.to(dev).eval()


def _rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-20))


def _cos(a, b):
    return float(F.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0))


def per_image_ce(logits, gt):
    """CE(ignore 255) averaged over each image's own valid pixels: [B] (the fused plan's loss)."""
    ce = F.cross_entropy(logits, gt, ignore_index=255, reduction="none")
    n = (gt != 255).flatten(1).sum(1).clamp_min(1)
    return ce.flatten(1).sum(1) / n


def mixed_loss(logits, gt):
    """Class-weighted CE + entropy over EVERY pixel (label 255 included) + squared logits on a strided slice: [B]."""
    w = torch.linspace(0.5, 2.0, logits.shape[1], device=logits.device, dtype=logits.dtype)
    ce = torch.stack([F.cross_entropy(logits[b:b + 1], gt[b:b + 1], weight=w, ignore_index=255) for b in range(logits.shape[0])])
    logp = logits.log_softmax(1)
    ent = -(logp.exp() * logp).sum(1).mean((1, 2))
    sq = logits[:, :, ::2, ::3].pow(2).mean((1, 2, 3))
    return ce + 0.5 * ent + 0.05 * sq


def _autograd_grad(m, x, gt, loss_fn=per_image_ce):
    xg = x.clone().requires_grad_(True)
    loss = loss_fn(m(xg), gt).sum()
    loss.backward()
    return xg.grad


def test_autograd_logits_are_the_fused_plan_bits(golden):
    """Both R50 goldens: logits of the autograd forward == infer(want_logits=True) == the non-grad forward, bit for bit."""
    dev = _dev()
    g = golden("seg_infer.pt")
    for tag in ("resnet50_64x128", "resnet50_128x256"):
        d = g[tag]
        _, m = _seg("resnet50", d["seed"], dev)
        x, gt = d["x"].to(dev), d["gt"].to(dev)
        ref = m.infer(x, gt, want_grad=True, want_logits=True)["logits"]
        with torch.no_grad():
            plain = m(x)
        assert plain.grad_fn is None
        xg = x.clone().requires_grad_(True)
        lg = m(xg)
        assert lg.grad_fn is not None
        assert torch.equal(lg.detach(), ref), tag
        assert torch.equal(plain, ref), tag
        assert torch.equal(m(x), ref), tag             # x without requires_grad: no graph, same bits


def test_ce_through_autograd_equals_fused_infer(golden):
    """Per-image CE(ignore 255) through autograd vs the fused loss head's gradient.  The forward is identical and the backward
    is linear in its seed, so only the rounding of the low-resolution d-logits differs.  Measured on a B200 (1000 W): the
    gradients were bit-identical on both fixtures (rms-rel 0); the losses agree to 1.6e-7."""
    dev = _dev()
    cases = []
    dc = golden("seg_conditioned.pt")
    cases.append(("conditioned", _seg("resnet50", dc["seed"], dev, bn3_gain=dc["bn3_gain"])[1], dc["x"], dc["gt"]))
    d = golden("seg_infer.pt")["resnet50_64x128"]
    cases.append(("resnet50_64x128", _seg("resnet50", d["seed"], dev)[1], d["x"], d["gt"]))
    for tag, m, x, gt in cases:
        x, gt = x.to(dev), gt.to(dev)
        fused = m.infer(x, gt)
        xg = x.clone().requires_grad_(True)
        loss = per_image_ce(m(xg), gt)
        loss.sum().backward()
        rel, cos = _rel(xg.grad, fused["grad"]), _cos(xg.grad, fused["grad"])
        lrel = _rel(loss.detach(), fused["loss"])
        print(f"{tag}: CE through autograd vs fused infer: grad rms-rel {rel:.3e} cosine {cos:.7f}; loss rel {lrel:.2e}")
        assert lrel < 1e-4, (tag, lrel)
        assert rel <= 1e-2 and cos >= 0.9999, (tag, rel, cos)


def test_arbitrary_loss_vs_oracle_autograd(golden):
    """Class-weighted CE + entropy over every pixel (ignored ones too) + squared logits on a strided slice, both images of the
    conditioned fixture, against torch autograd through the fp32 oracle (thresholds of the fused path on this fixture).
    Measured on a B200 (1000 W): cosine 0.9932 / 0.9930, rms-rel 0.116 / 0.119."""
    from oracle import deeplab
    dev = _dev()
    d = golden("seg_conditioned.pt")
    sd, m = _seg("resnet50", d["seed"], dev, bn3_gain=d["bn3_gain"])
    assert bool((d["gt"] == 255).any()), "the fixture must contain ignored pixels"
    grad = _autograd_grad(m, d["x"].to(dev), d["gt"].to(dev), mixed_loss).cpu()
    xr = d["x"].clone().requires_grad_(True)
    mixed_loss(deeplab.deeplab_forward(sd, xr, "resnet50"), d["gt"]).sum().backward()
    for b in range(d["x"].shape[0]):
        rel, cos = _rel(grad[b], xr.grad[b]), _cos(grad[b], xr.grad[b])
        print(f"mixed loss, conditioned image {b}: CUDA autograd vs fp32 oracle autograd: cosine {cos:.5f} rms-rel {rel:.3e}")
        assert cos >= 0.99 and rel <= 0.15, (b, cos, rel)


def test_output_stride_8_and_resnet101(golden):
    """CE through autograd vs the reference's gradient for R50 output stride 8 and R101 output stride 16 at 64x128, with the
    thresholds of test_gpu_seg.py for those fixtures.  Measured on a B200 (1000 W): os8 cosine 0.982 / rms-rel 0.19, R101
    cosine 0.971 / rms-rel 0.24."""
    dev = _dev()
    d8 = golden("seg_infer_os8.pt")["resnet50_os8_64x128"]
    d101 = golden("seg_infer.pt")["resnet101_64x128"]
    for tag, bb, os_, d in (("resnet50_os8", "resnet50", 8, d8), ("resnet101_os16", "resnet101", 16, d101)):
        _, m = _seg(bb, d["seed"], dev, output_stride=os_)
        grad = _autograd_grad(m, d["x"].to(dev), d["gt"].to(dev)).cpu()
        rel, cos = _rel(grad, d["grad"]), _cos(grad, d["grad"])
        print(f"{tag}: CE through autograd vs fp32 golden: cosine {cos:.5f} rms-rel {rel:.3e}")
        assert cos > 0.96 and rel < 0.30, (tag, cos, rel)


def test_graph_hygiene(golden):
    from weatherconverter_b200.seg_model.network import modeling
    dev = _dev()
    d = golden("seg_infer.pt")["resnet50_64x128"]
    _, m = _seg("resnet50", d["seed"], dev)
    x1, gt = d["x"].to(dev), d["gt"].to(dev)
    x2 = x1.flip(-1).contiguous()
    key = tuple([x1.shape[0]] + list(x1.shape[2:]))
    alone1, alone2 = _autograd_grad(m, x1, gt), _autograd_grad(m, x2, gt)
    # two live graphs, backpropagated in reverse order
    a, b = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    la, lb = per_image_ce(m(a), gt).sum(), per_image_ce(m(b), gt).sum()
    assert len(m._grad_plans[key]) == 2
    lb.backward()
    la.backward()
    assert torch.equal(a.grad, alone1) and torch.equal(b.grad, alone2)
    # torch.autograd.grad
    xg = x1.clone().requires_grad_(True)
    gx, = torch.autograd.grad(per_image_ce(m(xg), gt).sum(), xg)
    assert torch.equal(gx, alone1)
    # a non-contiguous incoming gradient gives the bits of its contiguous copy
    seed = torch.randn(1, 19, x1.shape[3], x1.shape[2], device=dev).transpose(2, 3)
    assert not seed.is_contiguous()
    xa, xb = x1.clone().requires_grad_(True), x1.clone().requires_grad_(True)
    m(xa).backward(seed)
    m(xb).backward(seed.contiguous())
    assert torch.equal(xa.grad, xb.grad)
    # a second backward through the same graph raises
    xg = x1.clone().requires_grad_(True)
    loss = per_image_ce(m(xg), gt).sum()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already been backpropagated"):
        loss.backward()
    # the parameters are constants
    assert all(p.grad is None for p in m.parameters())
    # the pool does not grow, and memory is constant across iterations
    del a, b, la, lb, xa, xb, xg, loss
    mem = []
    for _ in range(10):
        xg = x1.clone().requires_grad_(True)
        per_image_ce(m(xg), gt).sum().backward()
        del xg
        torch.cuda.synchronize()
        mem.append(torch.cuda.memory_allocated())
        assert len(m._grad_plans[key]) == 2
    assert len(set(mem)) == 1, mem
    # CPU input and train mode raise
    with pytest.raises(RuntimeError):
        m(d["x"].clone().requires_grad_(True))
    m.train()
    try:
        with pytest.raises(RuntimeError, match="eval"):
            m(x1.clone().requires_grad_(True))
    finally:
        m.eval()
    assert isinstance(m, modeling.DeepLabV3)


def test_inplace_weight_change_rebuilds_the_pool(golden):
    """load_state_dict copies into the same storage: the autograd path must see the new weights."""
    from oracle.weights import synth_state_dict
    dev = _dev()
    d = golden("seg_infer.pt")["resnet50_64x128"]
    _, m = _seg("resnet50", d["seed"], dev)
    x, gt = d["x"].to(dev), d["gt"].to(dev)
    before = m(x.clone().requires_grad_(True)).detach()
    ptrs = [p.data_ptr() for p in m.parameters()]
    m.load_state_dict(synth_state_dict(m.state_dict(), d["seed"] + 1))
    assert ptrs == [p.data_ptr() for p in m.parameters()]
    after = m(x.clone().requires_grad_(True)).detach()
    ref = m.infer(x, gt, want_grad=False, want_logits=True)["logits"]
    assert not torch.equal(after, before)
    assert torch.equal(after, ref)


def test_gsg_with_custom_criterion(golden):
    from weatherconverter_b200.sgg.sgg import apply_gsg_batch
    dev = _dev()
    d = golden("sgg.pt")["gsg"]
    _, m = _seg("resnet50", 42, dev)
    mu, sigma, sr_xt, gt = (d[k].to(dev) for k in ("mu", "sigma", "sr_xt", "gt"))
    ref = apply_gsg_batch(m, mu, sigma, sr_xt, gt, d["lam"])
    got = apply_gsg_batch(m, mu, sigma, sr_xt, gt, d["lam"], criterion=per_image_ce)
    base = mu + sigma
    rel = _rel(got - base, ref - base)
    print(f"apply_gsg_batch(criterion=per-image CE) vs fused: guidance-term rms-rel {rel:.3e}")   # B200: 0 (same bits)
    assert rel <= 1e-2
    with pytest.raises(ValueError, match="one loss per image"):
        apply_gsg_batch(m, mu, sigma, sr_xt, gt, d["lam"], criterion=lambda lg, g: F.cross_entropy(lg, g, ignore_index=255))


def test_sample_with_sgg_custom_criterion(golden):
    from oracle.weights import synth_state_dict
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet, param_spec
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    from weatherconverter_b200.srgan_model.models import Generator
    from weatherconverter_b200.translation import sample_with_sgg
    dev = _dev()
    d = golden("sgg.pt")["driver"]
    unet = Unet(d["cfg"]).to(dev).eval()
    unet.load_state_dict(synth_state_dict({k: (v, torch.float32) for k, v in param_spec(d["cfg"]).items()}, d["unet_seed"]))
    _, seg = _seg("resnet50", d["seg_seed"], dev)
    G = Generator(upscale_factor=4)
    G.load_state_dict(synth_state_dict(G.state_dict(), d["srgan_seed"]))
    G = G.to(dev).eval()
    sched = LinearNoiseScheduler(1000, 1e-4, 0.02)
    kw = dict(n_steps=3, noise=d["noise"], t_forward=d["t_fwd"], step_noise=d["zs"])
    default = sample_with_sgg(d["x0"], unet, sched, seg, d["gt"], G, **kw)
    custom = sample_with_sgg(d["x0"], unet, sched, seg, d["gt"], G, criterion=mixed_loss, **kw)
    assert torch.isfinite(custom).all()
    assert not torch.equal(custom, default)
    for bad in (dict(use_graph=True), dict(mode="lcg")):
        with pytest.raises(ValueError):
            sample_with_sgg(d["x0"], unet, sched, seg, d["gt"], G, criterion=mixed_loss, **kw, **bad)
