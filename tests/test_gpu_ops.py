"""GPU parity tests of the op-level C ABI (run on the B200 box: pytest -m gpu)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda")


def _bf(x):
    return x.to(torch.bfloat16).float()


def _rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-20))


def test_ddpm_step_bit_exact(golden):
    from weatherconverter_b200 import ops
    from oracle.scheduler import OracleScheduler
    dev = _dev()
    g = golden("scheduler.pt")
    s = OracleScheduler(1000, 1e-4, 0.02)
    for ti, d in g["sample_prev_timestep"].items():
        z = d["z"].to(dev) if ti != 0 else None
        sigma = 0.0
        if ti != 0:
            var = (1 - s.alpha_cum_prod[ti - 1]) / (1.0 - s.alpha_cum_prod[ti]) * s.betas[ti]
            sigma = float(var ** 0.5)
        out, mean, sigz = ops.ddpm_step(g["x0"].to(dev), g["eps"].to(dev), z, float(s.betas[ti]),
                                        float(s.sqrt_one_minus_alpha_cum_prod[ti]), float(torch.sqrt(s.alphas[ti])),
                                        sigma, want_parts=True)
        assert torch.equal(mean.cpu(), d["mean"]), ti
        if ti != 0:
            assert torch.equal(sigz.cpu(), d["sigma_z"]), ti
            assert torch.equal(out.cpu(), d["mean"] + d["sigma_z"]), ti
        else:
            assert torch.equal(out.cpu(), d["mean"])


def test_layout_roundtrip():
    from weatherconverter_b200 import ops
    dev = _dev()
    x = torch.randn(2, 24, 5, 7, device=dev)
    y = ops.to_nchw_f32(ops.to_nhwc_bf16(x))
    assert torch.equal(y, _bf(x))


CONV_CASES = [
    # Cin, Cout, H, W, K, stride, dil, transposed, B
    (64, 64, 16, 16, 3, 1, 1, False, 2),
    (128, 256, 16, 32, 3, 1, 1, False, 1),
    (64, 128, 8, 8, 1, 1, 1, False, 4),
    (192, 64, 32, 32, 3, 1, 1, False, 1),      # K not a multiple of 64 per tap? (192 = 3 blocks)
    (304, 256, 16, 32, 3, 1, 1, False, 1),     # channel tail (304 = 4.75 blocks): TMA zero-fill in C
    (128, 128, 16, 16, 4, 2, 1, False, 2),     # down-sample conv
    (128, 128, 8, 16, 4, 2, 1, True, 2),       # up-sample transposed conv
    (256, 256, 16, 32, 3, 1, 6, False, 1),     # atrous
    (256, 256, 16, 32, 3, 1, 18, False, 1),    # atrous, halo larger than the map
    (64, 64, 128, 256, 3, 1, 1, False, 1),     # wide rows: 128 x 1 tiles
    (64, 16, 16, 16, 3, 1, 1, False, 1),       # narrow N tile
    (768, 768, 16, 32, 3, 1, 1, False, 1),     # deep K, N = 3 x 256
    (128, 128, 16, 16, 3, 2, 1, False, 1),     # 3x3 stride 2 (ResNet)
    (256, 512, 16, 16, 1, 2, 1, False, 1),     # 1x1 stride 2 (ResNet downsample)
    (64, 64, 12, 20, 3, 1, 1, False, 2),       # non power-of-two spatial dims (over-hanging tiles)
]


@pytest.mark.parametrize("Cin,Cout,H,W,K,stride,dil,transposed,B", CONV_CASES)
def test_conv2d(Cin, Cout, H, W, K, stride, dil, transposed, B):
    from weatherconverter_b200 import ops
    dev = _dev()
    g = torch.Generator(device="cpu").manual_seed(Cin * 7 + Cout + K)
    x = torch.randn(B, Cin, H, W, generator=g).to(dev)
    wshape = (Cin, Cout, K, K) if transposed else (Cout, Cin, K, K)
    w = (torch.randn(wshape, generator=g) / math.sqrt(Cin * K * K)).to(dev)
    b = (0.1 * torch.randn(Cout, generator=g)).to(dev)
    xh = ops.to_nhwc_bf16(x)
    if transposed:
        pad = 1
        ref = F.conv_transpose2d(_bf(x), _bf(w), b, stride=2, padding=1)
    else:
        pad = 1 if (stride == 2 and K > 1) else (0 if K == 1 else dil * (K - 1) // 2)
        ref = F.conv2d(_bf(x), _bf(w), b, stride=stride, padding=pad, dilation=dil)
    y = ops.to_nchw_f32(ops.conv2d(xh, w, b, stride=stride, pad=pad, dil=dil, transposed=transposed))
    assert y.shape == ref.shape
    err = _rel(y, ref)
    assert err < 5e-3, err


def test_conv2d_fused_epilogue():
    """3x3 conv + bias + t-emb row bias + fused 1x1 residual conv (ResNet sub-layer tail, unet_base.py:148-150)."""
    from weatherconverter_b200 import ops
    dev = _dev()
    g = torch.Generator(device="cpu").manual_seed(3)
    B, Cin, Cout, H, W = 2, 128, 64, 16, 32
    a = torch.randn(B, Cout, H, W, generator=g).to(dev)
    x = torch.randn(B, Cin, H, W, generator=g).to(dev)
    w = (torch.randn(Cout, Cout, 3, 3, generator=g) / math.sqrt(Cout * 9)).to(dev)
    w2 = (torch.randn(Cout, Cin, 1, 1, generator=g) / math.sqrt(Cin)).to(dev)
    b = (0.1 * torch.randn(Cout, generator=g)).to(dev)
    rb = torch.randn(B, Cout, generator=g).to(dev)
    res = torch.randn(B, Cout, H, W, generator=g).to(dev)
    y = ops.conv2d(ops.to_nhwc_bf16(a), w, b, rowbias=rb, residual=ops.to_nhwc_bf16(res), x2=ops.to_nhwc_bf16(x),
                   weight2=w2, relu=True)
    ref = F.conv2d(_bf(a), _bf(w), b, padding=1) + rb[:, :, None, None] + F.conv2d(_bf(x), _bf(w2)) + _bf(res)
    ref = F.relu(ref)
    assert _rel(ops.to_nchw_f32(y), ref) < 5e-3


@pytest.mark.parametrize("Cin,Cout,H,W", [(768, 768, 16, 32), (256, 256, 64, 128), (512, 512, 32, 64), (128, 128, 64, 128)])
def test_conv1x1_residual_many_tiles_per_cta(Cin, Cout, H, W):
    """1x1 convolution + residual with several tiles per persistent CTA (the epilogue is the bottleneck there): regression
    test of the cross-proxy WAR race on the TMA residual staging buffer (generic-proxy reads vs the next TMA box), which
    corrupted a few per cent of the rows of SOME images at batch >= 3 in round 1.  Every image is checked on its own,
    three times (the race was timing dependent)."""
    from weatherconverter_b200 import ops
    dev = _dev()
    for B in (3, 5, 16, 32):
        g = torch.Generator(device="cpu").manual_seed(Cin + B)
        x = torch.randn(B, Cin, H, W, generator=g).to(dev)
        w = (torch.randn(Cout, Cin, 1, 1, generator=g) / math.sqrt(Cin)).to(dev)
        b = (0.1 * torch.randn(Cout, generator=g)).to(dev)
        res = torch.randn(B, Cout, H, W, generator=g).to(dev)
        ref = F.conv2d(_bf(x), _bf(w), b) + _bf(res)
        xh, rh = ops.to_nhwc_bf16(x), ops.to_nhwc_bf16(res)
        first = None
        for rep in range(3):
            y = ops.to_nchw_f32(ops.conv2d(xh, w, b, residual=rh))
            worst = max(_rel(y[i], ref[i]) for i in range(B))
            assert worst < 5e-3, (B, rep, worst)
            first = y if first is None else first
            assert torch.equal(y, first), (B, rep)


def test_conv_in_out():
    from weatherconverter_b200 import ops
    dev = _dev()
    g = torch.Generator(device="cpu").manual_seed(9)
    x = torch.randn(2, 3, 32, 64, generator=g).to(dev)
    w = (torch.randn(64, 3, 3, 3, generator=g) / math.sqrt(27)).to(dev)
    b = (0.1 * torch.randn(64, generator=g)).to(dev)
    y = ops.to_nchw_f32(ops.conv_in(x, w, b))
    ref = F.conv2d(x, w, b, padding=1)
    assert _rel(y, ref) < 4e-3
    w7 = (torch.randn(64, 3, 7, 7, generator=g) / math.sqrt(147)).to(dev)
    sc, sh = (1 + 0.1 * torch.randn(64, generator=g)).to(dev), (0.1 * torch.randn(64, generator=g)).to(dev)
    y = ops.to_nchw_f32(ops.conv_in(x, w7, None, sc, sh, stride=2, pad=3, relu=True))
    ref = F.relu(F.conv2d(x, w7, None, stride=2, padding=3) * sc[None, :, None, None] + sh[None, :, None, None])
    assert _rel(y, ref) < 4e-3
    h = torch.randn(2, 64, 32, 64, generator=g).to(dev)
    wo = (torch.randn(3, 64, 3, 3, generator=g) / math.sqrt(576)).to(dev)
    bo = (0.1 * torch.randn(3, generator=g)).to(dev)
    y = ops.conv_out(ops.to_nhwc_bf16(h), wo, bo)
    ref = F.conv2d(_bf(h), wo, bo, padding=1)
    assert _rel(y, ref) < 1e-4


@pytest.mark.parametrize("hd,N,B", [(64, 512, 2), (16, 1024, 1), (32, 256, 2), (128, 512, 1), (192, 512, 1),
                                    (64, 64, 2), (64, 2048, 1), (32, 200, 1)])
def test_attention(hd, N, B):
    from weatherconverter_b200 import ops
    dev = _dev()
    heads = 4
    g = torch.Generator(device="cpu").manual_seed(hd + N)
    q = torch.randn(B, heads, N, hd, generator=g).to(dev) * 1.5
    k = torch.randn(B, heads, N, hd, generator=g).to(dev) * 1.5
    v = torch.randn(B, heads, N, hd, generator=g).to(dev)
    o = ops.attention(q.bfloat16(), k.bfloat16(), v.transpose(2, 3).contiguous().bfloat16()).float()
    att = torch.softmax(_bf(q) @ _bf(k).transpose(-2, -1) / math.sqrt(hd), dim=-1)
    ref = (att @ _bf(v)).transpose(1, 2).reshape(B, N, heads * hd)
    err = _rel(o, ref)
    assert err < 1e-2, err


@pytest.mark.parametrize("hd,N,B,mode", [(16, 1024, 1, "grow"), (32, 1024, 1, "grow"), (16, 520, 2, "grow"), (32, 136, 1, "grow"),
                                          (16, 1024, 1, "big"), (32, 512, 1, "big"), (16, 384, 1, "shrink"),
                                          (16, 8192, 1, "plain"), (32, 8192, 1, "plain")])
def test_attention_small_heads_stale_max(hd, N, B, mode):
    """head_dim 16/32 kernel (csrc/attention_small.cu): the row maximum is tracked lazily (stale offset folded into the S
    accumulator, overflow detection on the packed P words).  Inputs whose row maximum keeps growing from one KV tile to the
    next by far more than the 2^9 slack, very large logits, maxima that only occur in the first tile, and ragged N must all
    match softmax(QK^T/sqrt(hd))V; the log-sum-exp rows saved for the backward are checked too."""
    from weatherconverter_b200 import ops
    dev = _dev()
    heads = 4
    g = torch.Generator(device="cpu").manual_seed(7 * hd + N)
    q = torch.randn(B, heads, N, hd, generator=g)
    k = torch.randn(B, heads, N, hd, generator=g)
    v = torch.randn(B, heads, N, hd, generator=g)
    if mode == "grow":      # key norms grow with the index: every later tile raises the row maximum
        k = k * torch.linspace(0.25, 14.0, N)[None, None, :, None]
    elif mode == "big":     # logits of several hundred (log2 units)
        q, k = q * 6.0, k * 6.0
    elif mode == "shrink":  # the largest logits are all in the first tile, later ones are far below
        k = k * torch.linspace(14.0, 0.05, N)[None, None, :, None]
    q, k, v = q.to(dev), k.to(dev), v.to(dev)
    o, lse = ops.attention_lse(q.bfloat16(), k.bfloat16(), v.transpose(2, 3).contiguous().bfloat16())
    o2 = ops.attention(q.bfloat16(), k.bfloat16(), v.transpose(2, 3).contiguous().bfloat16())
    assert torch.equal(o, o2)
    s = (_bf(q).double() @ _bf(k).double().transpose(-2, -1)) / math.sqrt(hd)
    att = torch.softmax(s, dim=-1)
    ref = (att @ _bf(v).double()).transpose(1, 2).reshape(B, N, heads * hd).float()
    err = _rel(o.float(), ref)
    assert torch.isfinite(o.float()).all()
    assert err < 1e-2, err
    lse_ref = (torch.logsumexp(s, dim=-1) * math.log2(math.e)).reshape(B * heads, N).float()
    # l is summed from bf16-rounded P: relative error <= 2^-9 per term -> absolute log2 error of a few 1e-3
    assert (lse - lse_ref).abs().max() < 2e-2 + 1e-5 * lse_ref.abs().max(), float((lse - lse_ref).abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("hd,N,B,mode", [(16, 8192, 1, "plain"), (16, 2048, 2, "grow"), (16, 2504, 1, "big"), (16, 1024, 1, "grow"),
                                          (32, 2048, 1, "plain"), (64, 1024, 1, "plain"), (128, 512, 1, "plain")])
def test_attention_prescaled_q(hd, N, B, mode):
    """scale < 0 (csrc/wc_host.h: kAttnScalePrescaled): Q already carries log2(e)/sqrt(hd) - what the UNet plan's QKV projection
    stores - and every attention kernel runs with a unit log2-domain scale (head_dim 16, N >= 2048: the UNIT variant of
    attention_small4_kernel without the per-logit multiply).  Reference: softmax over ln(2) * (q' . k) in float64."""
    from weatherconverter_b200 import ops
    dev = _dev()
    heads = 4
    g = torch.Generator(device="cpu").manual_seed(11 * hd + N)
    q = torch.randn(B, heads, N, hd, generator=g)
    k = torch.randn(B, heads, N, hd, generator=g)
    v = torch.randn(B, heads, N, hd, generator=g)
    if mode == "grow":
        k = k * torch.linspace(0.25, 14.0, N)[None, None, :, None]
    elif mode == "big":
        q, k = q * 6.0, k * 6.0
    qp = (q * (math.log2(math.e) / math.sqrt(hd))).to(dev).bfloat16()
    k, v = k.to(dev), v.to(dev)
    o = ops.attention(qp, k.bfloat16(), v.transpose(2, 3).contiguous().bfloat16(), scale=-1.0)
    s = (qp.double() @ _bf(k).double().transpose(-2, -1)) * math.log(2.0)
    ref = (torch.softmax(s, dim=-1) @ _bf(v).double()).transpose(1, 2).reshape(B, N, heads * hd).float()
    assert torch.isfinite(o.float()).all()
    err = _rel(o.float(), ref)
    assert err < 1e-2, err
