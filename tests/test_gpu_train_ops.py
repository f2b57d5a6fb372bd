"""GPU parity tests of the training-step building blocks (backward kernels, Adam) against torch autograd on the same
bf16-rounded inputs.  Reference semantics: loss.backward() / optimizer.step() in diffusion_model/train_ddpm.py:108-113."""
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


@pytest.mark.parametrize("Cin,Cout,H,W,K,stride,dil,transposed,B,Cin2", [
    (64, 64, 16, 16, 3, 1, 1, False, 2, 0),       # narrow layer: half-empty M tile, 9 taps of one block
    (128, 256, 16, 32, 3, 1, 1, False, 1, 0),
    (128, 64, 16, 32, 3, 1, 1, False, 2, 192),    # fused 1x1 residual conv of a second input (unet_base.py:150)
    (256, 256, 8, 16, 1, 1, 1, False, 2, 0),      # linear / 1x1
    (64, 192, 16, 16, 1, 1, 1, False, 2, 0),      # in_proj-like (N = 3C)
    (128, 128, 16, 16, 4, 2, 1, False, 2, 0),     # down_sample_conv (unet_base.py:129)
    (128, 128, 8, 16, 4, 2, 1, True, 2, 0),       # up_sample_conv (ConvTranspose2d, unet_base.py:333)
    (768, 768, 16, 32, 3, 1, 1, False, 1, 0),
    (64, 64, 12, 20, 3, 1, 1, False, 2, 0),       # ragged tiles (zero-filled by TMA)
    (64, 64, 128, 256, 3, 1, 1, False, 1, 0),     # many pixel splits
])
def test_conv2d_wgrad(Cin, Cout, H, W, K, stride, dil, transposed, B, Cin2):
    from weatherconverter_b200 import ops
    dev = _dev()
    g = torch.Generator(device="cpu").manual_seed(Cin + Cout + H + K)
    x = _bf(torch.randn(B, Cin, H, W, generator=g)).to(dev)
    if transposed:
        w = torch.zeros(Cin, Cout, K, K, device=dev, requires_grad=True)
        y = F.conv_transpose2d(x, w, stride=2, padding=1)
        pad = 1
    else:
        pad = 1 if (stride == 2 and K > 1) else dil * (K - 1) // 2
        w = torch.zeros(Cout, Cin, K, K, device=dev, requires_grad=True)
        y = F.conv2d(x, w, stride=stride, padding=pad, dilation=dil)
    dy = _bf(torch.randn(y.shape, generator=g)).to(dev)
    x2 = w2 = None
    if Cin2:
        x2 = _bf(torch.randn(B, Cin2, H, W, generator=g)).to(dev)
        w2 = torch.zeros(Cout, Cin2, 1, 1, device=dev, requires_grad=True)
        y = y + F.conv2d(x2, w2)
    y.backward(dy)
    got = ops.conv2d_wgrad(ops.to_nhwc_bf16(x), ops.to_nhwc_bf16(dy), K, stride=stride, pad=pad, dil=dil, transposed=transposed,
                           x2=ops.to_nhwc_bf16(x2) if Cin2 else None)
    if Cin2:
        got, got2 = got
        assert _rel(got2, w2.grad) < 1e-4, _rel(got2, w2.grad)
    assert got.shape == w.grad.shape
    assert not torch.isnan(got).any()
    assert _rel(got, w.grad) < 1e-4, _rel(got, w.grad)     # same bf16 inputs, fp32 accumulation on both sides


def test_mse_boundary_adam():
    from weatherconverter_b200 import ops
    dev = _dev()
    g = torch.Generator(device="cpu").manual_seed(5)
    # MSE
    pred, tgt = torch.randn(2, 3, 32, 64, generator=g).to(dev), torch.randn(2, 3, 32, 64, generator=g).to(dev)
    pr = pred.clone().requires_grad_(True)
    ref = F.mse_loss(pr, tgt)
    ref.backward()
    loss, dpred = ops.mse_loss_grad(pred, tgt)
    assert abs(float(loss) - float(ref)) < 1e-6 * abs(float(ref)) + 1e-7
    assert _rel(dpred, pr.grad) < 1e-6
    # boundary convolutions: conv_in weight/bias gradient, conv_out weight/bias gradient
    B, H, W = 2, 24, 40
    img = torch.randn(B, 3, H, W, generator=g).to(dev)
    w_in = torch.zeros(64, 3, 3, 3, device=dev, requires_grad=True)
    b_in = torch.zeros(64, device=dev, requires_grad=True)
    dh = _bf(torch.randn(B, 64, H, W, generator=g)).to(dev)
    F.conv2d(img, w_in, b_in, padding=1).backward(dh)
    dw, db = ops.boundary_wgrad(ops.to_nhwc_bf16(dh), img, +1)
    assert _rel(dw, w_in.grad) < 1e-5 and _rel(db, b_in.grad) < 1e-5
    fin = _bf(torch.randn(B, 64, H, W, generator=g)).to(dev)
    w_out = torch.zeros(3, 64, 3, 3, device=dev, requires_grad=True)
    b_out = torch.zeros(3, device=dev, requires_grad=True)
    dp = torch.randn(B, 3, H, W, generator=g).to(dev)
    F.conv2d(fin, w_out, b_out, padding=1).backward(dp)
    dw, db = ops.boundary_wgrad(ops.to_nhwc_bf16(fin), dp, -1)
    assert _rel(dw, w_out.grad) < 1e-5 and _rel(db, b_out.grad) < 1e-5
    # Adam vs torch.optim.Adam over three steps
    p0 = torch.randn(100003, generator=g).to(dev)
    p_ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([p_ref], lr=1e-4)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    for step in range(1, 4):
        gr = torch.randn(100003, generator=g).to(dev) * 0.01
        p_ref.grad = gr.clone()
        opt.step()
        ops.adam_step(p, gr, m, v, 1e-4, 0.9, 0.999, 1e-8, step)
        # within a few fp32 ulps of the parameter (the update itself is ~1e-4; torch fuses some of the ops with FMA)
        assert bool(((p - p_ref.detach()).abs() <= 4.8e-7 * p.abs() + 1e-10).all()), step


@pytest.mark.parametrize("hd,N,B", [(64, 512, 2), (64, 256, 1), (16, 1024, 1), (32, 256, 2), (128, 512, 1), (192, 512, 1),
                                    (64, 64, 2), (32, 200, 1)])
def test_attention_bwd(hd, N, B):
    from weatherconverter_b200 import ops
    dev = _dev()
    heads = 4
    C = heads * hd
    g = torch.Generator(device="cpu").manual_seed(hd + N)
    q = _bf(torch.randn(B, heads, N, hd, generator=g)).to(dev).requires_grad_(True)
    k = _bf(torch.randn(B, heads, N, hd, generator=g)).to(dev).requires_grad_(True)
    v = _bf(torch.randn(B, heads, N, hd, generator=g)).to(dev).requires_grad_(True)
    d_o = _bf(torch.randn(B, N, C, generator=g)).to(dev)
    att = torch.softmax(q @ k.transpose(-2, -1) / math.sqrt(hd), dim=-1)
    ref = (att @ v).transpose(1, 2).reshape(B, N, C)
    ref.backward(d_o)
    qb, kb, vb = q.detach().bfloat16(), k.detach().bfloat16(), v.detach().bfloat16()
    o, lse = ops.attention_lse(qb, kb, vb.transpose(2, 3).contiguous())
    lse_ref = torch.logsumexp(q.detach() @ k.detach().transpose(-2, -1) / math.sqrt(hd), dim=-1) / math.log(2.0)
    assert float((lse - lse_ref.reshape(B * heads, N)).abs().max()) < 2e-2
    dqkv = ops.attention_bwd(qb, kb, vb, o, d_o.bfloat16(), lse).float()

    def heads_of(t):    # [B,N,C] -> [B,heads,N,hd]
        return t.reshape(B, N, heads, hd).permute(0, 2, 1, 3)
    dq, dk, dv = heads_of(dqkv[..., :C]), heads_of(dqkv[..., C:2 * C]), heads_of(dqkv[..., 2 * C:])
    assert _rel(dv, v.grad) < 1.5e-2, ("dv", _rel(dv, v.grad))
    assert _rel(dk, k.grad) < 2e-2, ("dk", _rel(dk, k.grad))
    assert _rel(dq, q.grad) < 2e-2, ("dq", _rel(dq, q.grad))
