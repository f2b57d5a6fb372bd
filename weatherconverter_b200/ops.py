"""Op-level Python wrappers over the C ABI (torch tensors in, torch tensors out).

PyTorch is used only to own device memory and streams; all arithmetic happens inside libwc_b200.so.
Activation tensors at this level are NHWC bf16 (``[B,H,W,C]``, contiguous or channel-sliced views).
"""
import torch

from . import _lib
from ._lib import check, lib, ptr, require_cuda, stream_ptr


def to_nhwc_bf16(x: torch.Tensor) -> torch.Tensor:
    """[B,C,H,W] fp32 (reference layout) -> [B,H,W,C] bf16."""
    require_cuda(x)
    x = x.contiguous().float()
    B, Cc, H, W = x.shape
    y = torch.empty(B, H, W, Cc, device=x.device, dtype=torch.bfloat16)
    check(lib().wc_nchw_f32_to_nhwc_bf16(ptr(x), ptr(y), B, Cc, H * W, Cc, stream_ptr()))
    return y


def to_nchw_f32(x: torch.Tensor) -> torch.Tensor:
    """[B,H,W,C] bf16 -> [B,C,H,W] fp32."""
    require_cuda(x)
    B, H, W, Cc = x.shape
    assert x.stride(3) == 1 and x.stride(1) == W * x.stride(2) and x.stride(0) == H * x.stride(1)
    y = torch.empty(B, Cc, H, W, device=x.device, dtype=torch.float32)
    check(lib().wc_nhwc_bf16_to_nchw_f32(ptr(x), ptr(y), B, Cc, H * W, x.stride(2), stream_ptr()))
    return y


def groupnorm_silu(x, gamma, beta, silu=True, eps=1e-5):
    require_cuda(x, gamma, beta)
    B, H, W, Cc = x.shape
    y = torch.empty(B, H, W, Cc, device=x.device, dtype=torch.bfloat16)
    ws = torch.empty(lib().wc_groupnorm_workspace_bytes(B), device=x.device, dtype=torch.uint8)
    check(lib().wc_groupnorm_silu(ptr(x), ptr(y), B, H * W, Cc, pixel_stride(x), Cc, ptr(gamma), ptr(beta), eps,
                                  1 if silu else 0, ptr(ws), stream_ptr()))
    return y


def conv2d(x, weight, bias=None, stride=1, pad=None, dil=1, transposed=False, rowbias=None, residual=None,
           x2=None, weight2=None, relu=False):
    """x [B,H,W,Cin] bf16; weight fp32 PyTorch layout; returns [B,Ho,Wo,Cout] bf16."""
    require_cuda(x, weight)
    B, H, W, Cin = x.shape
    K = weight.shape[-1]
    Cout = weight.shape[1] if transposed else weight.shape[0]
    if pad is None:
        pad = dil * (K - 1) // 2
    Ho, Wo = (2 * H, 2 * W) if transposed else ((H // 2, W // 2) if stride == 2 else (H, W))
    y = torch.empty(B, Ho, Wo, Cout, device=x.device, dtype=torch.bfloat16)
    weight = weight.contiguous().float()
    if weight2 is not None:
        weight2 = weight2.contiguous().float()
    check(lib().wc_conv2d(ptr(x), B, H, W, Cin, x.stride(2), ptr(weight), ptr(bias), Cout, K, stride, pad, dil,
                          1 if transposed else 0, ptr(rowbias), ptr(residual),
                          residual.stride(2) if residual is not None else 0,
                          ptr(x2), x2.shape[3] if x2 is not None else 0, x2.stride(2) if x2 is not None else 0,
                          ptr(weight2), 1 if relu else 0, ptr(y), Cout, stream_ptr()))
    return y


def conv_in(x, weight, bias=None, scale=None, shift=None, stride=1, pad=None, relu=False):
    """Boundary conv from the reference layout: x [B,3,H,W] fp32 -> [B,Ho,Wo,Cout] bf16."""
    require_cuda(x, weight)
    B, Cc, H, W = x.shape
    Cout, _, K, _ = weight.shape
    if pad is None:
        pad = K // 2
    Ho, Wo = (H + 2 * pad - K) // stride + 1, (W + 2 * pad - K) // stride + 1
    y = torch.empty(B, Ho, Wo, Cout, device=x.device, dtype=torch.bfloat16)
    x, weight = x.contiguous(), weight.contiguous()    # named: must outlive the raw-pointer call
    check(lib().wc_conv_in(ptr(x), ptr(weight), ptr(bias), ptr(scale), ptr(shift), ptr(y),
                           B, H, W, Cout, K, stride, pad, Cout, 1 if relu else 0, stream_ptr()))
    return y


def conv_out(x, weight, bias=None, tanh_out=False):
    """Boundary conv to the reference layout: x [B,H,W,Cin] bf16 -> [B,3,H,W] fp32."""
    require_cuda(x, weight)
    B, H, W, Cin = x.shape
    K = weight.shape[-1]
    y = torch.empty(B, 3, H, W, device=x.device, dtype=torch.float32)
    weight = weight.contiguous()
    check(lib().wc_conv_out(ptr(x), ptr(weight), ptr(bias), ptr(y), B, H, W, Cin, K, x.stride(2),
                            1 if tanh_out else 0, stream_ptr()))
    return y


def attention(q, k, vt, scale=0.0):
    """q,k [B,heads,N,hd] bf16; vt [B,heads,hd,N] bf16 -> [B,N,heads*hd] bf16.  scale > 0: explicit softmax scale; 0: 1/sqrt(hd);
    < 0: q already carries log2(e)/sqrt(hd) (the UNet plan's QKV projection), the kernels run with a unit log2-domain scale."""
    require_cuda(q, k, vt)
    B, h, N, hd = q.shape
    out = torch.empty(B, N, h * hd, device=q.device, dtype=torch.bfloat16)
    q, k, vt = q.contiguous(), k.contiguous(), vt.contiguous()
    if scale == 0.0:
        check(lib().wc_attention(ptr(q), ptr(k), ptr(vt), ptr(out), B, h, N, hd, h * hd, stream_ptr()))
    else:
        check(lib().wc_attention_scaled(ptr(q), ptr(k), ptr(vt), ptr(out), B, h, N, hd, h * hd, float(scale), stream_ptr()))
    return out


def ddpm_step(xt, eps, z, beta, sqrt_one_minus_acp, sqrt_alpha, sigma, want_parts=False):
    """Fused posterior update; returns x_{t-1} (and (mean, sigma*z) when want_parts)."""
    require_cuda(xt, eps, z)
    xt, eps = xt.contiguous(), eps.contiguous()
    B = xt.shape[0]
    n = xt[0].numel()
    out = torch.empty_like(xt)
    mean = torch.empty_like(xt) if want_parts else None
    sigz = torch.empty_like(xt) if (want_parts and z is not None) else None
    z = z.contiguous() if z is not None else None
    check(lib().wc_ddpm_step(ptr(xt), ptr(eps), ptr(z), ptr(out), ptr(mean),
                             ptr(sigz), n, B, float(beta), float(sqrt_one_minus_acp), float(sqrt_alpha), float(sigma),
                             stream_ptr()))
    return (out, mean, sigz) if want_parts else out


def launch_count() -> int:
    return int(lib().wc_launch_count())


# ---------------------------------------------------------------------------------------------------------
# training-step building blocks (diffusion_model/train_ddpm.py:95-114)
def attention_lse(q, k, vt):
    """attention() that also returns the log2-domain log-sum-exp rows [B*heads, N] (saved for the backward)."""
    require_cuda(q, k, vt)
    B, h, N, hd = q.shape
    out = torch.empty(B, N, h * hd, device=q.device, dtype=torch.bfloat16)
    lse = torch.empty(B * h, N, device=q.device, dtype=torch.float32)
    q, k, vt = q.contiguous(), k.contiguous(), vt.contiguous()
    check(lib().wc_attention_lse(ptr(q), ptr(k), ptr(vt), ptr(out), ptr(lse), B, h, N, hd, h * hd, stream_ptr()))
    return out, lse


def attention_bwd(q, k, v, o, d_o, lse):
    """q,k,v [B,heads,N,hd] bf16; o, d_o [B,N,C] bf16 -> dqkv [B,N,3C] bf16 (dQ | dK | dV)."""
    require_cuda(q, k, v, o, d_o, lse)
    B, h, N, hd = q.shape
    q, k, v, o, d_o = q.contiguous(), k.contiguous(), v.contiguous(), o.contiguous(), d_o.contiguous()
    dqkv = torch.zeros(B, N, 3 * h * hd, device=q.device, dtype=torch.bfloat16)
    scratch = torch.empty(B * h * N, device=q.device, dtype=torch.float32)
    check(lib().wc_attention_bwd(ptr(q), ptr(k), ptr(v), ptr(o), ptr(d_o), ptr(lse), ptr(scratch), ptr(dqkv), B, h, N, hd,
                                 stream_ptr()))
    return dqkv


def conv2d_wgrad(x, dy, K, stride=1, pad=None, dil=1, transposed=False, x2=None):
    """Weight gradient: x [B,H,W,Cin] bf16, dy [B,Ho,Wo,Cout] bf16 -> dw fp32 (PyTorch layout) [, dw2]."""
    require_cuda(x, dy)
    B, H, W, Cin = x.shape
    Cout = dy.shape[3]
    if pad is None:
        pad = dil * (K - 1) // 2
    x, dy = x.contiguous(), dy.contiguous()
    shape = (Cin, Cout, K, K) if transposed else (Cout, Cin, K, K)
    dw = torch.full(shape, float("nan"), device=x.device, dtype=torch.float32)
    dw2 = None
    if x2 is not None:
        x2 = x2.contiguous()
        dw2 = torch.full((Cout, x2.shape[3], 1, 1), float("nan"), device=x.device, dtype=torch.float32)
    check(lib().wc_conv2d_wgrad(ptr(x), ptr(dy), B, H, W, Cin, Cout, K, stride, pad, dil, 1 if transposed else 0,
                                ptr(x2), x2.shape[3] if x2 is not None else 0, ptr(dw), ptr(dw2), stream_ptr()))
    return (dw, dw2) if x2 is not None else dw


def pixel_stride(x):
    """Pixel stride (elements) of an NHWC view [B,H,W,C] whose pixels are evenly spaced: a contiguous tensor or a channel slice
    of a wider one."""
    B, H, W, Cc = x.shape
    assert x.stride(3) == 1 and x.stride(1) == W * x.stride(2) and x.stride(0) == H * x.stride(1), x.stride()
    return x.stride(2)


def groupnorm_silu_fwd_bwd(x, gamma, beta, dy, silu=True, eps=1e-5, add1=None, add2=None):
    """Forward + backward of GroupNorm(8)[+SiLU]; returns (y, dx, dgamma, dbeta).  x, dy, add1, add2 may be channel slices."""
    require_cuda(x, gamma, beta, dy)
    B, H, W, Cc = x.shape
    y = torch.empty(B, H, W, Cc, device=x.device, dtype=torch.bfloat16)
    ws = torch.empty(lib().wc_groupnorm_workspace_bytes(B), device=x.device, dtype=torch.uint8)
    check(lib().wc_groupnorm_silu(ptr(x), ptr(y), B, H * W, Cc, pixel_stride(x), Cc, ptr(gamma), ptr(beta), eps, 1 if silu else 0,
                                  ptr(ws), stream_ptr()))
    dx = torch.empty_like(y)
    dg = torch.empty(Cc, device=x.device, dtype=torch.float32)
    db = torch.empty(Cc, device=x.device, dtype=torch.float32)
    ws2 = torch.empty(lib().wc_groupnorm_bwd_workspace_bytes(B, Cc), device=x.device, dtype=torch.uint8)
    lda1 = pixel_stride(add1) if add1 is not None else 8
    lda2 = pixel_stride(add2) if add2 is not None else 8
    check(lib().wc_groupnorm_silu_bwd(ptr(x), ptr(dy), ptr(dx), B, H * W, Cc, pixel_stride(x), pixel_stride(dy), Cc, ptr(gamma),
                                      ptr(beta), eps, 1 if silu else 0, ptr(ws), ptr(add1), lda1, ptr(add2), lda2, ptr(dg), ptr(db),
                                      ptr(ws2), stream_ptr()))
    return y, dx, dg, db


def colsum(x):
    """x [B,H,W,C] bf16 (may be a channel slice) -> (per-sample sums [B,C] fp32, total [C] fp32)."""
    require_cuda(x)
    B, H, W, Cc = x.shape
    rows = torch.empty(B, Cc, device=x.device, dtype=torch.float32)
    tot = torch.empty(Cc, device=x.device, dtype=torch.float32)
    ws = torch.empty(lib().wc_groupnorm_bwd_workspace_bytes(B, Cc), device=x.device, dtype=torch.uint8)
    check(lib().wc_colsum(ptr(x), B, H * W, Cc, pixel_stride(x), ptr(rows), Cc, ptr(tot), ptr(ws), stream_ptr()))
    return rows, tot


def mse_loss_grad(pred, target, grad_scale=1.0):
    require_cuda(pred, target)
    pred, target = pred.contiguous(), target.contiguous()
    dpred = torch.empty_like(pred)
    loss = torch.empty(1, device=pred.device, dtype=torch.float32)
    scratch = torch.empty(8192, device=pred.device, dtype=torch.uint8)
    check(lib().wc_mse_loss_grad(ptr(pred), ptr(target), ptr(dpred), pred.numel(), float(grad_scale), ptr(loss), ptr(scratch),
                                 stream_ptr()))
    return loss, dpred


def boundary_wgrad(wide, narrow, sign):
    """sign +1: conv_in (wide = d conv_in output [B,H,W,64] bf16, narrow = image [B,3,H,W] fp32) -> dw [64,3,3,3], db [64];
    sign -1: conv_out (wide = its input, narrow = dpred) -> dw [3,64,3,3], db [3]."""
    require_cuda(wide, narrow)
    B, H, W, Cc = wide.shape
    assert Cc == 64
    wide, narrow = wide.contiguous(), narrow.contiguous()
    dw = torch.empty((64, 3, 3, 3) if sign > 0 else (3, 64, 3, 3), device=wide.device, dtype=torch.float32)
    db = torch.empty(64 if sign > 0 else 3, device=wide.device, dtype=torch.float32)
    scratch = torch.empty(lib().wc_boundary_wgrad_scratch_bytes(), device=wide.device, dtype=torch.uint8)
    check(lib().wc_boundary_wgrad(ptr(wide), ptr(narrow), B, H, W, sign, ptr(dw), ptr(db), ptr(scratch), stream_ptr()))
    return dw, db


def adam_step(p, g, m, v, lr, beta1, beta2, eps, step, grad_scale=1.0):
    """In-place torch.optim.Adam update over flat fp32 buffers."""
    require_cuda(p, g, m, v)
    check(lib().wc_adam_step(ptr(p), ptr(g), ptr(m), ptr(v), p.numel(), lr, beta1, beta2, eps, step, grad_scale, stream_ptr()))
