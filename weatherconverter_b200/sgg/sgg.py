"""Semantic-gradient guidance with the reference's entry point (sgg/sgg.py:9-24).

``apply_gsg(seg_model, mu, sigma, sr_xt, gt, _lambda)`` = segmentation forward + CE + input gradient
(csrc/seg.cu), then ONE fused kernel for ``avg_pool2d(4)`` -> de-normalise -> channel L2 (float64) ->
``mu + lambda*sigma*mag + sigma`` (csrc/elementwise.cu: sgg_update_kernel).  The reference returns float64
(numpy promotion, SURVEY D7); this returns fp32 rounded from the same float64 arithmetic (the repaired driver casts
back to fp32 anyway).  ``apply_lcg`` raises as shipped (SURVEY D3); here it runs with the documented repair of its final masked sum.

``criterion``: GSG with any segmentation loss.  ``criterion(logits [B,19,H,W], gt [B,H,W]) -> [B]`` per-image losses; the
gradient d(sum_b loss_b)/d sr_xt comes from torch autograd through the segmentor (DeepLabV3.forward), then goes through the
same update kernel with its unfused average pooling.  ``None`` keeps the fused CE(ignore 255) plan.

``apply_gsg_through_srgan``: GSG guided by the exact gradient d loss / d x_t through the SRGAN generator (chain rule through
Generator.forward's autograd path) instead of the reference's stand-in avg_pool2d(d loss / d sr_xt, 4).  Its magnitude has a
different scale from the pooled stand-in, so ``lambda`` may need retuning (DESIGN.md section 4).
"""
import torch

from .. import _lib
from .._lib import check, lib, ptr, stream_ptr
from ..seg_model.inference import infer_batch


def _criterion_grad(seg_model, sr_xt, gt, criterion):
    """d(sum_b criterion(seg_model(x), gt)_b)/dx at x = sr_xt by torch autograd through the segmentor."""
    B = sr_xt.shape[0]
    if gt.dim() == 4:
        gt = gt.squeeze(1)
    gt = gt.long()
    with torch.enable_grad():
        x = sr_xt.detach().contiguous().float().requires_grad_(True)
        logits = seg_model(x)
        loss = criterion(logits, gt)
        if not torch.is_tensor(loss) or tuple(loss.shape) != (B,):
            shape = tuple(loss.shape) if torch.is_tensor(loss) else type(loss).__name__
            raise ValueError(f"criterion must return one loss per image, shape ({B},); got {shape} "
                             "(a batch-mean scalar would scale every image's guidance by 1/B)")
        grad, = torch.autograd.grad(loss.sum(), x)
    return dict(grad=grad, loss=loss.detach(), logits=logits.detach())


def apply_gsg_batch(seg_model, mu, sigma, sr_xt, gt, _lambda, pool=None, return_aux=False, fused_pool=True, criterion=None):
    """Batched GSG: every image uses its own loss/gradient (vmap of the reference's B = 1 semantics).  ``criterion``
    (optional): callable (logits [B,19,H,W], gt [B,H,W]) -> per-image losses [B] replacing the fused CE(ignore 255); image b
    is guided by d loss_b / d sr_xt[b].  It runs torch autograd, so it cannot be captured in a CUDA graph."""
    if criterion is not None and not callable(criterion):
        raise TypeError("criterion must be a callable (logits, gt) -> per-image losses [B]")
    _lib.require_cuda(mu, sigma, sr_xt, gt)
    B, _, h, w = mu.shape
    if pool is None:
        pool = sr_xt.shape[-1] // w
    if criterion is not None:
        if torch.cuda.is_current_stream_capturing():
            raise ValueError("apply_gsg_batch: a custom criterion runs torch autograd and cannot be captured in a CUDA graph")
        out = _criterion_grad(seg_model, sr_xt, gt, criterion)
        mu, sigma = mu.contiguous().float(), sigma.contiguous().float()
        xt = torch.empty_like(mu)
        check(lib().wc_sgg_update(ptr(out["grad"]), ptr(mu), ptr(sigma), ptr(xt), None, B, h, w, pool, float(_lambda),
                                  stream_ptr()))
        return (xt, out) if return_aux else xt
    # avg_pool2d(grad, pool) (sgg.py:18) is folded into the segmentor's stem data-gradient kernel when possible
    fused = fused_pool and pool in (2, 4, 6, 8)
    out = infer_batch(seg_model, sr_xt, gt, grad_pool=pool if fused else 1)
    mu, sigma = mu.contiguous().float(), sigma.contiguous().float()
    xt = torch.empty_like(mu)
    check(lib().wc_sgg_update(ptr(out["grad"]), ptr(mu), ptr(sigma), ptr(xt), None, B, h, w, 1 if fused else pool,
                              float(_lambda), stream_ptr()))
    return (xt, out) if return_aux else xt


def apply_gsg(seg_model, mu, sigma, sr_xt, gt, _lambda, criterion=None):
    return apply_gsg_batch(seg_model, mu, sigma, sr_xt, gt, _lambda, criterion=criterion)


def apply_lcg(seg_model, mu, sigma, sr_xt, gt, _lambda, num_classes=19, pool=None):
    """Local class guidance (reference sgg.py:27-60).  The per-class body is the reference's: mask the image and
    the labels with mc = (gt == c), take the segmentation-loss gradient, pool, magnitude.  The shipped final sum
    multiplies 128x128 tensors by 512x512 masks and raises (SURVEY D3); the repair (documented in DESIGN.md section 4) average-pools the class masks to the latent resolution and leaves pixels without a class
    unguided:  xt = mu + sigma + lambda * sigma * sum_c avg_pool(mc)_c * |g4_c|.
    All classes of all images run as ONE batch of B*19 masked images through the segmentor plan."""
    _lib.require_cuda(mu, sigma, sr_xt, gt)
    B, _, h, w = mu.shape
    Hs, Ws = sr_xt.shape[-2:]
    if pool is None:
        pool = Ws // w
    sr_xt, gt = sr_xt.contiguous().float(), gt.contiguous().long()
    xm = torch.empty(B * num_classes, 3, Hs, Ws, device=mu.device)
    gm = torch.empty(B * num_classes, Hs, Ws, dtype=torch.long, device=mu.device)
    check(lib().wc_lcg_prepare(ptr(sr_xt), ptr(gt), ptr(xm), ptr(gm), B, num_classes, Hs, Ws, stream_ptr()))
    g4 = infer_batch(seg_model, xm, gm, grad_pool=pool)["grad"]
    mu, sigma = mu.contiguous().float(), sigma.contiguous().float()
    xt = torch.empty_like(mu)
    check(lib().wc_lcg_combine(ptr(g4), ptr(gt), ptr(mu), ptr(sigma), ptr(xt), B, num_classes, h, w, pool, float(_lambda),
                               stream_ptr()))
    return xt


def apply_gsg_through_srgan(seg_model, srgan_model, mu, sigma, xt, gt, _lambda, criterion=None, return_aux=False):
    """GSG with image b guided by d loss_b / d x_t[b]: sr = srgan_model(x_t) (the bits of srgan_inference), g_sr = d(sum_b
    loss_b)/d sr from the fused CE(ignore 255) plan (``criterion=None``) or from torch autograd through the segmentor, then
    g_x = g_sr pulled back through the generator by autograd, and the update kernel without pooling (same de-normalise and
    channel L2).  ``return_aux`` adds dict(sr, loss, grad = g_x).  Runs torch autograd: no CUDA-graph capture."""
    if criterion is not None and not callable(criterion):
        raise TypeError("criterion must be a callable (logits, gt) -> per-image losses [B]")
    _lib.require_cuda(mu, sigma, xt, gt)
    if torch.cuda.is_current_stream_capturing():
        raise ValueError("apply_gsg_through_srgan runs torch autograd and cannot be captured in a CUDA graph")
    B, _, h, w = mu.shape
    with torch.enable_grad():
        x = xt.detach().contiguous().float().requires_grad_(True)
        sr = srgan_model(x)
        if criterion is None:
            out = infer_batch(seg_model, sr.detach(), gt, grad_pool=1)
        else:
            out = _criterion_grad(seg_model, sr.detach(), gt, criterion)
        g_x, = torch.autograd.grad(sr, x, out["grad"])
    mu, sigma = mu.contiguous().float(), sigma.contiguous().float()
    new_xt = torch.empty_like(mu)
    check(lib().wc_sgg_update(ptr(g_x), ptr(mu), ptr(sigma), ptr(new_xt), None, B, h, w, 1, float(_lambda), stream_ptr()))
    return (new_xt, dict(sr=sr.detach(), loss=out["loss"], grad=g_x)) if return_aux else new_xt
