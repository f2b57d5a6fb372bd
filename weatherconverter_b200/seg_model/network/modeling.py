"""DeepLabV3+ factories with the reference's names and signatures (seg_model/network/modeling.py:182-202),
backed by the C plan in csrc/seg.cu (forward, loss head and input gradient on libwc_b200.so).

Autograd: with grad mode on and ``x.requires_grad``, ``forward(x)`` returns logits with a ``grad_fn``, so any loss on them
backpropagates to ``x`` (``loss.backward()`` fills ``x.grad``; ``torch.autograd.grad(loss, x)`` works).  The graph is a
function of ``x`` only: the parameters are constants, no weight gradient is computed and every ``p.grad`` stays ``None``
(eval-mode BatchNorm is folded into the convolutions; segmentor training is not supported).  The backward is the plan's
data-gradient pass seeded with dL/dlogits (``wc_seg_backward_seeded``).  A graph holds one plan (its saved activations)
until its backward has run or it is freed; the plans live in a pool per (B, H, W).  A graph can be backpropagated once.
The handles, workspaces, pool and autograd Function are those of ``_plans.py``.

Only the ResNet-50/101 DeepLabV3+ variants reachable from the reference's configured model name are provided
(SURVEY.md section 2, rows 10-12); output_stride 16 (the reference's config, seg_model/config/config.yaml:66).
The returned module's state_dict has the reference's keys/shapes/order (368 tensors for R50, 674 for R101).
"""
import ctypes as C
import math

import torch
import torch.nn as nn

from ... import _lib
from ..._lib import check, lib, ptr, stream_ptr
from ..._params import register_dotted
from ..._plans import PlanFunction, PlanHandle, PlanPool, c_tensor_args

__all__ = ["deeplabv3plus_resnet50", "deeplabv3plus_resnet101", "DeepLabV3"]

_LAYERS = {"resnet50": [3, 4, 6, 3], "resnet101": [3, 4, 23, 3]}


def block_plan(backbone):
    """[(prefix, inplanes, planes, has_downsample)] following ResNet._make_layer (resnet.py:164-194) for os=16."""
    out, inplanes = [], 64
    for li, (planes, n, stride) in enumerate(zip([64, 128, 256, 512], _LAYERS[backbone], [1, 2, 2, 1])):
        for b in range(n):
            out.append((f"backbone.layer{li + 1}.{b}", inplanes, planes, b == 0 and (stride != 1 or inplanes != planes * 4)))
            inplanes = planes * 4
    return out


def param_spec(backbone="resnet50", num_classes=19):
    """Ordered {name: (shape, kind)}; kind in {'conv','bn_w','bn_b','mean','var','count','bias'} in the reference's
    registration order (backbone.* then classifier.*)."""
    spec = {}

    def conv(p, o, i, k):
        spec[p + ".weight"] = ((o, i, k, k), "conv")

    def bn(p, c):
        spec[p + ".weight"] = ((c,), "bn_w"); spec[p + ".bias"] = ((c,), "bn_b")
        spec[p + ".running_mean"] = ((c,), "mean"); spec[p + ".running_var"] = ((c,), "var")
        spec[p + ".num_batches_tracked"] = ((), "count")

    conv("backbone.conv1", 64, 3, 7); bn("backbone.bn1", 64)
    for (p, inpl, planes, down) in block_plan(backbone):
        conv(p + ".conv1", planes, inpl, 1); bn(p + ".bn1", planes)
        conv(p + ".conv2", planes, planes, 3); bn(p + ".bn2", planes)
        conv(p + ".conv3", planes * 4, planes, 1); bn(p + ".bn3", planes * 4)
        if down:
            conv(p + ".downsample.0", planes * 4, inpl, 1); bn(p + ".downsample.1", planes * 4)
    c = "classifier"
    conv(c + ".project.0", 48, 256, 1); bn(c + ".project.1", 48)
    conv(c + ".aspp.convs.0.0", 256, 2048, 1); bn(c + ".aspp.convs.0.1", 256)
    for k in (1, 2, 3):
        conv(f"{c}.aspp.convs.{k}.0", 256, 2048, 3); bn(f"{c}.aspp.convs.{k}.1", 256)
    conv(c + ".aspp.convs.4.1", 256, 2048, 1); bn(c + ".aspp.convs.4.2", 256)
    conv(c + ".aspp.project.0", 256, 1280, 1); bn(c + ".aspp.project.1", 256)
    conv(c + ".classifier.0", 256, 304, 3); bn(c + ".classifier.1", 256)
    spec[c + ".classifier.3.weight"] = ((num_classes, 256, 1, 1), "conv")
    spec[c + ".classifier.3.bias"] = ((num_classes,), "bias")
    return spec


class DeepLabV3(nn.Module):
    """DeepLabV3+ (ResNet backbone) with the reference's forward contract: x [B,3,H,W] fp32 -> logits [B,nc,H,W]."""

    def __init__(self, backbone_name, num_classes, output_stride=16):
        super().__init__()
        self.backbone_name, self.num_classes, self.output_stride = backbone_name, num_classes, output_stride
        for name, (shape, kind) in param_spec(backbone_name, num_classes).items():
            if kind == "conv":      # kaiming_normal_ (fan_out for the backbone resnet.py:155, fan_in for the head _deeplab.py:56)
                fan = (shape[0] if name.startswith("backbone") else shape[1]) * shape[2] * shape[3]
                register_dotted(self, name, torch.randn(shape) * math.sqrt(2.0 / fan))
            elif kind == "bn_w":
                register_dotted(self, name, torch.ones(shape))
            elif kind in ("bn_b",):
                register_dotted(self, name, torch.zeros(shape))
            elif kind == "bias":
                register_dotted(self, name, torch.empty(shape).uniform_(-1 / 16.0, 1 / 16.0))
            elif kind == "mean":
                register_dotted(self, name, torch.zeros(shape), buffer=True)
            elif kind == "var":
                register_dotted(self, name, torch.ones(shape), buffer=True)
            else:
                register_dotted(self, name, torch.zeros(shape, dtype=torch.long), buffer=True)
        self._infer = PlanPool()
        self._grad_plans = PlanPool()    # (B, H, W) -> plans with a with-grad workspace: the autograd path's plan pool

    # ---- C handle --------------------------------------------------------------------------------------
    def _tensors(self):
        sd = {}
        for n, p in self.named_parameters():
            sd[n] = p
        for n, b in self.named_buffers():
            if b.dtype == torch.float32:
                sd[n] = b
        return sd

    def _make_plan(self, ts, device):
        names, ptrs, _ = c_tensor_args(ts, device, "seg")
        layers = (C.c_int * 4)(*_LAYERS[self.backbone_name])
        L = lib()
        plan = PlanHandle(L.wc_seg_create, L.wc_seg_destroy, layers, self.num_classes, len(ts), names, ptrs, stream_ptr(),
                          keep=list(ts.values()))
        check(L.wc_seg_set_output_stride(plan.handle, self.output_stride))
        return plan

    def _inference_plan(self, device):
        ts = self._tensors()
        key = (str(device), tuple((t.data_ptr(), t._version) for t in ts.values()))
        return self._infer.one(key, lambda: self._make_plan(ts, device))

    def _grad_plan(self, B, H, W, device):
        """A free autograd plan for (B, H, W) with a with-grad workspace, created when every plan of that shape is held by a
        live graph.  Its first forward binds it and packs the weights."""
        ts = self._tensors()
        key = (str(device), self.output_stride, tuple((t.data_ptr(), t._version) for t in ts.values()))

        def make():
            plan = self._make_plan(ts, device)
            plan.workspace((B, H, W), lambda: lib().wc_seg_workspace_bytes(plan.handle, B, H, W, 1), device)
            return plan
        return self._grad_plans.lease(key, (B, H, W), make)

    def _workspace(self, plan, B, H, W, with_grad, device):
        return plan.workspace((B, H, W, with_grad),
                              lambda: lib().wc_seg_workspace_bytes(plan.handle, B, H, W, 1 if with_grad else 0), device)

    def infer(self, x, labels, want_grad=True, want_logits=False, grad_pool=1):
        """Forward + argmax + per-image CE(ignore 255) + input gradient in one stream-ordered plan.
        Returns dict(pred int64 [B,H,W], grad fp32 [B,3,H/grad_pool,W/grad_pool] | None, loss [B], logits | None).
        grad_pool > 1 returns F.avg_pool2d(grad, grad_pool) computed by a fused stem kernel (sgg/sgg.py:18)."""
        _lib.require_cuda(x, labels)
        if self.training:
            raise RuntimeError("the B200 DeepLabV3+ path implements eval-mode BatchNorm only; call .eval()")
        x = x.contiguous().float()
        labels = labels.contiguous().long()
        B, _, H, W = x.shape
        plan = self._inference_plan(x.device)
        ws = self._workspace(plan, B, H, W, want_grad, x.device)
        pred = torch.empty(B, H, W, dtype=torch.long, device=x.device)
        grad = torch.empty(B, 3, H // grad_pool, W // grad_pool, device=x.device) if want_grad else None
        loss = torch.empty(B, dtype=torch.float32, device=x.device)
        logits = torch.empty(B, self.num_classes, H, W, device=x.device) if want_logits else None
        check(lib().wc_seg_infer_pooled(plan.handle, ptr(x), ptr(labels), ptr(pred), ptr(grad), ptr(loss), ptr(logits), B, H, W,
                                        int(grad_pool), ptr(ws), ws.numel(), stream_ptr()))
        self._last = (x, labels)
        return dict(pred=pred, grad=grad, loss=loss, logits=logits)

    def shared_replica(self):
        """A second module object over the SAME parameter tensors with its own C plan / workspace binding.  A plan is bound to
        one (batch, H, W) at a time and re-binding frees the packed weights a captured CUDA graph still points to, so a loop
        that alternates two batch shapes under graphs (GSG on B images, LCG on 19 B masked images) gives each shape its own
        replica."""
        import copy
        r = copy.copy(self)          # shares _parameters / _buffers (no new tensors)
        r._infer, r._grad_plans = PlanPool(), PlanPool()
        return r

    def forward(self, x):
        """x [B,3,H,W] -> logits fp32 [B,num_classes,H,W].  With grad mode on and ``x.requires_grad`` the result carries an
        autograd graph of ``x`` (the parameters are constants: no weight gradients, ``p.grad`` stays None)."""
        _lib.require_cuda(x)
        if self.training:
            raise RuntimeError("the B200 DeepLabV3+ path implements eval-mode BatchNorm only; call .eval()")
        if torch.is_grad_enabled() and x.requires_grad:
            return PlanFunction.apply(self, x.contiguous().float())
        x = x.contiguous().float()
        B, _, H, W = x.shape
        plan = self._inference_plan(x.device)
        ws = self._workspace(plan, B, H, W, False, x.device)
        logits = torch.empty(B, self.num_classes, H, W, device=x.device)
        check(lib().wc_seg_forward(plan.handle, ptr(x), ptr(logits), B, H, W, 0, ptr(ws), ws.numel(), stream_ptr()))
        self._last = (x,)
        return logits

    def flops(self):
        plan = self._infer.plan
        handle = plan.handle if plan is not None else None
        return (float(lib().wc_seg_flops(handle, 0)), float(lib().wc_seg_flops(handle, 1)))

    # ---- the autograd path (PlanFunction): the plan saves its activations; the backward seeded with dL/dlogits gives dL/dx
    def _grad_forward(self, plan, x):
        B, _, H, W = x.shape
        logits = torch.empty(B, self.num_classes, H, W, device=x.device)
        check(lib().wc_seg_forward(plan.handle, ptr(x), ptr(logits), B, H, W, 1, ptr(plan.ws), plan.ws.numel(), stream_ptr()))
        return logits

    def _grad_backward(self, plan, g, needs_input_grad, x):
        dx = torch.empty_like(x)
        check(lib().wc_seg_backward_seeded(plan.handle, ptr(g), ptr(dx), stream_ptr()))
        return (dx,)


def _build(backbone, num_classes, output_stride, pretrained_backbone):
    if output_stride not in (8, 16):
        raise ValueError("output_stride must be 8 or 16 (seg_model/network/modeling.py:34-39)")
    if pretrained_backbone:
        raise RuntimeError("pretrained_backbone=True needs a network download (resnet.py:216-222); load a checkpoint instead")
    return DeepLabV3(backbone, num_classes, output_stride)


def deeplabv3plus_resnet50(num_classes=21, output_stride=8, pretrained_backbone=True):
    return _build("resnet50", num_classes, output_stride, pretrained_backbone)


def deeplabv3plus_resnet101(num_classes=21, output_stride=8, pretrained_backbone=True):
    return _build("resnet101", num_classes, output_stride, pretrained_backbone)
