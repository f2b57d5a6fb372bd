"""DeepLabV3+ factories with the reference's names and signatures (seg_model/network/modeling.py:182-202),
backed by the C plan in csrc/seg.cu (forward, loss head and input gradient on libwc_b200.so).

Autograd: with grad mode on and ``x.requires_grad``, ``forward(x)`` returns logits with a ``grad_fn``, so any loss on them
backpropagates to ``x`` (``loss.backward()`` fills ``x.grad``; ``torch.autograd.grad(loss, x)`` works).  The graph is a
function of ``x`` only: the parameters are constants, no weight gradient is computed and every ``p.grad`` stays ``None``
(eval-mode BatchNorm is folded into the convolutions; segmentor training is not supported).  The backward is the plan's
data-gradient pass seeded with dL/dlogits (``wc_seg_backward_seeded``).  A graph holds one plan (its saved activations)
until its backward has run or it is freed; the plans live in a pool per (B, H, W).  A graph can be backpropagated once.

Only the ResNet-50/101 DeepLabV3+ variants reachable from the reference's configured model name are provided
(SURVEY.md section 2, rows 10-12); output_stride 16 (the reference's config, seg_model/config/config.yaml:66).
The returned module's state_dict has the reference's keys/shapes/order (368 tensors for R50, 674 for R101).
"""
import ctypes as C
import math

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from ... import _lib
from ..._lib import check, lib, ptr, stream_ptr
from ..._params import register_dotted
from ..._plans import Lease, lease_plan

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
        self._handle = None
        self._key = None
        self._ws = {}
        self._keep = None
        self._grad_plans = {}        # (B, H, W) -> [_SegGradPlan]: the autograd path's plan pool
        self._grad_key = None

    # ---- C handle --------------------------------------------------------------------------------------
    def _tensors(self):
        sd = {}
        for n, p in self.named_parameters():
            sd[n] = p
        for n, b in self.named_buffers():
            if b.dtype == torch.float32:
                sd[n] = b
        return sd

    def _destroy(self):
        if self._handle is not None:
            lib().wc_seg_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    def _create_handle(self, ts, device):
        for n, t in ts.items():
            if t.device != device or not t.is_contiguous():
                raise RuntimeError(f"seg parameter {n} must be contiguous on {device}; call .to(device)")
        n = len(ts)
        names = (C.c_char_p * n)(*[k.encode() for k in ts])
        ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in ts.values()])
        layers = (C.c_int * 4)(*_LAYERS[self.backbone_name])
        h = C.c_void_p()
        check(lib().wc_seg_create(C.byref(h), layers, self.num_classes, n, names, ptrs, stream_ptr()))
        check(lib().wc_seg_set_output_stride(h, self.output_stride))
        return h

    def _ensure(self, device):
        ts = self._tensors()
        key = (str(device), tuple((t.data_ptr(), t._version) for t in ts.values()))
        if self._handle is not None and key == self._key:
            return
        self._destroy()
        h = self._create_handle(ts, device)
        self._handle, self._key, self._keep, self._ws = h, key, list(ts.values()), {}

    def _lease_plan(self, B, H, W, device):
        """A free autograd plan for (B, H, W), created when every plan of that shape is held by a live graph.  A plan packs
        the weights once, when it is first bound, so the pool is rebuilt whenever a tensor's storage or version changes
        (.to(), load_state_dict, any in-place update); a live graph keeps its own plan."""
        ts = self._tensors()
        key = (str(device), self.output_stride, tuple((t.data_ptr(), t._version) for t in ts.values()))
        if key != self._grad_key:
            self._grad_plans, self._grad_key = {}, key
        return lease_plan(self._grad_plans, (B, H, W), lambda: _SegGradPlan(self, ts, B, H, W, device))

    def _workspace(self, B, H, W, with_grad, device):
        k = (B, H, W, with_grad)
        if k not in self._ws:
            nbytes = lib().wc_seg_workspace_bytes(self._handle, B, H, W, 1 if with_grad else 0)
            if nbytes == 0:
                check(1)
            self._ws = {k: torch.empty(nbytes, dtype=torch.uint8, device=device)}
        return self._ws[k]

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
        self._ensure(x.device)
        ws = self._workspace(B, H, W, want_grad, x.device)
        pred = torch.empty(B, H, W, dtype=torch.long, device=x.device)
        grad = torch.empty(B, 3, H // grad_pool, W // grad_pool, device=x.device) if want_grad else None
        loss = torch.empty(B, dtype=torch.float32, device=x.device)
        logits = torch.empty(B, self.num_classes, H, W, device=x.device) if want_logits else None
        check(lib().wc_seg_infer_pooled(self._handle, ptr(x), ptr(labels), ptr(pred), ptr(grad), ptr(loss), ptr(logits), B, H, W,
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
        r._handle, r._key, r._ws, r._keep = None, None, {}, None
        r._grad_plans, r._grad_key = {}, None
        return r

    def forward(self, x):
        """x [B,3,H,W] -> logits fp32 [B,num_classes,H,W].  With grad mode on and ``x.requires_grad`` the result carries an
        autograd graph of ``x`` (the parameters are constants: no weight gradients, ``p.grad`` stays None)."""
        _lib.require_cuda(x)
        if self.training:
            raise RuntimeError("the B200 DeepLabV3+ path implements eval-mode BatchNorm only; call .eval()")
        if torch.is_grad_enabled() and x.requires_grad:
            return _SegFunction.apply(self, x.contiguous().float())
        x = x.contiguous().float()
        B, _, H, W = x.shape
        self._ensure(x.device)
        ws = self._workspace(B, H, W, False, x.device)
        logits = torch.empty(B, self.num_classes, H, W, device=x.device)
        check(lib().wc_seg_forward(self._handle, ptr(x), ptr(logits), B, H, W, 0, ptr(ws), ws.numel(), stream_ptr()))
        self._last = (x,)
        return logits

    def flops(self):
        return (float(lib().wc_seg_flops(self._handle, 0)), float(lib().wc_seg_flops(self._handle, 1)))


class _SegGradPlan:
    """A C handle of its own with a with-grad workspace, bound to (B, H, W) by its first forward (which packs the weights).
    Keeps the module's tensors alive: the handle reads them in place."""

    def __init__(self, seg, ts, B, H, W, device):
        self.handle, self.busy = None, False
        self._keep = list(ts.values())
        self.handle = seg._create_handle(ts, device)
        nbytes = lib().wc_seg_workspace_bytes(self.handle, B, H, W, 1)
        if nbytes == 0:
            check(1)
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=device)

    def __del__(self):
        try:
            if self.handle is not None:
                lib().wc_seg_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class _SegFunction(torch.autograd.Function):
    """logits = DeepLabV3(x) on a leased plan that saves its activations; backward seeded with dL/dlogits gives dL/dx.
    Inputs: the module, x [B,3,H,W] fp32 contiguous."""

    @staticmethod
    def forward(ctx, seg, x):
        B, _, H, W = x.shape
        lease = Lease(seg._lease_plan(B, H, W, x.device), x)
        plan = lease.plan
        logits = torch.empty(B, seg.num_classes, H, W, device=x.device)
        check(lib().wc_seg_forward(plan.handle, ptr(x), ptr(logits), B, H, W, 1, ptr(plan.ws), plan.ws.numel(), stream_ptr()))
        ctx.lease = lease
        return logits

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_logits):
        lease = ctx.lease
        plan = lease.plan
        if plan is None:
            raise RuntimeError("DeepLabV3 autograd: this graph has already been backpropagated; its saved activations are gone "
                               "(retain_graph=True re-backward is not supported: run the forward again)")
        x = lease.inputs[0]
        g = grad_logits.contiguous().float()
        dx = torch.empty_like(x)
        check(lib().wc_seg_backward_seeded(plan.handle, ptr(g), ptr(dx), stream_ptr()))
        lease.release()
        return None, dx


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
