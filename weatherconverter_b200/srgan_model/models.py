"""Swift-SRGAN Generator with the reference's constructor / forward contract (srgan_model/models.py:65-92) running
on the C plan in csrc/srgan.cu.  state_dict keys/shapes/order equal the reference's (283 tensors for the defaults).
Eval-mode BatchNorm only.

Autograd: with grad mode on and ``x.requires_grad``, ``forward(x)`` returns an image with a ``grad_fn``, so any loss on it
backpropagates to ``x`` (``seg(G(x))`` chains with the differentiable DeepLabV3+).  The graph is a function of ``x`` only: the
parameters are constants, no weight gradient is computed and every ``p.grad`` stays ``None``.  The backward is the plan's
data-gradient pass seeded with dL/dy (``wc_srgan_backward_seeded``).  A graph holds one plan (its saved activations) until its
backward has run or it is freed; the plans live in a pool per (B, h, w).  A graph can be backpropagated once.  Every other call
(no grad mode, ``x`` without grad, ``srgan_model.inference.inference``) runs the inference plan.
"""
import ctypes as C
import math

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from .. import _lib
from .._lib import check, lib, ptr, stream_ptr
from .._params import register_dotted
from .._plans import Lease, lease_plan


def param_spec(in_channels=3, nc=64, num_blocks=16, upscale_factor=4):
    """Ordered {name: (shape, kind)}, kind in {'w','b','prelu','bn_w','bn_b','mean','var','count'}."""
    spec = {}

    def sep(p, ci, co, k, bias):
        spec[p + ".depthwise.weight"] = ((ci, 1, k, k), "w")
        if bias:
            spec[p + ".depthwise.bias"] = ((ci,), "b")
        spec[p + ".pointwise.weight"] = ((co, ci, 1, 1), "w")
        if bias:
            spec[p + ".pointwise.bias"] = ((co,), "b")

    def convblock(p, ci, co, k, use_bn):
        sep(p + ".cnn", ci, co, k, not use_bn)
        if use_bn:
            spec[p + ".bn.weight"] = ((co,), "bn_w"); spec[p + ".bn.bias"] = ((co,), "bn_b")
            spec[p + ".bn.running_mean"] = ((co,), "mean"); spec[p + ".bn.running_var"] = ((co,), "var")
            spec[p + ".bn.num_batches_tracked"] = ((), "count")
        spec[p + ".act.weight"] = ((co,), "prelu")

    convblock("initial", in_channels, nc, 9, False)
    for i in range(num_blocks):
        convblock(f"residual.{i}.block1", nc, nc, 3, True)
        convblock(f"residual.{i}.block2", nc, nc, 3, True)
    convblock("convblock", nc, nc, 3, True)
    for i in range(upscale_factor // 2):
        sep(f"upsampler.{i}.conv", nc, nc * 4, 3, True)
        spec[f"upsampler.{i}.act.weight"] = ((nc,), "prelu")
    sep("final_conv", nc, in_channels, 9, True)
    return spec


class Generator(nn.Module):
    """Swift-SRGAN Generator (in_channels, num_channels, num_blocks, upscale_factor) -> super-resolved image in [0,1]."""

    def __init__(self, in_channels: int = 3, num_channels: int = 64, num_blocks: int = 16, upscale_factor: int = 4):
        super().__init__()
        if in_channels != 3 or num_channels != 64:
            raise NotImplementedError("the B200 SRGAN plan is built for in_channels=3, num_channels=64 (the reference's use)")
        self.num_blocks, self.upscale_factor = num_blocks, upscale_factor
        for name, (shape, kind) in param_spec(in_channels, num_channels, num_blocks, upscale_factor).items():
            if kind == "w":
                fan_in = shape[1] * shape[2] * shape[3]
                register_dotted(self, name, torch.empty(shape).uniform_(-1 / math.sqrt(fan_in), 1 / math.sqrt(fan_in)))
            elif kind == "b":
                register_dotted(self, name, torch.zeros(shape))
            elif kind == "prelu":
                register_dotted(self, name, torch.full(shape, 0.25))
            elif kind == "bn_w":
                register_dotted(self, name, torch.ones(shape))
            elif kind == "bn_b":
                register_dotted(self, name, torch.zeros(shape))
            elif kind == "mean":
                register_dotted(self, name, torch.zeros(shape), buffer=True)
            elif kind == "var":
                register_dotted(self, name, torch.ones(shape), buffer=True)
            else:
                register_dotted(self, name, torch.zeros(shape, dtype=torch.long), buffer=True)
        self._handle, self._key, self._ws, self._keep = None, None, {}, None
        self._grad_plans = {}        # (B, h, w) -> [_SrganGradPlan]: the autograd path's plan pool
        self._grad_key = None

    def _tensors(self):
        sd = dict(self.named_parameters())
        sd.update({n: b for n, b in self.named_buffers() if b.dtype == torch.float32})
        return sd

    def _destroy(self):
        if self._handle is not None:
            lib().wc_srgan_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    def _create_handle(self, ts, device):
        for n, t in ts.items():
            if t.device != device or not t.is_contiguous():
                raise RuntimeError(f"SRGAN parameter {n} must be contiguous on {device}; call .to(device)")
        n = len(ts)
        names = (C.c_char_p * n)(*[k.encode() for k in ts])
        ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in ts.values()])
        h = C.c_void_p()
        check(lib().wc_srgan_create(C.byref(h), self.num_blocks, self.upscale_factor, n, names, ptrs, stream_ptr()))
        return h

    def _ensure(self, device):
        ts = self._tensors()
        key = (str(device), tuple((t.data_ptr(), t._version) for t in ts.values()))
        if self._handle is not None and key == self._key:
            return
        self._destroy()
        h = self._create_handle(ts, device)
        self._handle, self._key, self._keep, self._ws = h, key, list(ts.values()), {}

    def _lease_plan(self, B, h, w, device):
        """A free autograd plan for (B, h, w), created when every plan of that shape is held by a live graph.  A plan packs
        the weights once, when it is first bound, so the pool is rebuilt whenever a tensor's storage or version changes
        (.to(), load_state_dict, any in-place update); a live graph keeps its own plan."""
        ts = self._tensors()
        key = (str(device), tuple((t.data_ptr(), t._version) for t in ts.values()))
        if key != self._grad_key:
            self._grad_plans, self._grad_key = {}, key
        return lease_plan(self._grad_plans, (B, h, w), lambda: _SrganGradPlan(self, ts, B, h, w, device))

    def forward(self, x, out=None):
        """x [B,3,h,w] -> y [B,3,u*h,u*w] in [0,1].  With grad mode on and ``x.requires_grad`` the result carries an autograd
        graph of ``x`` (the parameters are constants: no weight gradients, ``p.grad`` stays None); ``out=`` is then rejected."""
        _lib.require_cuda(x)
        if self.training:
            raise RuntimeError("the B200 SRGAN path implements eval-mode BatchNorm only; call .eval()")
        if torch.is_grad_enabled() and x.requires_grad:
            if out is not None:
                raise RuntimeError("Generator.forward: out= is not supported when the result carries an autograd graph "
                                   "(x.requires_grad under grad mode)")
            return _SrganFunction.apply(self, x.contiguous().float())
        x = x.contiguous().float()
        B, _, h, w = x.shape
        self._ensure(x.device)
        k = (B, h, w)
        if k not in self._ws:
            nbytes = lib().wc_srgan_workspace_bytes(self._handle, B, h, w)
            if nbytes == 0:
                check(1)
            self._ws = {k: torch.empty(nbytes, dtype=torch.uint8, device=x.device)}
        ws = self._ws[k]
        if out is None:
            out = torch.empty(B, 3, h * self.upscale_factor, w * self.upscale_factor, device=x.device)
        check(lib().wc_srgan_forward(self._handle, ptr(x), ptr(out), B, h, w, ptr(ws), ws.numel(), stream_ptr()))
        self._last = x
        return out

    def flops(self):
        return float(lib().wc_srgan_flops(self._handle)) if self._handle is not None else 0.0


class _SrganGradPlan:
    """A C handle of its own with a with-grad workspace, bound to (B, h, w) by its first forward (which packs the weights).
    Keeps the module's tensors alive: the handle reads them in place."""

    def __init__(self, G, ts, B, h, w, device):
        self.handle, self.busy = None, False
        self._keep = list(ts.values())
        self.handle = G._create_handle(ts, device)
        nbytes = lib().wc_srgan_grad_workspace_bytes(self.handle, B, h, w)
        if nbytes == 0:
            check(1)
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=device)

    def __del__(self):
        try:
            if self.handle is not None:
                lib().wc_srgan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class _SrganFunction(torch.autograd.Function):
    """y = Generator(x) on a leased plan that saves what the backward reads (every PReLU's pre-activation and a copy of y, so
    the backward reads no caller memory); backward seeded with dL/dy gives dL/dx.  Inputs: the module, x [B,3,h,w] fp32
    contiguous."""

    @staticmethod
    def forward(ctx, G, x):
        B, _, h, w = x.shape
        lease = Lease(G._lease_plan(B, h, w, x.device))
        plan = lease.plan
        u = G.upscale_factor
        y = torch.empty(B, 3, h * u, w * u, device=x.device)
        check(lib().wc_srgan_forward_saved(plan.handle, ptr(x), ptr(y), B, h, w, ptr(plan.ws), plan.ws.numel(), stream_ptr()))
        ctx.lease, ctx.x_shape = lease, x.shape
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y):
        lease = ctx.lease
        plan = lease.plan
        if plan is None:
            raise RuntimeError("Generator autograd: this graph has already been backpropagated; its saved activations are gone "
                               "(retain_graph=True re-backward is not supported: run the forward again)")
        g = grad_y.contiguous().float()
        dx = torch.empty(ctx.x_shape, device=g.device)
        check(lib().wc_srgan_backward_seeded(plan.handle, ptr(g), ptr(dx), stream_ptr()))
        lease.release()
        return None, dx
