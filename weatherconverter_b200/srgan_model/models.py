"""Swift-SRGAN Generator with the reference's constructor / forward contract (srgan_model/models.py:65-92) running
on the C plan in csrc/srgan.cu.  state_dict keys/shapes/order equal the reference's (283 tensors for the defaults).
Eval-mode BatchNorm only.

Autograd: with grad mode on and ``x.requires_grad``, ``forward(x)`` returns an image with a ``grad_fn``, so any loss on it
backpropagates to ``x`` (``seg(G(x))`` chains with the differentiable DeepLabV3+).  The graph is a function of ``x`` only: the
parameters are constants, no weight gradient is computed and every ``p.grad`` stays ``None``.  The backward is the plan's
data-gradient pass seeded with dL/dy (``wc_srgan_backward_seeded``).  A graph holds one plan (its saved activations) until its
backward has run or it is freed; the plans live in a pool per (B, h, w).  A graph can be backpropagated once.  Every other call
(no grad mode, ``x`` without grad, ``srgan_model.inference.inference``) runs the inference plan.  The handles, workspaces, pool
and autograd Function are those of ``_plans.py``.
"""
import math

import torch
import torch.nn as nn

from .. import _lib
from .._lib import check, lib, ptr, stream_ptr
from .._params import register_dotted
from .._plans import PlanFunction, PlanHandle, PlanPool, c_tensor_args


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
        self._infer = PlanPool()
        self._grad_plans = PlanPool()    # (B, h, w) -> plans with a with-grad workspace: the autograd path's plan pool

    def _tensors(self):
        sd = dict(self.named_parameters())
        sd.update({n: b for n, b in self.named_buffers() if b.dtype == torch.float32})
        return sd

    def _make_plan(self, ts, device):
        names, ptrs, _ = c_tensor_args(ts, device, "SRGAN")
        L = lib()
        return PlanHandle(L.wc_srgan_create, L.wc_srgan_destroy, self.num_blocks, self.upscale_factor, len(ts), names, ptrs,
                          stream_ptr(), keep=list(ts.values()))

    def _inference_plan(self, device):
        ts = self._tensors()
        key = (str(device), tuple((t.data_ptr(), t._version) for t in ts.values()))
        return self._infer.one(key, lambda: self._make_plan(ts, device))

    def _grad_plan(self, B, h, w, device):
        """A free autograd plan for (B, h, w) with a with-grad workspace, created when every plan of that shape is held by a
        live graph.  Its first forward binds it and packs the weights."""
        ts = self._tensors()
        key = (str(device), tuple((t.data_ptr(), t._version) for t in ts.values()))

        def make():
            plan = self._make_plan(ts, device)
            plan.workspace((B, h, w), lambda: lib().wc_srgan_grad_workspace_bytes(plan.handle, B, h, w), device)
            return plan
        return self._grad_plans.lease(key, (B, h, w), make)

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
            return PlanFunction.apply(self, x.contiguous().float())
        x = x.contiguous().float()
        B, _, h, w = x.shape
        plan = self._inference_plan(x.device)
        ws = plan.workspace((B, h, w), lambda: lib().wc_srgan_workspace_bytes(plan.handle, B, h, w), x.device)
        if out is None:
            out = torch.empty(B, 3, h * self.upscale_factor, w * self.upscale_factor, device=x.device)
        check(lib().wc_srgan_forward(plan.handle, ptr(x), ptr(out), B, h, w, ptr(ws), ws.numel(), stream_ptr()))
        self._last = x
        return out

    def flops(self):
        plan = self._infer.plan
        return float(lib().wc_srgan_flops(plan.handle)) if plan is not None else 0.0

    # ---- the autograd path (PlanFunction): the plan saves what the backward reads (every PReLU's pre-activation and a copy
    # of y, so the backward reads no caller memory); the backward seeded with dL/dy gives dL/dx
    def _grad_forward(self, plan, x):
        B, _, h, w = x.shape
        u = self.upscale_factor
        y = torch.empty(B, 3, h * u, w * u, device=x.device)
        check(lib().wc_srgan_forward_saved(plan.handle, ptr(x), ptr(y), B, h, w, ptr(plan.ws), plan.ws.numel(), stream_ptr()))
        return y

    def _grad_backward(self, plan, g, needs_input_grad, x):
        dx = torch.empty_like(x)
        check(lib().wc_srgan_backward_seeded(plan.handle, ptr(g), ptr(dx), stream_ptr()))
        return (dx,)
