"""How a Python object owns a C plan of libwc_b200.so: one module for every model (Unet, its training plans, the legacy
UNet, DeepLabV3+, the SRGAN generator) and for DenoisingTrainer.

* ``c_tensor_args`` checks an ordered {name: tensor} and builds the name / pointer / numel arrays every ``wc_*_create`` takes.
* ``PlanHandle`` owns one C handle, the tensors it reads in place, and the workspace of its current binding.
* ``PlanPool`` holds the plans made under one rebuild key: a module's inference plan (``one``) or, for the autograd paths,
  plans per input shape that live graphs lease (``lease``).
* ``PlanFunction`` is the ``torch.autograd.Function`` of the differentiable models.  A C plan bound to one input shape holds
  one forward's activations until its backward has run, so each live graph leases a plan of its own together with the
  inputs the plan reads; the lease ends when the graph's backward has been enqueued or when the graph is freed without one.
"""
import ctypes as C

import torch
from torch.autograd.function import once_differentiable

from ._lib import check


def c_tensor_args(tensors, device, owner, dtype=None):
    """ctypes (names, pointers, numels) of an ordered {name: tensor}, after checking that every tensor is contiguous, on
    ``device`` and, when given, of ``dtype``.  The handle made from them reads the tensors in place."""
    for name, t in tensors.items():
        if t.device != device or not t.is_contiguous() or (dtype is not None and t.dtype != dtype):
            kind = "" if dtype is None else str(dtype).replace("torch.", "") + " "
            raise RuntimeError(f"{owner} tensor {name} must be a contiguous {kind}tensor on {device}; call .to(device)")
    n = len(tensors)
    return ((C.c_char_p * n)(*[name.encode() for name in tensors]),
            (C.c_void_p * n)(*[t.data_ptr() for t in tensors.values()]),
            (C.c_int64 * n)(*[t.numel() for t in tensors.values()]))


class PlanHandle:
    """One C handle made by ``create(&handle, *args)`` and freed once by ``destroy``, with the tensors it reads in place
    (``keep``, alive as long as the handle) and at most one workspace, that of its current binding.  A plan leased by an
    autograd graph carries ``busy``."""

    def __init__(self, create, destroy, *args, keep=None):
        self.handle, self._destroy = None, destroy
        handle = C.c_void_p()
        check(create(C.byref(handle), *args))
        self.handle, self.keep = handle, keep
        self.ws, self._ws_key, self.busy = None, None, False

    def workspace(self, key, nbytes_fn, device):
        """The workspace of binding ``key``: cached while the key stays, else sized by ``nbytes_fn()`` (0: the library
        refused the binding, raised through ``check``).  The old workspace is dropped before the new one is allocated, so
        the two are never held together."""
        if key != self._ws_key:
            nbytes = nbytes_fn()
            if nbytes == 0:
                check(1)
            self.ws, self._ws_key = None, None
            self.ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
            self._ws_key = key
        return self.ws

    def __del__(self):
        try:
            if self.handle is not None:
                self._destroy(self.handle)
                self.handle = None
        except Exception:      # interpreter shutdown may have torn down the library already
            pass


class PlanPool(dict):
    """{shape: [plans]} made under one rebuild key.  A call with another key destroys them first.

    Every model builds its own key, and the keys differ on purpose:
    * Unet inference: device, ``_weights_epoch`` (DenoisingTrainer updates the weights in place by kernel, which no
      ``_version`` sees), and data_ptr and ``_version`` of every parameter: the plan packs the weights once.
    * Unet training pool: device and the parameters' data_ptrs only; every differentiable forward re-packs the weights.
    * DeepLabV3+ inference plan: device, and data_ptr and ``_version`` of the parameters and fp32 buffers; its autograd
      pool adds ``output_stride``.  Every plan packs the weights once.
    * SRGAN inference plan and pool: device, and data_ptr and ``_version`` of the parameters and fp32 buffers.
    * Legacy UNet: device, and data_ptr and ``_version`` of the fp32 ``state_dict`` entries, taken before the attention
      padding (which makes new tensors on every build).
    """

    key = None

    def _plans(self, key, shape):
        if key != self.key:
            self.clear()                        # the old handles are destroyed before a new one is made
            self.key = key
        return self.setdefault(shape, [])

    @property
    def plan(self):
        """The plan ``one`` returned last, or None before the first call."""
        plans = dict.get(self, None)
        return plans[0] if plans else None

    def one(self, key, make):
        """The pool's one plan (an inference plan: never leased), made with ``make()`` when there is none."""
        plans = self._plans(key, None)
        if not plans:
            plans.append(make())
        return plans[0]

    def lease(self, key, shape, make):
        """A free plan of ``shape``, made with ``make()`` when every plan of that shape is held by a live graph; marked
        busy.  ``pool[shape]`` lists the plans of one shape."""
        plans = self._plans(key, shape)
        plan = next((p for p in plans if not p.busy), None)
        if plan is None:
            plan = make()
            plans.append(plan)
        plan.busy = True
        return plan


class Lease:
    """A plan held by one autograd graph, with the forward's inputs (the backward may read them).  Released when the backward
    has been enqueued, or when the graph is freed without one (the Function's ctx, which owns the lease, dies)."""

    def __init__(self, plan, *inputs):
        self.plan, self.inputs = plan, inputs

    def release(self):
        if self.plan is not None:
            self.plan.busy = False
        self.plan, self.inputs = None, None

    def __del__(self):
        self.release()


class PlanFunction(torch.autograd.Function):
    """``model(x, *rest)`` on a plan leased with ``model._grad_plan(B, H, W, device)``; its backward is seeded with the
    output's gradient.  The model supplies the two calls:
      ``model._grad_forward(plan, x, *rest)`` -> the output;
      ``model._grad_backward(plan, grad, needs_input_grad, x, *rest)`` -> the gradients of (x, *rest), ``needs_input_grad``
      being those inputs' flags.
    A graph can be backpropagated once: its plan goes back to the pool as soon as the backward is enqueued."""

    @staticmethod
    def forward(ctx, model, x, *rest):
        B, _, H, W = x.shape
        lease = Lease(model._grad_plan(B, H, W, x.device), x, *rest)
        out = model._grad_forward(lease.plan, x, *rest)
        ctx.lease, ctx.model = lease, model
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        lease = ctx.lease
        if lease.plan is None:
            raise RuntimeError(f"{type(ctx.model).__name__} autograd: this graph has already been backpropagated; its saved "
                               "activations are gone (retain_graph=True re-backward is not supported: run the forward again)")
        grads = ctx.model._grad_backward(lease.plan, grad.contiguous().float(), ctx.needs_input_grad[1:], *lease.inputs)
        lease.release()
        return (None, *grads)
