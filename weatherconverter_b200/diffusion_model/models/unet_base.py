"""Unet with the reference's interface (diffusion_model/models/unet_base.py:372-488) running on libwc_b200.so.

``Unet(model_config).forward(x, t)`` takes the reference's tensors (x [B,3,H,W] fp32 NCHW, t int tensor [1] or
[B] / int / tuple) and returns noise_pred [B,3,H,W] fp32.  ``state_dict()`` has exactly the reference's key
names and shapes (382 tensors for config.yaml), so reference checkpoints load with ``load_state_dict``.

The module only owns parameters and device buffers; the layer graph, weight re-packing (bf16, K-major) and all
arithmetic live in the C library (csrc/unet.cu), and the C handles, their workspaces and the plan pool are held through
``_plans.py``.  By default outputs carry no autograd graph.

Autograd (opt-in): with ``model.differentiable = True``, grad mode on and ``x`` or any parameter requiring grad,
``forward`` runs the training plan (csrc/unet_train.cu) under ``_plans.PlanFunction`` whose inputs are ``x``,
``t`` and every parameter, so ``loss.backward()`` with any loss, hooks, ``clip_grad_norm_``, gradient accumulation
and any ``torch.optim`` optimizer work as on the reference module; ``x.grad`` is dL/dx.  The backward is
``wc_unet_train_backward_seeded`` fed with dL/d(noise_pred); it skips the parameter-gradient launches when no
parameter needs a gradient.  A graph holds one training plan (its saved activations) until its backward has run or
it is freed; the plans live in a pool per (B, H, W).  A graph can be backpropagated once (no ``retain_graph``
re-backward, no double backward).  The switch is off by default because the training plan keeps every activation
and is slower than the inference plan, which sampling and translation call with grad mode on.
"""
import ctypes as C
import math

import torch
import torch.nn as nn

from ... import _lib
from ..._lib import UnetConfigStruct, check, lib, ptr, stream_ptr
from ..._plans import PlanFunction, PlanHandle, PlanPool, c_tensor_args


def _cfg_get(cfg, k):
    return cfg[k] if isinstance(cfg, dict) else getattr(cfg, k)


def param_spec(cfg):
    """Ordered {name: shape} of the reference Unet's parameters for a ModelConfig
    (structure of unet_base.py:378-449: t_proj, conv_in, downs, mids, ups, norm_out, conv_out)."""
    dc, mc, ds = list(_cfg_get(cfg, "down_channels")), list(_cfg_get(cfg, "mid_channels")), list(_cfg_get(cfg, "down_sample"))
    T, ims, imc = _cfg_get(cfg, "time_emb_dim"), _cfg_get(cfg, "im_size"), _cfg_get(cfg, "im_channels")
    attn_res = list(_cfg_get(cfg, "attn_resolutions"))
    spec = {}

    def wb(prefix, wshape):
        spec[prefix + ".weight"] = tuple(wshape)
        spec[prefix + ".bias"] = (wshape[0],)

    def stage(prefix, cin, cout, n_res, n_attn):
        for l in range(n_res):
            ci = cin if l == 0 else cout
            wb(f"{prefix}.resnet_conv_first.{l}.0", (ci,))
            wb(f"{prefix}.resnet_conv_first.{l}.2", (cout, ci, 3, 3))
        for l in range(n_res):
            wb(f"{prefix}.t_emb_layers.{l}.1", (cout, T))
        for l in range(n_res):
            wb(f"{prefix}.resnet_conv_second.{l}.0", (cout,))
            wb(f"{prefix}.resnet_conv_second.{l}.2", (cout, cout, 3, 3))
        for l in range(n_attn):
            wb(f"{prefix}.attention_norms.{l}", (cout,))
        for l in range(n_attn):
            spec[f"{prefix}.attentions.{l}.in_proj_weight"] = (3 * cout, cout)
            spec[f"{prefix}.attentions.{l}.in_proj_bias"] = (3 * cout,)
            wb(f"{prefix}.attentions.{l}.out_proj", (cout, cout))
        for l in range(n_res):
            wb(f"{prefix}.residual_input_conv.{l}", (cout, cin if l == 0 else cout, 1, 1))

    wb("t_proj.0", (T, T))
    wb("t_proj.2", (T, T))
    wb("conv_in", (dc[0], imc, 3, 3))
    levels = len(dc) - 1
    for i in range(levels):
        attn = (ims // 2 ** i) in attn_res
        stage(f"downs.{i}", dc[i], dc[i + 1], _cfg_get(cfg, "num_down_layers"), _cfg_get(cfg, "num_down_layers") if attn else 0)
        if ds[i]:
            wb(f"downs.{i}.down_sample_conv", (dc[i + 1], dc[i + 1], 4, 4))
    for i in range(len(mc) - 1):
        stage(f"mids.{i}", mc[i], mc[i + 1], _cfg_get(cfg, "num_mid_layers") + 1, _cfg_get(cfg, "num_mid_layers"))
    for j, i in enumerate(reversed(range(levels))):
        attn = (ims // 2 ** i) in attn_res
        stage(f"ups.{j}", 2 * dc[i], dc[i - 1] if i != 0 else dc[0], _cfg_get(cfg, "num_up_layers"),
              _cfg_get(cfg, "num_up_layers") if attn else 0)
        if ds[i]:
            spec[f"ups.{j}.up_sample_conv.weight"] = (dc[i], dc[i], 4, 4)   # ConvTranspose2d: [Cin, Cout, 4, 4]
            spec[f"ups.{j}.up_sample_conv.bias"] = (dc[i],)
    wb("norm_out", (dc[0],))
    wb("conv_out", (imc, dc[0], 3, 3))
    return spec


class _Node(nn.Module):
    """Anonymous container: gives parameters the reference's dotted state_dict names."""


def _init_param(name, shape):
    leaf = name.rsplit(".", 1)[-1]
    if len(shape) == 1:
        if leaf == "weight":          # GroupNorm scale
            return torch.ones(shape)
        if "norm" in name or ".0.bias" in name and "resnet_conv" in name:
            return torch.zeros(shape)
        if leaf in ("in_proj_bias",) or name.endswith("out_proj.bias"):
            return torch.zeros(shape)
        return None                   # conv / linear bias: filled with its weight's fan-in below
    if leaf == "in_proj_weight":
        bound = math.sqrt(6.0 / (shape[0] + shape[1]))    # xavier_uniform (nn.MultiheadAttention default)
    else:
        fan_in = 1
        for s in shape[1:]:
            fan_in *= s
        if "up_sample_conv" in name:
            fan_in = shape[0] * shape[2] * shape[3]
        bound = 1.0 / math.sqrt(fan_in)                   # kaiming_uniform(a=sqrt(5)) (nn.Conv2d / nn.Linear default)
    return torch.empty(shape).uniform_(-bound, bound)


class Unet(nn.Module):
    r"""Unet comprising down blocks, mid blocks and up blocks (same constructor/forward contract as the reference)."""

    def __init__(self, model_config):
        super().__init__()
        g = lambda k: _cfg_get(model_config, k)  # noqa: E731
        self.down_channels = list(g("down_channels"))
        self.mid_channels = list(g("mid_channels"))
        self.t_emb_dim = g("time_emb_dim")
        self.down_sample = list(g("down_sample"))
        self.num_down_layers = g("num_down_layers")
        self.num_mid_layers = g("num_mid_layers")
        self.num_up_layers = g("num_up_layers")
        self.attn_resolutions = list(g("attn_resolutions"))
        self.num_heads = g("num_heads")
        self.im_size = g("im_size")
        self.im_channels = g("im_channels")
        assert self.mid_channels[0] == self.down_channels[-1]
        assert self.mid_channels[-1] == self.down_channels[-2]
        assert len(self.down_sample) == len(self.down_channels) - 1
        self._spec = param_spec(model_config)
        for name, shape in self._spec.items():
            init = _init_param(name, shape)
            if init is None:   # bias of a conv / linear: U(-1/sqrt(fan_in), 1/sqrt(fan_in)) of its weight
                wshape = self._spec[name[:-4] + "weight"]
                fan_in = 1
                for s in wshape[1:]:
                    fan_in *= s
                init = torch.empty(shape).uniform_(-1.0 / math.sqrt(fan_in), 1.0 / math.sqrt(fan_in))
            self._register(name, nn.Parameter(init))
        self._infer = PlanPool()      # the inference plan
        self._weights_epoch = 0      # bumped by DenoisingTrainer.optimizer_step (in-place kernel updates of the weights)
        self.differentiable = False  # True: forward under grad mode builds an autograd graph (module docstring)
        self._train_plans = PlanPool()   # (B, H, W) -> training plans: the autograd path's plan pool

    def _register(self, dotted, param):
        node = self
        parts = dotted.split(".")
        for p in parts[:-1]:
            if p not in node._modules:
                node.add_module(p, _Node())
            node = node._modules[p]
        node.register_parameter(parts[-1], param)

    # ---- C handle management ---------------------------------------------------------------------------
    def _config_struct(self):
        c = UnetConfigStruct()
        c.im_channels, c.im_size, c.time_emb_dim = self.im_channels, self.im_size, self.t_emb_dim
        c.num_down_layers, c.num_mid_layers, c.num_up_layers = self.num_down_layers, self.num_mid_layers, self.num_up_layers
        c.num_heads = self.num_heads
        c.n_down_channels = len(self.down_channels)
        c.n_mid_channels = len(self.mid_channels)
        c.n_attn_resolutions = len(self.attn_resolutions)
        for i, v in enumerate(self.down_channels):
            c.down_channels[i] = v
        for i, v in enumerate(self.mid_channels):
            c.mid_channels[i] = v
        for i, v in enumerate(self.down_sample):
            c.down_sample[i] = 1 if v else 0
        for i, v in enumerate(self.attn_resolutions):
            c.attn_resolutions[i] = v
        return c

    def _inference_plan(self, device):
        params = dict(self.named_parameters())
        key = (str(device), self._weights_epoch, tuple((p.data_ptr(), p._version) for p in params.values()))
        return self._infer.one(key, lambda: self._make_inference_plan(params, device))

    def _make_inference_plan(self, params, device):
        tensors = {n: p.detach() for n, p in params.items()}
        names, ptrs, numels = c_tensor_args(tensors, device, "Unet", torch.float32)
        cfg = self._config_struct()
        set_time_factor_table(self.t_emb_dim, device)
        L = lib()
        return PlanHandle(L.wc_unet_create, L.wc_unet_destroy, C.byref(cfg), len(tensors), names, ptrs, numels, stream_ptr(),
                          keep=tensors)

    def _grad_plan(self, B, H, W, device):
        """A free training plan for (B, H, W), created when every plan of that shape is held by a live graph.  Each plan has
        its own workspace and flat fp32 gradient buffer (every tensor's slice 16-byte aligned, as in DenoisingTrainer); it
        reads the module's parameters in place (the backward reads GroupNorm and t-embedding weights)."""
        named = list(self.named_parameters())
        key = (str(device), tuple(p.data_ptr() for _, p in named))
        return self._train_plans.lease(key, (B, H, W), lambda: self._make_train_plan(named, B, H, W, device))

    def _make_train_plan(self, named, B, H, W, device):
        params = {n: p.detach() for n, p in named}
        names, pp, _ = c_tensor_args(params, device, "Unet", torch.float32)
        set_time_factor_table(self.t_emb_dim, device)
        slices, off = [], 0
        for p in params.values():
            off = (off + 3) & ~3
            slices.append((off, p.numel(), p.shape))
            off += p.numel()
        grads = torch.zeros(off, device=device, dtype=torch.float32)
        _, gp, _ = c_tensor_args({n: grads[o:o + k] for n, (o, k, _) in zip(params, slices)}, device, "Unet gradient")
        cfg = self._config_struct()
        L = lib()
        plan = PlanHandle(L.wc_unet_train_create, L.wc_unet_train_destroy, C.byref(cfg), len(params), names, pp, gp,
                          keep=(params, grads))
        plan.grads, plan.slices = grads, slices
        ws = plan.workspace((B, H, W), lambda: L.wc_unet_train_workspace_bytes(plan.handle, B, H, W), device)
        check(L.wc_unet_train_bind(plan.handle, B, H, W, ptr(ws), ws.numel(), stream_ptr()))
        return plan

    # ---- reference API ---------------------------------------------------------------------------------
    def forward(self, x, t, out=None):
        _lib.require_cuda(x)
        x = x.contiguous().float()
        B, Cc, H, W = x.shape
        if Cc != self.im_channels:
            raise RuntimeError(f"expected {self.im_channels} input channels, got {Cc}")
        t = torch.as_tensor(t).long().to(x.device).reshape(-1)     # reference :461
        if t.numel() not in (1, B):
            raise RuntimeError("t must have 1 or batch entries")
        if self.differentiable and torch.is_grad_enabled():
            params = list(self.parameters())
            if x.requires_grad or any(p.requires_grad for p in params):
                if out is not None:
                    raise RuntimeError("Unet.forward: out= cannot be combined with the autograd path "
                                       "(differentiable = True under grad mode)")
                return PlanFunction.apply(self, x, t.expand(B).contiguous(), *params)
        plan = self._inference_plan(x.device)
        ws = plan.workspace((B, H, W), lambda: lib().wc_unet_workspace_bytes(plan.handle, B, H, W), x.device)
        if out is None:
            out = torch.empty_like(x)
        check(lib().wc_unet_forward(plan.handle, ptr(x), ptr(t), t.numel(), ptr(out), B, H, W, ptr(ws), ws.numel(),
                                    stream_ptr()))
        self._last_io = (x, t)   # keep inputs alive until the stream has consumed them
        return out

    def flops_per_forward(self) -> float:
        """Algorithmic FLOPs (2*MAC) of the last bound forward."""
        plan = self._infer.plan
        return float(lib().wc_unet_flops(plan.handle)) if plan is not None else 0.0

    def launches_per_forward(self) -> int:
        plan = self._infer.plan
        return int(lib().wc_unet_launches(plan.handle)) if plan is not None else 0

    # ---- the autograd path (PlanFunction): inputs x [B,3,H,W] fp32, t int64 [B], then every parameter in
    # named_parameters() order
    def _grad_forward(self, plan, x, t, *params):
        pred = torch.empty_like(x)
        check(lib().wc_unet_train_forward(plan.handle, ptr(x), ptr(t), None, ptr(pred), None, 1.0, 1, stream_ptr()))
        return pred

    def _grad_backward(self, plan, g, needs_input_grad, x, t, *params):
        dx = torch.empty_like(x) if needs_input_grad[0] else None
        need = needs_input_grad[2:]
        param_grads = any(need)
        check(lib().wc_unet_train_backward_seeded(plan.handle, ptr(g), ptr(dx), int(param_grads), stream_ptr()))
        grads = [None] * len(need)
        if param_grads:
            # a fresh copy: AccumulateGrad may adopt these views as p.grad, and the plan's buffer is overwritten by the
            # next backward
            flat = plan.grads.clone()
            grads = [flat[o:o + n].view(shape) if nd else None for (o, n, shape), nd in zip(plan.slices, need)]
        return (dx, None, *grads)


_FACTOR_SET = {}


def set_time_factor_table(temb_dim, device):
    """Hand the reference's factor table (reference :22-24, evaluated by torch on the host exactly as written there) to the
    library once per (device, dim): every time-embedding kernel then divides t by the reference's own fp32 factors."""
    key = (str(device), temb_dim)
    if _FACTOR_SET.get("key") == key:
        return
    half = temb_dim // 2
    factor = 10000 ** (torch.arange(start=0, end=half, dtype=torch.float32) / half)
    arr = (C.c_float * half)(*factor.tolist())
    with torch.cuda.device(device):
        check(lib().wc_set_time_factor_table(arr, half))
    _FACTOR_SET["key"] = key


def get_time_embedding(time_steps, temb_dim):
    """Sinusoidal embedding (reference :7-30) as its own kernel (csrc/direct.cu: time_embedding_kernel - the same code
    the UNet plan runs inside temb_mlp_kernel): [B] int tensor on the GPU -> [B, temb_dim] fp32."""
    assert temb_dim % 2 == 0, "time embedding dimension must be divisible by 2"
    _lib.require_cuda(time_steps)
    t = time_steps.long().contiguous().reshape(-1)
    set_time_factor_table(temb_dim, t.device)
    out = torch.empty(t.numel(), temb_dim, device=t.device)
    check(lib().wc_time_embedding(ptr(t), t.numel(), temb_dim, ptr(out), stream_ptr()))
    return out
