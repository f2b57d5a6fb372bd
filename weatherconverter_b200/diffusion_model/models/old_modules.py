"""Legacy UNet with the reference's interface (diffusion_model/models/old_modules.py:230-360) running on libwc_b200.so.

``UNet().forward(x, t)`` takes x [B,3,128,128] fp32 and t [B,1,1,1] fp32 (the noise variance 1 - alpha_bar_t that
sample_integrated.py:60 passes) and returns the predicted noise [B,3,128,128].  ``state_dict()`` has the reference's key
names, shapes and buffers (BatchNorm running statistics), so reference checkpoints load with ``load_state_dict``.
Inference only (eval-mode BatchNorm, as load_model at sample_integrated.py:70-75 sets up); the layer graph and all
arithmetic live in csrc/legacy.cu, and the C handle and its workspace are held through ``_plans.py``.
"""
import math

import torch
import torch.nn as nn

from ... import _lib
from ..._lib import check, lib, ptr, stream_ptr
from ..._plans import PlanHandle, PlanPool, c_tensor_args
from .unet_base import _Node

DEPTH = 3
_DOWN = [("down1", 64, 32), ("down2", 32, 64), ("down3", 64, 96), ("down4", 96, 128)]
_UP = [("up1", 256, 128, 128), ("up2", 128, 96, 96), ("up3", 96, 64, 64), ("up4", 64, 32, 32)]
_SUPPORTED_HD = (16, 32, 64, 128, 192)


def legacy_param_spec():
    """Ordered {name: (shape, dtype)} in the registration order of old_modules.UNet.__init__ (:244-281)."""
    f32, i64 = torch.float32, torch.int64
    spec = {"pre_conv.weight": ((32, 3, 3, 3), f32)}

    def rb(p, cin, cout):
        spec[p + ".res.weight"] = ((cout, cin, 1, 1), f32)
        for k in ("weight", "bias", "running_mean", "running_var"):
            spec[f"{p}.double_conv.0.{k}"] = ((cin,), f32)
        spec[p + ".double_conv.0.num_batches_tracked"] = ((), i64)
        spec[p + ".double_conv.1.weight"] = ((cout, cin, 3, 3), f32)
        spec[p + ".double_conv.3.weight"] = ((cout, cout, 3, 3), f32)

    def attn(p, c):
        spec[p + ".mha.in_proj_weight"] = ((3 * c, c), f32); spec[p + ".mha.in_proj_bias"] = ((3 * c,), f32)
        spec[p + ".mha.out_proj.weight"] = ((c, c), f32); spec[p + ".mha.out_proj.bias"] = ((c,), f32)
        spec[p + ".ln.weight"] = ((c,), f32); spec[p + ".ln.bias"] = ((c,), f32)
        spec[p + ".ff_self.0.weight"] = ((c,), f32); spec[p + ".ff_self.0.bias"] = ((c,), f32)
        spec[p + ".ff_self.1.weight"] = ((c, c), f32); spec[p + ".ff_self.1.bias"] = ((c,), f32)
        spec[p + ".ff_self.3.weight"] = ((c, c), f32); spec[p + ".ff_self.3.bias"] = ((c,), f32)

    for i in range(DEPTH):
        rb(f"down1.residual_blocks.{i}", 64 if i == 0 else 32, 32)
    for i in range(DEPTH):
        rb(f"down2.residual_blocks.{i}", 32 if i == 0 else 64, 64)
    attn("attn_down3", 64)
    for i in range(DEPTH):
        rb(f"down3.residual_blocks.{i}", 64 if i == 0 else 96, 96)
    attn("attn_down4", 96)
    for i in range(DEPTH):
        rb(f"down4.residual_blocks.{i}", 96 if i == 0 else 128, 128)
    rb("bottleneck1", 128, 256)
    attn("attn_bottleneck", 256)
    rb("bottleneck2", 256, 256)
    for name, cin, cout, cskip in _UP:
        for i in range(DEPTH):
            rb(f"{name}.residual_blocks.{i}", (cin if i == 0 else cout) + cskip, cout)
        if name == "up1":
            attn("attn_up1", 128)
        if name == "up2":
            attn("attn_up2", 96)
    spec["output.weight"] = ((3, 32, 3, 3), f32)
    return spec


def _init(name, shape, dtype):
    leaf = name.rsplit(".", 1)[-1]
    if dtype == torch.int64:
        return torch.zeros(shape, dtype=dtype)
    if leaf == "running_mean":
        return torch.zeros(shape)
    if leaf == "running_var":
        return torch.ones(shape)
    if len(shape) == 1:
        if leaf == "weight":
            return torch.ones(shape)
        if leaf == "in_proj_bias" or ".ln." in name or "double_conv.0" in name or name.endswith("out_proj.bias") or ".ff_self.0." in name:
            return torch.zeros(shape)
        fan_in = shape[0]
        return torch.empty(shape).uniform_(-1.0 / math.sqrt(fan_in), 1.0 / math.sqrt(fan_in))
    fan_in = 1
    for s in shape[1:]:
        fan_in *= s
    bound = math.sqrt(6.0 / (shape[0] + shape[1])) if leaf == "in_proj_weight" else 1.0 / math.sqrt(fan_in)
    return torch.empty(shape).uniform_(-bound, bound)


class UNet(nn.Module):
    """Same constructor defaults and forward contract as the reference's old_modules.UNet."""
    requires_alpha_hat_timestep = True

    def __init__(self, c_in=3, c_out=3, image_size=128, conv_dim=64, block_depth=3, time_emb_dim=256):
        super().__init__()
        if (c_in, c_out, image_size, block_depth) != (3, 3, 128, 3):
            raise RuntimeError("the legacy UNet plan is built for c_in = c_out = 3, image_size = 128, block_depth = 3 "
                               "(the reference hard-codes its attention sizes for that geometry, old_modules.py:256-270)")
        self.image_size = image_size
        for name, (shape, dtype) in legacy_param_spec().items():
            t = _init(name, shape, dtype)
            leaf = name.rsplit(".", 1)[-1]
            if leaf in ("running_mean", "running_var", "num_batches_tracked"):
                self._register(name, t, buffer=True)
            else:
                self._register(name, nn.Parameter(t))
        self._infer = PlanPool()

    def _register(self, dotted, tensor, buffer=False):
        node = self
        parts = dotted.split(".")
        for p in parts[:-1]:
            if p not in node._modules:
                node.add_module(p, _Node())
            node = node._modules[p]
        if buffer:
            node.register_buffer(parts[-1], tensor)
        else:
            node.register_parameter(parts[-1], tensor)

    # ---- head-dimension padding: nn.MultiheadAttention(C, 4) has head_dim C/4 in {16, 24, 32, 64}; the tcgen05 attention
    # kernel supports {16, 32, 64, 128, 192}, so each head's q/k/v rows (and the out-projection's columns) are zero-padded
    # to the next supported size.  Zero q/k columns leave every dot product unchanged and zero v rows give zero outputs
    # that meet zero out-projection columns; the softmax scale stays 1/sqrt(C/4) (passed explicitly).
    @staticmethod
    def _pad_attention(sd, prefix, Cc, heads=4):
        hd = Cc // heads
        hdp = next(h for h in _SUPPORTED_HD if h >= hd)
        w, b = sd[prefix + ".mha.in_proj_weight"], sd[prefix + ".mha.in_proj_bias"]
        wo = sd[prefix + ".mha.out_proj.weight"]
        if hdp == hd:
            return w, b, wo
        wp = w.new_zeros(3, heads, hdp, Cc)
        wp[:, :, :hd] = w.view(3, heads, hd, Cc)
        bp = b.new_zeros(3, heads, hdp)
        bp[:, :, :hd] = b.view(3, heads, hd)
        wop = wo.new_zeros(Cc, heads, hdp)
        wop[:, :, :hd] = wo.view(Cc, heads, hd)
        return wp.reshape(3 * heads * hdp, Cc).contiguous(), bp.reshape(-1).contiguous(), wop.reshape(Cc, heads * hdp).contiguous()

    def _inference_plan(self, device):
        sd = {k: v for k, v in self.state_dict().items() if v.dtype == torch.float32}
        key = (str(device), tuple((v.data_ptr(), v._version) for v in sd.values()))
        return self._infer.one(key, lambda: self._make_inference_plan(sd, device))

    def _make_inference_plan(self, sd, device):
        tensors = {k: v.detach().contiguous() for k, v in sd.items()}
        for prefix, Cc in (("attn_down3", 64), ("attn_down4", 96), ("attn_bottleneck", 256), ("attn_up1", 128), ("attn_up2", 96)):
            w, b, wo = self._pad_attention(tensors, prefix, Cc)
            tensors[prefix + ".mha.in_proj_weight"], tensors[prefix + ".mha.in_proj_bias"] = w, b
            tensors[prefix + ".mha.out_proj.weight"] = wo
        names, ptrs, numels = c_tensor_args(tensors, device, "UNet")
        L = lib()
        return PlanHandle(L.wc_legacy_unet_create, L.wc_legacy_unet_destroy, len(tensors), names, ptrs, numels, keep=tensors)

    def forward(self, x, t, out=None):
        _lib.require_cuda(x)
        x = x.contiguous().float()
        B, Cc, H, W = x.shape
        if (Cc, H, W) != (3, self.image_size, self.image_size):
            raise RuntimeError(f"expected [B,3,{self.image_size},{self.image_size}] input, got {tuple(x.shape)}")
        t = torch.as_tensor(t, dtype=torch.float32, device=x.device).reshape(-1).contiguous()
        if t.numel() == 1 and B > 1:
            t = t.expand(B).contiguous()
        if t.numel() != B:
            raise RuntimeError("t must have one entry per sample")
        plan = self._inference_plan(x.device)
        ws = plan.workspace(B, lambda: lib().wc_legacy_unet_workspace_bytes(plan.handle, B, H), x.device)
        if out is None:
            out = torch.empty_like(x)
        check(lib().wc_legacy_unet_forward(plan.handle, ptr(x), ptr(t), ptr(out), B, H, ptr(ws), ws.numel(), stream_ptr()))
        self._last_io = (x, t)
        return out

    def flops_per_forward(self):
        plan = self._infer.plan
        return float(lib().wc_legacy_unet_flops(plan.handle)) if plan is not None else 0.0

    def launches_per_forward(self):
        plan = self._infer.plan
        return int(lib().wc_legacy_unet_launches(plan.handle)) if plan is not None else 0
