"""ctypes binding of libwc_b200.so (the C ABI declared in include/wc_b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is present when a kernel
entry point is called, the call raises.  Build with ``python -c "import __graft_entry__ as g; g.build()"``
(or ``make -C weatherconverter_b200/csrc``).
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libwc_b200.so")

_lib = None

c_f32p = C.c_void_p
c_ptr = C.c_void_p


class UnetConfigStruct(C.Structure):
    _fields_ = [
        ("im_channels", C.c_int), ("im_size", C.c_int), ("time_emb_dim", C.c_int),
        ("num_down_layers", C.c_int), ("num_mid_layers", C.c_int), ("num_up_layers", C.c_int),
        ("num_heads", C.c_int),
        ("n_down_channels", C.c_int), ("down_channels", C.c_int * 8),
        ("n_mid_channels", C.c_int), ("mid_channels", C.c_int * 8),
        ("down_sample", C.c_int * 8),
        ("n_attn_resolutions", C.c_int), ("attn_resolutions", C.c_int * 8),
    ]


_SIGS = {
    "wc_last_error": (C.c_char_p, []),
    "wc_abi_version": (C.c_int, []),
    "wc_launch_count": (C.c_longlong, []),
    "wc_profile_begin": (None, []),
    "wc_profile_detail": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "wc_profile_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_double)]),
    "wc_ddpm_step": (C.c_int, [c_ptr] * 6 + [C.c_size_t, C.c_int] + [C.c_float] * 4 + [c_ptr]),
    "wc_ddpm_step_batched": (C.c_int, [c_ptr] * 6 + [C.c_size_t, C.c_int] + [c_ptr] * 4 + [C.c_int, c_ptr]),
    "wc_ddpm_step_indexed": (C.c_int, [c_ptr] * 6 + [C.c_size_t, C.c_int, c_ptr, c_ptr, C.c_int, c_ptr]),
    "wc_ddim_step": (C.c_int, [c_ptr] * 6 + [C.c_size_t, C.c_int] + [C.c_float] * 5 + [c_ptr]),
    "wc_ddim_step_indexed": (C.c_int, [c_ptr] * 6 + [C.c_size_t, C.c_int, c_ptr, c_ptr, C.c_int, c_ptr]),
    "wc_add_noise": (C.c_int, [c_ptr] * 3 + [C.c_size_t, C.c_int] + [c_ptr] * 3 + [C.c_int, c_ptr]),
    "wc_set_time_factor_table": (C.c_int, [C.POINTER(C.c_float), C.c_int]),
    "wc_time_embedding": (C.c_int, [c_ptr, C.c_int, C.c_int, c_ptr, c_ptr]),
    "wc_sgg_update": (C.c_int, [c_ptr] * 5 + [C.c_int] * 4 + [C.c_float, c_ptr]),
    "wc_lcg_prepare": (C.c_int, [c_ptr] * 4 + [C.c_int] * 4 + [c_ptr]),
    "wc_lcg_combine": (C.c_int, [c_ptr] * 5 + [C.c_int] * 5 + [C.c_float, c_ptr]),
    "wc_groupnorm_workspace_bytes": (C.c_size_t, [C.c_int]),
    "wc_groupnorm_silu": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 5 + [c_ptr, c_ptr, C.c_float, C.c_int, c_ptr, c_ptr]),
    "wc_conv2d": (C.c_int, [c_ptr] + [C.c_int] * 5 + [c_ptr, c_ptr] + [C.c_int] * 6 + [c_ptr, c_ptr, C.c_int, c_ptr,
                            C.c_int, C.c_int, c_ptr, C.c_int, c_ptr, C.c_int, c_ptr]),
    "wc_conv2d_dgrad": (C.c_int, [c_ptr] + [C.c_int] * 4 + [c_ptr] + [C.c_int] * 4 + [c_ptr] * 4),
    "wc_maxpool3x3s2": (C.c_int, [c_ptr] * 3 + [C.c_int] * 4 + [c_ptr]),
    "wc_maxpool3x3s2_bwd": (C.c_int, [c_ptr] * 4 + [C.c_int] * 4 + [c_ptr]),
    "wc_bilinear": (C.c_int, [c_ptr] * 2 + [C.c_int] * 6 + [c_ptr]),
    "wc_bilinear_bwd": (C.c_int, [c_ptr] * 3 + [C.c_int] * 6 + [c_ptr]),
    "wc_seg_loss_head": (C.c_int, [c_ptr] * 8 + [C.c_int] * 5 + [c_ptr]),
    "wc_conv1_dgrad": (C.c_int, [c_ptr] * 4 + [C.c_int] * 3 + [c_ptr]),
    "wc_conv_in": (C.c_int, [c_ptr] * 6 + [C.c_int] * 9 + [c_ptr]),
    "wc_conv_out": (C.c_int, [c_ptr] * 4 + [C.c_int] * 7 + [c_ptr]),
    "wc_nchw_f32_to_nhwc_bf16": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 4 + [c_ptr]),
    "wc_nhwc_bf16_to_nchw_f32": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 4 + [c_ptr]),
    "wc_attention": (C.c_int, [c_ptr] * 4 + [C.c_int] * 5 + [c_ptr]),
    "wc_ddpm_grid_u8": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 5 + [c_ptr]),
    "wc_postprocess_u8": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 3 + [C.POINTER(C.c_float), C.POINTER(C.c_float), c_ptr]),
    "wc_label_encode": (C.c_int, [c_ptr, C.c_int, c_ptr, c_ptr] + [C.c_int] * 4 + [c_ptr, C.c_int, c_ptr, c_ptr]),
    "wc_resample_u8": (C.c_int, [c_ptr] * 3 + [C.c_int] * 5 + [c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, C.c_int, c_ptr]),
    "wc_u8_to_tensor": (C.c_int, [c_ptr] + [C.c_int] * 6 + [C.POINTER(C.c_float), C.POINTER(C.c_float), c_ptr, c_ptr]),
    "wc_attention_lse": (C.c_int, [c_ptr] * 5 + [C.c_int] * 5 + [c_ptr]),
    "wc_attention_scaled": (C.c_int, [c_ptr] * 4 + [C.c_int] * 5 + [C.c_float, c_ptr]),
    "wc_attention_bwd": (C.c_int, [c_ptr] * 8 + [C.c_int] * 4 + [c_ptr]),
    "wc_conv2d_wgrad": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 10 + [c_ptr, C.c_int, c_ptr, c_ptr, c_ptr]),
    "wc_groupnorm_bwd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "wc_groupnorm_silu_bwd": (C.c_int, [c_ptr] * 3 + [C.c_int] * 3 + [c_ptr, c_ptr, C.c_float, C.c_int] + [c_ptr] * 7),
    "wc_colsum": (C.c_int, [c_ptr] + [C.c_int] * 3 + [c_ptr] * 4),
    "wc_mse_loss_grad": (C.c_int, [c_ptr] * 3 + [C.c_size_t, C.c_float, c_ptr, c_ptr, c_ptr]),
    "wc_boundary_wgrad_scratch_bytes": (C.c_size_t, []),
    "wc_boundary_wgrad": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 4 + [c_ptr] * 4),
    "wc_adam_step": (C.c_int, [c_ptr] * 4 + [C.c_size_t] + [C.c_float] * 4 + [C.c_int, C.c_float, c_ptr]),
    "wc_unet_create": (C.c_int, [C.POINTER(c_ptr), C.POINTER(UnetConfigStruct), C.c_int, C.POINTER(C.c_char_p),
                                 C.POINTER(c_ptr), C.POINTER(C.c_int64), c_ptr]),
    "wc_unet_destroy": (None, [c_ptr]),
    "wc_unet_workspace_bytes": (C.c_size_t, [c_ptr, C.c_int, C.c_int, C.c_int]),
    "wc_unet_forward": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, C.c_size_t,
                                  c_ptr]),
    "wc_unet_flops": (C.c_double, [c_ptr]),
    "wc_unet_launches": (C.c_int, [c_ptr]),
    "wc_unet_train_create": (C.c_int, [C.POINTER(c_ptr), C.POINTER(UnetConfigStruct), C.c_int, C.POINTER(C.c_char_p),
                                       C.POINTER(c_ptr), C.POINTER(c_ptr)]),
    "wc_unet_train_destroy": (None, [c_ptr]),
    "wc_unet_train_workspace_bytes": (C.c_size_t, [c_ptr, C.c_int, C.c_int, C.c_int]),
    "wc_unet_train_bind": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, C.c_size_t, c_ptr]),
    "wc_unet_train_forward": (C.c_int, [c_ptr] * 6 + [C.c_float, C.c_int, c_ptr]),
    "wc_unet_train_num_backward_ops": (C.c_int, [c_ptr]),
    "wc_unet_train_backward": (C.c_int, [c_ptr, C.c_int, C.c_int, c_ptr]),
    "wc_unet_train_backward_seeded": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, c_ptr]),
    "wc_unet_train_grad_ready_op": (C.c_int, [c_ptr, C.c_char_p]),
    "wc_unet_train_flops": (C.c_double, [c_ptr, C.c_int]),
    "wc_legacy_unet_create": (C.c_int, [C.POINTER(c_ptr), C.c_int, C.POINTER(C.c_char_p), C.POINTER(c_ptr), C.POINTER(C.c_int64)]),
    "wc_legacy_unet_destroy": (None, [c_ptr]),
    "wc_legacy_unet_workspace_bytes": (C.c_size_t, [c_ptr, C.c_int, C.c_int]),
    "wc_legacy_unet_forward": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, c_ptr, C.c_size_t, c_ptr]),
    "wc_legacy_unet_flops": (C.c_double, [c_ptr]),
    "wc_legacy_unet_launches": (C.c_int, [c_ptr]),
    "wc_seg_create": (C.c_int, [C.POINTER(c_ptr), C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_char_p),
                                C.POINTER(c_ptr), c_ptr]),
    "wc_seg_set_output_stride": (C.c_int, [c_ptr, C.c_int]),
    "wc_seg_destroy": (None, [c_ptr]),
    "wc_seg_workspace_bytes": (C.c_size_t, [c_ptr, C.c_int, C.c_int, C.c_int, C.c_int]),
    "wc_seg_infer": (C.c_int, [c_ptr] * 7 + [C.c_int] * 3 + [c_ptr, C.c_size_t, c_ptr]),
    "wc_seg_infer_pooled": (C.c_int, [c_ptr] * 7 + [C.c_int] * 4 + [c_ptr, C.c_size_t, c_ptr]),
    "wc_seg_forward": (C.c_int, [c_ptr] * 3 + [C.c_int] * 4 + [c_ptr, C.c_size_t, c_ptr]),
    "wc_seg_backward_seeded": (C.c_int, [c_ptr] * 4),
    "wc_seg_flops": (C.c_double, [c_ptr, C.c_int]),
    "wc_seg_launches": (C.c_int, [c_ptr]),
    "wc_srgan_create": (C.c_int, [C.POINTER(c_ptr), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p), C.POINTER(c_ptr), c_ptr]),
    "wc_srgan_destroy": (None, [c_ptr]),
    "wc_srgan_workspace_bytes": (C.c_size_t, [c_ptr, C.c_int, C.c_int, C.c_int]),
    "wc_srgan_forward": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, C.c_size_t, c_ptr]),
    "wc_srgan_grad_workspace_bytes": (C.c_size_t, [c_ptr, C.c_int, C.c_int, C.c_int]),
    "wc_srgan_forward_saved": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, C.c_size_t, c_ptr]),
    "wc_srgan_backward_seeded": (C.c_int, [c_ptr] * 4),
    "wc_srgan_flops": (C.c_double, [c_ptr]),
    "wc_srgan_launches": (C.c_int, [c_ptr]),
}

EXPORTS = tuple(_SIGS.keys())


def lib():
    """Load libwc_b200.so (once) and declare the signatures.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: the CUDA extension has not been built "
                "(run __graft_entry__.build()); this package has no CPU fallback")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().wc_last_error()
        raise RuntimeError("wc_b200: " + (msg.decode() if msg else f"error {rc}"))


def require_cuda(*tensors):
    if not torch.cuda.is_available():
        raise RuntimeError("wc_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("wc_b200 kernels take CUDA tensors; got a tensor on " + str(t.device))


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
