"""CPU tests of the C plans' workspace queries: every plan handle is created with a dummy parameter table (a workspace query
is a dry build, which reads no parameter and touches no device), and the workspace each plan needs at the bench geometries
is pinned, so that a change to how a plan lays out its workspace shows up without a GPU."""
import ctypes as C

import pytest

import __graft_entry__
from weatherconverter_b200 import _lib

# (batch, H, W) of the bench workloads (bench.py WORKLOADS): UNet latents, segmentor inputs (4x the latent), SRGAN inputs
UNET = {"c1": (64, 4, 64, 64), "c3": (64, 32, 64, 128), "c2": (128, 16, 128, 256), "ref": (128, 1, 128, 128)}
UNET_TRAIN_C5 = (128, 64, 128, 256)

EXPECTED = {
    "unet": {"c1": 241_721_344, "c3": 3_866_267_648, "c2": 5_314_793_472, "ref": 166_110_208},
    "unet_train_c5": 44_128_971_008,
    # (backbone, batch, H, W, output_stride) -> (without, with input gradient)
    "seg": {("resnet50", 32, 256, 512, 16): (2_923_581_568, 5_540_974_848),
            ("resnet50", 32, 256, 512, 8): (5_163_339_904, 9_819_164_928),
            ("resnet101", 1, 512, 512, 16): (236_200_452, 453_260_544),
            ("resnet101", 1, 512, 512, 8): (536_617_476, 1_041_511_680)},
    # SRGAN x4 (batch, h, w) -> (plain, with input gradient)
    "srgan": {(32, 64, 128): (2_264_928_256, 5_083_500_544), (1, 128, 128): (141_561_856, 317_722_624)},
    "legacy_b4": 205_197_312,
}


@pytest.fixture(scope="module")
def L():
    __graft_entry__.build()
    return _lib.lib()


def dummy_params():
    """A one-entry parameter table with a non-null pointer no dry build may read."""
    return 1, (C.c_char_p * 1)(b"unused"), (C.c_void_p * 1)(4096), (C.c_int64 * 1)(1)


def unet_config(im_size):
    from weatherconverter_b200.diffusion_model.config.models import ModelConfig
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet
    return Unet(ModelConfig(im_size=im_size))._config_struct()


def create(L, fn, *args):
    h = C.c_void_p()
    assert fn(C.byref(h), *args) == 0, L.wc_last_error()
    return h


def workspaces(L):
    n, names, ptrs, numels = dummy_params()
    out = {"unet": {}}
    for name, (im, B, H, W) in UNET.items():
        cfg = unet_config(im)
        h = create(L, L.wc_unet_create, C.byref(cfg), n, names, ptrs, numels, None)
        out["unet"][name] = L.wc_unet_workspace_bytes(h, B, H, W)
        L.wc_unet_destroy(h)
    im, B, H, W = UNET_TRAIN_C5
    cfg = unet_config(im)
    h = create(L, L.wc_unet_train_create, C.byref(cfg), n, names, ptrs, ptrs)
    out["unet_train_c5"] = L.wc_unet_train_workspace_bytes(h, B, H, W)
    L.wc_unet_train_destroy(h)
    out["seg"] = {}
    for backbone, blocks, B, H, W in (("resnet50", (3, 4, 6, 3), 32, 256, 512), ("resnet101", (3, 4, 23, 3), 1, 512, 512)):
        h = create(L, L.wc_seg_create, (C.c_int * 4)(*blocks), 19, n, names, ptrs, None)
        for os_ in (16, 8):
            assert L.wc_seg_set_output_stride(h, os_) == 0
            out["seg"][(backbone, B, H, W, os_)] = tuple(L.wc_seg_workspace_bytes(h, B, H, W, g) for g in (0, 1))
        L.wc_seg_destroy(h)
    out["srgan"] = {}
    h = create(L, L.wc_srgan_create, 16, 4, n, names, ptrs, None)
    for B, hh, ww in ((32, 64, 128), (1, 128, 128)):
        out["srgan"][(B, hh, ww)] = (L.wc_srgan_workspace_bytes(h, B, hh, ww), L.wc_srgan_grad_workspace_bytes(h, B, hh, ww))
    L.wc_srgan_destroy(h)
    h = create(L, L.wc_legacy_unet_create, n, names, ptrs, numels)
    out["legacy_b4"] = L.wc_legacy_unet_workspace_bytes(h, 4, 128)
    L.wc_legacy_unet_destroy(h)
    return out


def test_unet_create_needs_no_device(L):
    n, names, ptrs, numels = dummy_params()
    cfg = unet_config(64)
    h = create(L, L.wc_unet_create, C.byref(cfg), n, names, ptrs, numels, None)
    L.wc_unet_destroy(h)


def test_workspace_bytes_at_the_bench_geometries(L):
    assert workspaces(L) == EXPECTED


def test_workspace_query_leaves_the_handle_unbound(L):
    """A query is a dry build: it records no op, so the handle still reports no plan."""
    n, names, ptrs, numels = dummy_params()
    h = create(L, L.wc_srgan_create, 16, 4, n, names, ptrs, None)
    assert L.wc_srgan_grad_workspace_bytes(h, 2, 32, 32) > 0
    assert L.wc_srgan_launches(h) == 0 and L.wc_srgan_flops(h) == 0.0
    L.wc_srgan_destroy(h)
