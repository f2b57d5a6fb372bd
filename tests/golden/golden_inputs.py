"""Seeded inputs of the larger golden fixtures, regenerated from their seeds instead of stored.

make_golden.py draws the inputs of these fixtures here and saves only what the reference computed from them, plus a
SHA-256 of the inputs.  The tests' `golden` fixture (tests/conftest.py) draws them again, checks the digest and puts them
back into the loaded dictionary, so the tests see the same keys as before.  A change of the RNG streams therefore fails
loudly instead of comparing the reference's outputs with other inputs.
"""
import hashlib

import numpy as np
import torch


def block_labels(g, B, H, W, blk=8):
    """Cityscapes-shaped label maps: blk x blk blocks of one class in 0..18, 5 % of the blocks ignored (255)."""
    lab = torch.randint(0, 19, (B, H // blk, W // blk), generator=g)
    ign = torch.rand(B, H // blk, W // blk, generator=g) < 0.05
    lab[ign] = 255
    return lab.repeat_interleave(blk, 1).repeat_interleave(blk, 2)


SEG_INFER_CASES = (("resnet50", (64, 128)), ("resnet50", (128, 256)), ("resnet101", (64, 128)))


def seg_infer():
    g = torch.Generator().manual_seed(31)
    out = {}
    for backbone, (H, W) in SEG_INFER_CASES:
        x = torch.rand(1, 3, H, W, generator=g)
        out[f"{backbone}_{H}x{W}"] = dict(x=x, gt=block_labels(g, 1, H, W))
    return out


def seg_conditioned():
    g = torch.Generator().manual_seed(131)
    x = torch.rand(2, 3, 128, 256, generator=g)
    return dict(x=x, gt=block_labels(g, 2, 128, 256))


LEGACY_TRAJ_SAMPLES = 24576      # a quarter of the 2 x 3 x 128 x 128 elements of each trajectory step


def legacy_unet():
    """Inputs of the legacy UNet forward and of the 3-step sample_integrated loop, and `traj_idx`: the fixed sample of
    flattened element indices at which the fixture keeps each step of the reference's trajectory (all of it is 1.2 MB)."""
    g = torch.Generator().manual_seed(91)
    x = torch.randn(2, 3, 128, 128, generator=g)
    xT = torch.randn(2, 3, 128, 128, generator=g)
    zs = torch.stack([torch.randn(2, 3, 128, 128, generator=g) for _ in range(3)])
    idx = torch.randperm(xT.numel(), generator=torch.Generator().manual_seed(92))[:LEGACY_TRAJ_SAMPLES].sort().values
    return dict(x=x, xT=xT, zs=zs, traj_idx=idx)


DIFFUSION_INPUT_SIZES = ((405, 720), (333, 500), (200, 150))


def image_io():
    rng = np.random.default_rng(2024)
    # label ids 0..33 in 16 x 16 blocks at 1080 x 1920, 2 % of the pixels moved to the next id
    lab = np.kron(rng.integers(0, 34, (68, 120), dtype=np.uint8), np.ones((16, 16), dtype=np.uint8))[:1080, :1920]
    lab = (lab + (rng.random(lab.shape) < 0.02) * 1).clip(0, 33).astype(np.uint8)
    img_small = rng.integers(0, 256, (96, 160, 3), dtype=np.uint8)
    diffusion_inputs = []
    for (h, w) in DIFFUSION_INPUT_SIZES:
        im = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        im = np.clip(im // 3 + np.linspace(0, 160, w, dtype=np.int64)[None, :, None], 0, 255).astype(np.uint8)   # ramp + noise
        diffusion_inputs.append(dict(image=torch.from_numpy(im)))
    g = torch.Generator().manual_seed(8)
    ddpm_xt = torch.randn(5, 3, 24, 40, generator=g) * 0.8
    legacy_xt = torch.randn(2, 3, 16, 24, generator=g) * 2.0
    return dict(label_ids=torch.from_numpy(lab), image_small=torch.from_numpy(img_small), diffusion_inputs=diffusion_inputs,
                ddpm_xt=ddpm_xt, legacy_xt=legacy_xt)


REGENERATED = {"seg_infer.pt": seg_infer, "seg_conditioned.pt": seg_conditioned, "legacy_unet.pt": legacy_unet,
               "image_io.pt": image_io}


def digest(tree):
    """SHA-256 over every tensor of a nested dict / list, in key order: name, dtype, shape and bytes."""
    h = hashlib.sha256()

    def walk(o, path):
        if isinstance(o, torch.Tensor):
            t = o.contiguous()
            h.update(f"{path}|{t.dtype}|{tuple(t.shape)}|".encode())
            h.update(t.numpy().tobytes())
        elif isinstance(o, dict):
            for k in sorted(o):
                walk(o[k], f"{path}.{k}")
        elif isinstance(o, (list, tuple)):
            for i, v in enumerate(o):
                walk(v, f"{path}[{i}]")
        else:
            raise TypeError(f"{path}: {type(o).__name__} is not an input tensor")
    walk(tree, "")
    return h.hexdigest()


def _merge(dst, src):
    if isinstance(src, dict):
        for k, v in src.items():
            if k in dst:
                _merge(dst[k], v)
            else:
                dst[k] = v
    else:
        assert isinstance(src, list) and len(src) == len(dst)
        for a, b in zip(dst, src):
            _merge(a, b)


def attach(name, fixture):
    """Put the regenerated inputs back into a loaded fixture (no-op for fixtures that store their inputs)."""
    if name not in REGENERATED:
        return fixture
    inputs = REGENERATED[name]()
    want = fixture.pop("inputs_sha256")
    got = digest(inputs)
    assert got == want, (f"{name}: the regenerated inputs (sha256 {got}) are not the ones the golden outputs were computed "
                         f"from ({want}); the torch / numpy random streams have changed")
    _merge(fixture, inputs)
    return fixture
