"""Pin the CPU oracle against golden vectors produced by the reference's own modules
(tests/golden/make_golden.py).  Runs on CPU; no CUDA involved."""
import torch

from oracle import deeplab, sgg, srgan, unet
from oracle.scheduler import OracleScheduler
from oracle.weights import synth_state_dict


def test_scheduler_tables_exact(golden):
    g = golden("scheduler.pt")
    for T in (1000, 50):
        s = OracleScheduler(T, 1e-4, 0.02)
        for k, v in g[f"tables_{T}"].items():
            assert torch.equal(getattr(s, k), v), k


def test_scheduler_steps(golden):
    g = golden("scheduler.pt")
    s = OracleScheduler(1000, 1e-4, 0.02)
    assert torch.equal(s.add_noise(g["x0"], g["eps"], g["t"]), g["add_noise"])
    assert torch.equal(s.add_noise2(g["x0"], g["eps"], g["t"]), g["add_noise2"])
    for ti, d in g["sample_prev_timestep"].items():
        mean, sz, _ = s.sample_prev_timestep(g["x0"], g["eps"], ti, z=d["z"])
        assert torch.equal(mean, d["mean"])
        if ti == 0:
            assert sz is None and d["sigma_z"] is None
        else:
            assert torch.equal(sz, d["sigma_z"])
    d = g["sample_prev_timestep2"]
    mean, sz, _ = s.sample_prev_timestep2(g["x0"], g["eps"], d["t"], z=d["z"])
    assert torch.equal(mean, d["mean"]) and torch.equal(sz, d["sigma_z"])
    assert torch.equal(unet.get_time_embedding(torch.arange(0, 1000, 37), 128), g["time_embedding"])


def test_unet_forward(golden):
    g = golden("unet_forward.pt")
    for tag, d in g.items():
        sd = synth_state_dict(unet.unet_param_spec(d["cfg"]), d["seed"])
        with torch.no_grad():
            y = unet.unet_forward(sd, d["cfg"], d["x"], d["t"])
        assert (y - d["y"]).abs().max() < 2e-5, tag


def test_sample_trajectory(golden):
    d = golden("sample_traj.pt")
    sd = synth_state_dict(unet.unet_param_spec(d["cfg"]), d["seed"])
    s = OracleScheduler(d["T"], 1e-4, 0.02)
    xt = d["xT"]
    with torch.no_grad():
        for k, i in enumerate(reversed(range(d["T"]))):
            eps = unet.unet_forward(sd, d["cfg"], xt, torch.tensor([i]))
            mean, sz, _ = s.sample_prev_timestep(xt, eps, i, z=d["zs"][i])
            xt = mean + sz if i != 0 else mean
            assert (xt - d["traj"][k]).abs().max() < 1e-3, (k, float((xt - d["traj"][k]).abs().max()))


def test_seg_infer(golden):
    g = golden("seg_infer.pt")
    for tag, d in g.items():
        bb = tag.split("_")[0]
        sd = synth_state_dict(deeplab.deeplab_param_spec(bb), d["seed"])
        taps = {}
        with torch.no_grad():
            deeplab.deeplab_forward(sd, d["x"], bb, taps)
        assert (taps["logits_lowres"] - d["logits_lowres"]).abs().max() < 1e-4, tag
        pred, grad, _ = deeplab.infer(sd, d["x"], d["gt"], bb)
        assert (pred[0].to(torch.uint8) == d["pred"]).float().mean() > 0.9999, tag
        assert (grad - d["grad"]).abs().max() <= 1e-5 * d["grad"].abs().max() + 1e-9, tag


def test_seg_infer_output_stride_8(golden):
    """output_stride = 8 (the reference factories' default argument, modeling.py:182-202): layers 3-4 dilated, ASPP 12/24/36."""
    for tag, d in golden("seg_infer_os8.pt").items():
        sd = synth_state_dict(deeplab.deeplab_param_spec("resnet50"), d["seed"])
        taps = {}
        with torch.no_grad():
            deeplab.deeplab_forward(sd, d["x"], "resnet50", taps, output_stride=8)
        assert (taps["logits_lowres"] - d["logits_lowres"]).abs().max() < 1e-4, tag
        pred, grad, _ = deeplab.infer(sd, d["x"], d["gt"], "resnet50", output_stride=8)
        assert (pred[0].to(torch.uint8) == d["pred"]).float().mean() > 0.9999, tag
        assert (grad - d["grad"]).abs().max() <= 1e-5 * d["grad"].abs().max() + 1e-9, tag


def test_srgan(golden):
    d = golden("srgan.pt")
    sd = synth_state_dict(srgan.srgan_param_spec(), d["seed"])
    with torch.no_grad():
        y = srgan.generator_forward(sd, d["x"])
    assert (y - d["y"]).abs().max() < 1e-5


def test_gsg_and_repaired_driver(golden):
    g = golden("sgg.pt")
    d = g["gsg"]
    seg_sd = synth_state_dict(deeplab.deeplab_param_spec("resnet50"), 42)
    xt, _, _ = sgg.apply_gsg(seg_sd, d["mu"], d["sigma"], d["sr_xt"], d["gt"], d["lam"])
    assert (xt.double() - d["xt"]).abs().max() < 1e-5
    d = g["lcg"]
    xt = sgg.apply_lcg(seg_sd, d["mu"], d["sigma"], d["sr_xt"], d["gt"], d["lam"])
    assert (xt - d["xt"]).abs().max() < 1e-5
    d = g["driver"]
    usd = synth_state_dict(unet.unet_param_spec(d["cfg"]), d["unet_seed"])
    gsd = synth_state_dict(srgan.srgan_param_spec(), d["srgan_seed"])
    rec = []
    out = sgg.sample_with_sgg(usd, d["cfg"], OracleScheduler(1000, 1e-4, 0.02), seg_sd, gsd, d["x0"], d["gt"],
                              d["noise"], d["t_fwd"], list(d["zs"]), lam=60.0, n_steps=d["N"], record=rec)
    assert (torch.stack(rec) - d["traj"]).abs().max() < 1e-3
    assert (out - d["sr_x0"]).abs().max() < 1e-3


def test_train_step(golden):
    """oracle.train.train_step vs the reference's own step (train_ddpm.py:95-114, golden made by make_golden.g_train)."""
    import zlib
    from oracle.train import train_step
    d = golden("train_step.pt")
    sd = synth_state_dict(unet.unet_param_spec(d["cfg"]), d["seed"])
    loss, grads, new_sd = train_step(sd, d["cfg"], d["images"], d["noise"], d["t"], OracleScheduler(1000, 1e-4, 0.02), lr=d["lr"])
    assert abs(float(loss) - float(d["loss"])) < 1e-5 * abs(float(d["loss"]))
    assert set(grads) == set(d["params"])
    for k, ref in d["params"].items():
        g = torch.Generator().manual_seed(zlib.crc32(k.encode()) & 0x7FFFFFFF)
        idx = torch.randint(0, grads[k].numel(), (min(32, grads[k].numel()),), generator=g)
        gn = float(ref["grad_norm"])
        assert abs(float(grads[k].norm()) - gn) <= 2e-3 * gn + 1e-7, k
        assert (grads[k].flatten()[idx] - ref["grad_samples"]).abs().max() <= 2e-3 * gn / grads[k].numel() ** 0.5 * 8 + 1e-7, k
        # Adam's first step moves every weight by ~lr * sign(grad): compare the post-step values
        assert (new_sd[k].flatten()[idx] - ref["new_samples"]).abs().max() < 2.5e-5, k


def test_legacy_unet(golden):
    """oracle.legacy_unet vs the reference's old_modules.UNet (eval) and 3 steps of the sample_integrated loop (the
    trajectory at the fixture's fixed sample of elements, `traj_idx`)."""
    from oracle.legacy_unet import legacy_param_spec, legacy_unet_forward
    d = golden("legacy_unet.pt")
    sd = synth_state_dict(legacy_param_spec(), d["seed"])
    s = OracleScheduler(1000, 1e-4, 0.02)
    with torch.no_grad():
        y = legacy_unet_forward(sd, d["x"], s.one_minus_cum_prod[d["t_idx"]].view(-1, 1, 1, 1))
        assert (y - d["y"]).abs().max() < 2e-4 * d["y"].abs().max(), float((y - d["y"]).abs().max())
        xt = d["xT"]
        for k, i in enumerate(reversed(range(3))):
            t = torch.full((xt.size(0),), i, dtype=torch.long)
            eps = legacy_unet_forward(sd, xt, s.one_minus_cum_prod[t].view(-1, 1, 1, 1))
            mean, sz, _ = s.sample_prev_timestep2(xt, eps, t, z=d["zs"][i])
            xt = mean + sz if i != 0 else mean
            assert (xt.flatten()[d["traj_idx"]] - d["traj"][k]).abs().max() < 1e-3 * d["traj"][k].abs().max(), k


def test_image_io(golden):
    """oracle.image_io (numpy restatement incl. Pillow's resampling) vs tensors produced by the reference's own transforms."""
    import numpy as np
    from oracle import image_io as io
    d = golden("image_io.pt")
    enc = io.encode_label(d["label_ids"].numpy())
    assert np.array_equal(enc, d["encoded_label"].numpy().astype(np.int64))
    assert np.array_equal(io.normalize_image(d["image_small"].numpy()), d["normalized"].numpy())
    for e in d["diffusion_inputs"]:
        assert np.array_equal(io.diffusion_input(e["image"].numpy()), e["tensor"].numpy())
    assert np.array_equal(io.ddpm_grid_uint8(d["ddpm_xt"].numpy(), 2), d["ddpm_grid"].numpy())
    assert np.array_equal(io.ddpm_grid_uint8(d["ddpm_xt"].numpy()[:1], 2), d["ddpm_grid_single"].numpy())
    assert np.array_equal(io.postprocess_uint8(d["legacy_xt"].numpy()), d["legacy_u8"].numpy())
