"""Generate the golden fixtures in tests/golden/*.pt from the UNMODIFIED reference.

Runs only where /root/reference exists (the build container):
    python tests/golden/make_golden.py
Every tensor below is produced by the reference's own modules/functions (imported through
ref_shim); the oracle is NOT involved.  Weights come from oracle.weights.synth_state_dict, a pure
function of (name, shape, seed), loaded into the reference modules with load_state_dict.  The seeded
inputs of the larger fixtures come from golden_inputs.py and are not stored (see there).
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402

ref_shim.install()
import io  # noqa: E402
import contextlib  # noqa: E402
import lzma  # noqa: E402
import torch  # noqa: E402
import golden_inputs  # noqa: E402
from golden_inputs import block_labels  # noqa: E402
from oracle.weights import synth_state_dict  # noqa: E402
from oracle.unet import DEFAULT_MODEL_CONFIG  # noqa: E402

from diffusion_model.models.unet_base import Unet, get_time_embedding  # noqa: E402
from diffusion_model.config.models import ModelConfig  # noqa: E402
from diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler  # noqa: E402
import seg_model.network as network  # noqa: E402
import seg_model.inference as seg_infer  # noqa: E402
from srgan_model.models import Generator  # noqa: E402
import srgan_model.inference as srgan_infer  # noqa: E402
from sgg.sgg import apply_gsg  # noqa: E402

torch.set_num_threads(os.cpu_count())


def _drop_inputs(obj, inputs):
    for k, v in inputs.items() if isinstance(inputs, dict) else enumerate(inputs):
        if isinstance(v, torch.Tensor):
            obj.pop(k, None)
        else:
            _drop_inputs(obj[k], v)


def save(name, obj, inputs=None, xz=False):
    """With `inputs` (drawn by golden_inputs.py) the fixture keeps their digest instead of the tensors; `xz` compresses it."""
    if inputs is not None:
        _drop_inputs(obj, inputs)
        obj["inputs_sha256"] = golden_inputs.digest(inputs)
    path = os.path.join(HERE, name)
    if xz:
        buf = io.BytesIO()
        torch.save(obj, buf)
        path += ".xz"
        with open(path, "wb") as f:
            f.write(lzma.compress(buf.getvalue(), preset=9))
    else:
        torch.save(obj, path)
    print(f"{os.path.basename(path)}: {os.path.getsize(path) / 1024:.0f} KiB")


class InjectedRandn:
    """Patch torch.randn so the scheduler's CPU draw (scheduler.py:110) returns a recorded tensor."""

    def __init__(self, zs):
        self.zs, self.i, self.orig = list(zs), 0, torch.randn

    def __enter__(self):
        def fake(*a, **k):
            z = self.zs[self.i]; self.i += 1
            return z.clone()
        torch.randn = fake
        return self

    def __exit__(self, *a):
        torch.randn = self.orig


def g_scheduler():
    out = {}
    for T in (1000, 50):
        s = LinearNoiseScheduler(T, 1e-4, 0.02)
        out[f"tables_{T}"] = {k: getattr(s, k).clone() for k in (
            "betas", "alphas", "alpha_cum_prod", "sqrt_alpha_cum_prod", "one_minus_cum_prod",
            "sqrt_one_minus_alpha_cum_prod")}
    s = LinearNoiseScheduler(1000, 1e-4, 0.02)
    g = torch.Generator().manual_seed(11)
    x0 = torch.rand(3, 3, 8, 16, generator=g) * 2 - 1
    eps = torch.randn(3, 3, 8, 16, generator=g)
    t = torch.tensor([0, 499, 999])
    out["x0"], out["eps"], out["t"] = x0, eps, t
    out["add_noise"] = s.add_noise(x0, eps, t)
    out["add_noise2"] = s.add_noise2(x0, eps, t)
    steps = {}
    for ti in (0, 1, 10, 499, 999):
        z = torch.randn(3, 3, 8, 16, generator=g)
        with InjectedRandn([z]):
            mean, sig, _ = s.sample_prev_timestep(x0, eps, torch.as_tensor(ti))
        steps[ti] = dict(z=z, mean=mean, sigma_z=sig)
    out["sample_prev_timestep"] = steps
    tb = torch.tensor([0, 5, 999])
    z = torch.randn(3, 3, 8, 16, generator=g)
    with InjectedRandn([z]):
        mean, sig, _ = s.sample_prev_timestep2(x0, eps, tb)
    out["sample_prev_timestep2"] = dict(t=tb, z=z, mean=mean, sigma_z=sig)
    out["time_embedding"] = get_time_embedding(torch.arange(0, 1000, 37), 128)
    save("scheduler.pt", out)


def unet_for(cfg, seed):
    m = Unet(ModelConfig(**cfg)).eval()
    sd = synth_state_dict(m.state_dict(), seed)
    m.load_state_dict(sd)
    return m


def g_unet():
    out = {}
    g = torch.Generator().manual_seed(5)
    for tag, ims, shape, t in (("im64_b2_64x64", 64, (2, 3, 64, 64), [7]),
                               ("im128_b2_32x64", 128, (2, 3, 32, 64), [3, 500]),
                               ("im128_b1_64x128", 128, (1, 3, 64, 128), [999])):
        cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = ims
        m = unet_for(cfg, 3455)
        x = torch.randn(shape, generator=g)
        with torch.no_grad():
            y = m(x, torch.tensor(t))
        out[tag] = dict(cfg=cfg, seed=3455, x=x, t=torch.tensor(t), y=y)
        print(tag, float(y.std()))
    save("unet_forward.pt", out)


def g_sample():
    """sample_ddpm.sample loop (sample_ddpm.py:35-44) B=2, 32x32, T=12, im_size=64, recorded noise."""
    cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = 64
    m = unet_for(cfg, 3455)
    T = 12
    s = LinearNoiseScheduler(T, 1e-4, 0.02)
    g = torch.Generator().manual_seed(21)
    xT = torch.randn(2, 3, 32, 32, generator=g)
    zs = [torch.randn(2, 3, 32, 32, generator=g) for _ in range(T)]
    traj = []
    xt = xT
    with torch.no_grad():
        for i in reversed(range(T)):
            eps = m(xt, torch.as_tensor(i).unsqueeze(0))
            with InjectedRandn([zs[i]]):
                mean, sigma, _ = s.sample_prev_timestep(xt, eps, torch.as_tensor(i))
            xt = mean + sigma if i != 0 else mean
            traj.append(xt.clone())
    save("sample_traj.pt", dict(cfg=cfg, seed=3455, T=T, xT=xT, zs=torch.stack(zs), traj=torch.stack(traj)))


def seg_for(backbone, seed, output_stride=16):
    m = network.modeling.__dict__["deeplabv3plus_" + backbone](num_classes=19, output_stride=output_stride,
                                                               pretrained_backbone=False).eval()
    sd = synth_state_dict(m.state_dict(), seed)
    m.load_state_dict(sd)
    return m


def g_seg():
    out = {}
    inputs = golden_inputs.seg_infer()
    for backbone, (H, W) in golden_inputs.SEG_INFER_CASES:
        m = seg_for(backbone, 42)
        x, gt = inputs[f"{backbone}_{H}x{W}"]["x"], inputs[f"{backbone}_{H}x{W}"]["gt"]
        feats = {}
        hook = m.classifier.classifier.register_forward_hook(lambda mod, i, o: feats.__setitem__("low", o.detach()))
        with contextlib.redirect_stdout(io.StringIO()):
            pred, grad, _ = seg_infer.infer(m, x.clone(), gt)
        hook.remove()
        out[f"{backbone}_{H}x{W}"] = dict(seed=42, x=x, gt=gt, logits_lowres=feats["low"],
                                           pred=torch.from_numpy(pred).to(torch.uint8), grad=grad.detach().clone())
        print(backbone, H, W, float(grad.abs().max()))
    save("seg_infer.pt", out, inputs)
    g_seg_os8()


def g_seg_os8():
    """output_stride = 8, the default argument of the reference factories (modeling.py:182-202): layers 3 and 4 dilated, ASPP
    rates 12 / 24 / 36."""
    g = torch.Generator().manual_seed(33)
    H, W = 64, 128
    m = seg_for("resnet50", 42, output_stride=8)
    x = torch.rand(1, 3, H, W, generator=g)
    gt = block_labels(g, 1, H, W)
    feats = {}
    hook = m.classifier.classifier.register_forward_hook(lambda mod, i, o: feats.__setitem__("low", o.detach()))
    with contextlib.redirect_stdout(io.StringIO()):
        pred, grad, _ = seg_infer.infer(m, x.clone(), gt)
    hook.remove()
    save("seg_infer_os8.pt", {"resnet50_os8_64x128": dict(seed=42, output_stride=8, x=x, gt=gt, logits_lowres=feats["low"],
                                                           pred=torch.from_numpy(pred).to(torch.uint8), grad=grad.detach().clone())})


def g_seg_conditioned():
    """DeepLabV3+-R50 input gradient on a WELL-CONDITIONED fixture: the last BatchNorm scale of every bottleneck (bn3.weight)
    is multiplied by 0.2, i.e. residual branches are small corrections of the identity path as in a trained ResNet
    (zero_init_residual training recipes start them at 0).  The plain random-init net of seg_infer.pt is chaotic at bf16
    resolution (DESIGN.md section 4); this one is not, so the gradient tolerance can be tight."""
    inputs = golden_inputs.seg_conditioned()
    m = network.modeling.deeplabv3plus_resnet50(num_classes=19, output_stride=16, pretrained_backbone=False).eval()
    sd = synth_state_dict(m.state_dict(), 42)
    for k in sd:
        if k.endswith("bn3.weight"):
            sd[k] = sd[k] * 0.2
    m.load_state_dict(sd)
    x, gt = inputs["x"], inputs["gt"]
    preds, grads = [], []
    for b in range(2):
        with contextlib.redirect_stdout(io.StringIO()):
            pred, grad, _ = seg_infer.infer(m, x[b:b + 1].clone(), gt[b:b + 1])
        preds.append(torch.from_numpy(pred).to(torch.uint8)); grads.append(grad.detach().clone())
    save("seg_conditioned.pt", dict(seed=42, bn3_gain=0.2, x=x, gt=gt, pred=torch.stack(preds), grad=torch.cat(grads)), inputs)


def g_srgan():
    G = Generator(upscale_factor=4).eval()
    sd = synth_state_dict(G.state_dict(), 0)
    G.load_state_dict(sd)
    g = torch.Generator().manual_seed(41)
    x = torch.rand(2, 3, 16, 32, generator=g) * 2 - 1
    y = srgan_infer.inference(G, x)
    save("srgan.pt", dict(seed=0, x=x, y=y))
    return G


def g_gsg_and_driver(G):
    """apply_gsg (sgg.py:9-24) on one image and the repaired sample_with_sgg driver (SURVEY 8c) for 3 steps."""
    out = {}
    g = torch.Generator().manual_seed(51)
    seg = seg_for("resnet50", 42)
    h, w = 16, 32
    mu = torch.randn(1, 3, h, w, generator=g)
    sig = 0.1 * torch.randn(1, 3, h, w, generator=g)
    sr = torch.rand(1, 3, 4 * h, 4 * w, generator=g)
    gt = block_labels(g, 1, 4 * h, 4 * w)
    with contextlib.redirect_stdout(io.StringIO()):
        xt = apply_gsg(seg, mu, sig, sr.clone(), gt, 60.0)
    out["gsg"] = dict(mu=mu, sigma=sig, sr_xt=sr, gt=gt, lam=60.0, xt=xt)       # xt is float64 (D7)
    # repaired LCG (sgg.py:27-60 per-class body verbatim through the reference's infer / compute_gradient_magnitude;
    # final masked sum repaired as documented in oracle/sgg.py:apply_lcg)
    import torch.nn.functional as F
    acc = torch.zeros(h, w, dtype=torch.float64)
    with contextlib.redirect_stdout(io.StringIO()):
        for c in range(19):
            mc = (gt == c).long().unsqueeze(1)
            xm = (sr * mc).clone()
            gm = gt * mc.squeeze(0)
            _, gr, _ = seg_infer.infer(seg, xm, gm)
            mag = seg_infer.compute_gradient_magnitude(F.avg_pool2d(gr, 4, 4), denormalize=True, norm=False)
            acc = acc + F.avg_pool2d(mc.float(), 4, 4)[0, 0].double() * mag
    out["lcg"] = dict(mu=mu, sigma=sig, sr_xt=sr, gt=gt, lam=60.0, xt=((mu + 60.0 * sig * acc) + sig).float())
    # repaired driver
    cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = 64
    m = unet_for(cfg, 3455)

    def lcg_repaired(mu_, sigma_, sr_xt):
        """sgg.py:39-54 per-class body through the reference's own infer / compute_gradient_magnitude, final sum repaired as
        documented in oracle/sgg.py:apply_lcg."""
        acc_ = torch.zeros(h, w, dtype=torch.float64)
        for c in range(19):
            mc = (gt == c).long().unsqueeze(1)
            _, gr, _ = seg_infer.infer(seg, (sr_xt * mc).clone(), gt * mc.squeeze(0))
            mag = seg_infer.compute_gradient_magnitude(F.avg_pool2d(gr, 4, 4), denormalize=True, norm=False)
            acc_ = acc_ + F.avg_pool2d(mc.float(), 4, 4)[0, 0].double() * mag
        return ((mu_ + 60.0 * sigma_ * acc_) + sigma_).float()

    def run_driver(N, mode):
        """Repaired driver (SURVEY 8c).  mode 'gsg': GSG on every step; 'alternate': the shipped schedule of
        translation.py:84-87 (LCG when i is even, GSG when i is odd).  Records x_t and the unguided mu + sigma per step."""
        g2 = torch.Generator().manual_seed(52 if mode == "gsg" else 53)
        x0 = torch.rand(1, 3, h, w, generator=g2) * 2 - 1
        noise = torch.randn(1, 3, h, w, generator=g2)
        t_fwd = torch.tensor([N - 1])
        zs = [torch.randn(1, 3, h, w, generator=g2) for _ in range(N)]
        traj, base = [], []
        with torch.no_grad():
            xt = s.add_noise2(x0, noise, t_fwd)
            for i in reversed(range(N)):
                eps = m(xt, torch.as_tensor(i).unsqueeze(0))
                with InjectedRandn([zs[i]]):
                    mu_, sigma_, _ = s.sample_prev_timestep(xt, eps, torch.as_tensor(i))
                if i == 0:
                    xt = mu_
                    base.append(mu_.clone())
                else:
                    base.append(mu_ + sigma_)
                    sr_xt = srgan_infer.inference(G, xt)
                    with torch.enable_grad(), contextlib.redirect_stdout(io.StringIO()):
                        if mode == "alternate" and i % 2 == 0:
                            xt = lcg_repaired(mu_, sigma_, sr_xt)
                        else:
                            xt = apply_gsg(seg, mu_, sigma_, sr_xt, gt, 60.0).float()
                traj.append(xt.clone())
            sr_x0 = srgan_infer.inference(G, xt)
            # segmentation argmax of the FINAL image (north-star: label maps of the final images)
            final_pred = seg(sr_x0).argmax(1).to(torch.uint8)
        return dict(cfg=cfg, unet_seed=3455, seg_seed=42, srgan_seed=0, N=N, x0=x0, noise=noise, t_fwd=t_fwd, mode=mode,
                    zs=torch.stack(zs), gt=gt, traj=torch.stack(traj), base=torch.stack(base), sr_x0=sr_x0, final_pred=final_pred)

    s = LinearNoiseScheduler(1000, 1e-4, 0.02)
    out["driver"] = run_driver(3, "gsg")
    out["driver_alternate"] = run_driver(5, "alternate")
    save("sgg.pt", out)


def sample_idx(name, numel, k=32):
    """Fixed pseudo-random element indices of a parameter (shared with tests/test_oracle_golden.py)."""
    import zlib
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()) & 0x7FFFFFFF)
    return torch.randint(0, numel, (min(k, numel),), generator=g)


def g_train():
    """One training step exactly as train_ddpm.py:95-114 runs it (add_noise -> model -> MSELoss -> backward ->
    Adam(lr=1e-4).step()), B=2, 64x64, im_size=64.  The full gradients are 110 M floats, so the fixture keeps the loss,
    every parameter's gradient norm and 32 sampled entries of its gradient and of its post-step value."""
    cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = 64
    m = unet_for(cfg, 3455).train()
    sched = LinearNoiseScheduler(1000, 1e-4, 0.02)
    g = torch.Generator().manual_seed(77)
    images = torch.rand(2, 3, 64, 64, generator=g) * 2 - 1
    noise = torch.randn(2, 3, 64, 64, generator=g)
    t = torch.tensor([37, 811])
    opt = torch.optim.Adam(m.parameters(), lr=1e-4)
    crit = torch.nn.MSELoss()
    opt.zero_grad()
    noisy = sched.add_noise(images, noise, t)
    pred = m(noisy, t)
    loss = crit(pred, noise)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in m.named_parameters()}
    opt.step()
    out = dict(cfg=cfg, seed=3455, images=images, noise=noise, t=t, loss=loss.detach(), pred=pred.detach(), lr=1e-4, params={})
    for k, p in m.named_parameters():
        idx = sample_idx(k, p.numel())
        out["params"][k] = dict(grad_norm=grads[k].norm(), grad_sum=grads[k].double().sum().float(),
                                grad_samples=grads[k].flatten()[idx].clone(), new_samples=p.detach().flatten()[idx].clone())
    save("train_step.pt", out)


def g_legacy():
    """Legacy old_modules.UNet (eval) forward, B=2, and 3 steps of the sample_integrated loop (sample_integrated.py:52-65)
    with recorded noise; each trajectory step is kept at the fixed element sample golden_inputs.legacy_unet()["traj_idx"]."""
    from diffusion_model.models.old_modules import UNet as LegacyUNet
    m = LegacyUNet().eval()
    sd = synth_state_dict(m.state_dict(), 21)
    m.load_state_dict(sd)
    sched = LinearNoiseScheduler(1000, 1e-4, 0.02)
    inputs = golden_inputs.legacy_unet()
    x = inputs["x"]
    t_idx = torch.tensor([40, 900])
    out = dict(seed=21, x=x, t_idx=t_idx)
    with torch.no_grad():
        out["y"] = m(x, sched.one_minus_cum_prod[t_idx].view(-1, 1, 1, 1))
        T = 3
        xt, zs = inputs["xT"].clone(), inputs["zs"]
        out["xT"], out["zs"], traj = xt.clone(), zs, []
        for i in reversed(range(T)):
            t = torch.full((xt.size(0),), i, dtype=torch.long)
            noise_pred = m(xt, sched.one_minus_cum_prod[t].view(-1, 1, 1, 1))
            with InjectedRandn([zs[i]]):
                mean, sigma, _ = sched.sample_prev_timestep2(xt, noise_pred, t)
            xt = mean + sigma if i != 0 else mean
            traj.append(xt.clone())
        out["traj"] = torch.stack(traj).flatten(1)[:, inputs["traj_idx"]].clone()
    save("legacy_unet.pt", out, inputs)


def g_io():
    """Image / label edges, produced by the reference's own transforms (seg_model/utils/ext_transforms.py,
    acdc.encode_target, sample_integrated.postprocess) and by the exact PIL / torchvision calls of translation.py:138-145
    and sample_ddpm.py:47-51."""
    import numpy as np
    from PIL import Image
    import torchvision
    from torchvision import transforms
    from torchvision.utils import make_grid
    from seg_model.datasets.acdc import ACDCDataset
    from seg_model.utils.ext_transforms import ExtCompose, ExtResize, ExtCenterCrop, ExtToTensor, ExtNormalize
    from diffusion_model.sample_integrated import postprocess
    inputs = golden_inputs.image_io()
    out = {}
    # --- seg preprocessing (inference.py:75-82,103-104): label ids 0..33 in 16x16 blocks + a small image
    lab, img_small = inputs["label_ids"].numpy(), inputs["image_small"].numpy()
    val_transform = ExtCompose([ExtResize(size=(1080 // 2, 1920 // 2), interpolation=Image.BILINEAR, just_label=True),
                                ExtCenterCrop(size=(512, 512), just_label=True), ExtToTensor(),
                                ExtNormalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    input_tensor, lbl_tensor = val_transform(Image.fromarray(img_small), Image.fromarray(lab))
    enc = torch.from_numpy(np.array(ACDCDataset.encode_target(lbl_tensor))).unsqueeze(0).long()
    out["label_ids"] = torch.from_numpy(lab)
    out["encoded_label"] = enc.to(torch.uint8)            # train ids 0..18 / 255 fit a byte (kept small)
    out["image_small"] = torch.from_numpy(img_small)
    out["normalized"] = input_tensor.unsqueeze(0)
    # --- diffusion input (translation.py:138-145)
    tf = transforms.Compose([transforms.Resize(128, transforms.InterpolationMode.BILINEAR), transforms.CenterCrop(128),
                             transforms.ToTensor(), transforms.Lambda(lambd=lambda x: x * 2.0 - 1.0)])
    out["diffusion_inputs"] = []
    for e in inputs["diffusion_inputs"]:
        im = e["image"].numpy()
        out["diffusion_inputs"].append(dict(image=torch.from_numpy(im), tensor=tf(Image.fromarray(im)).unsqueeze(0)))
    # --- sample_ddpm.py:47-51
    xt = inputs["ddpm_xt"]
    ims = torch.clamp(xt, -1., 1.).detach().cpu()
    ims = (ims + 1) / 2
    grid = make_grid(ims, nrow=2)
    img = torchvision.transforms.ToPILImage()(grid)
    out["ddpm_xt"], out["ddpm_grid"] = xt, torch.from_numpy(np.array(img))
    grid1 = make_grid(ims[:1], nrow=2)
    out["ddpm_grid_single"] = torch.from_numpy(np.array(torchvision.transforms.ToPILImage()(grid1)))
    # --- sample_integrated.postprocess
    xl = inputs["legacy_xt"]
    out["legacy_xt"], out["legacy_u8"] = xl, postprocess(xl)
    save("image_io.pt", out, inputs, xz=True)


if __name__ == "__main__":
    only = sys.argv[1:]
    if only == ["io"]:
        g_io()
        sys.exit(0)
    if only == ["train"]:
        g_train()
        sys.exit(0)
    if only == ["legacy"]:
        g_legacy()
        sys.exit(0)
    if only == ["seg_os8"]:
        g_seg_os8()
        sys.exit(0)
    if only == ["sgg"]:
        g_gsg_and_driver(g_srgan())
        g_seg_conditioned()
        sys.exit(0)
    g_scheduler()
    g_unet()
    g_sample()
    g_seg()
    g_seg_conditioned()
    G = g_srgan()
    g_gsg_and_driver(G)
    g_train()
    g_legacy()
    g_io()
