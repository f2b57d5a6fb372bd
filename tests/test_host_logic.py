"""CPU tests: C-ABI library loads and exports every declared symbol, host-side logic, product/oracle separation,
world_size-2 gloo run of the sharding path."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    ge.build()
    from weatherconverter_b200 import _lib
    handle = _lib.lib()
    header = open(os.path.join(ROOT, "include", "wc_b200.h")).read()
    declared = set(re.findall(r"\b(wc_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/wc_b200.h but not exported"
    assert set(_lib.EXPORTS) <= declared
    assert handle.wc_abi_version() >= 1


def test_product_fails_loudly_without_cuda():
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    from weatherconverter_b200 import ops
    with pytest.raises(RuntimeError):
        ops.to_nhwc_bf16(torch.zeros(1, 8, 4, 4))
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet
    from weatherconverter_b200.diffusion_model.config.models import ModelConfig
    m = Unet(ModelConfig(down_channels=[64, 64], mid_channels=[64, 64], down_sample=[True], im_size=16,
                         attn_resolutions=[8]))
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 16, 16), torch.tensor([1]))


def test_no_oracle_in_product():
    bad = []
    for dp, _, fns in os.walk(os.path.join(ROOT, "weatherconverter_b200")):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, fn)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M) or "oracle/" in src:
                    bad.append(os.path.join(dp, fn))
    assert not bad, bad


def test_no_environment_switches():
    """The library reads no environment variables: every tuning choice is fixed in the code (DESIGN.md section 8)."""
    bad = []
    for dp, _, fns in os.walk(os.path.join(ROOT, "weatherconverter_b200")):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, fn)).read()
                if re.search(r"\bgetenv\s*\(|\bos\.environ\b|\bos\.getenv\b", src):
                    bad.append(os.path.join(dp, fn))
    assert not bad, bad


def test_unet_state_dict_matches_oracle_spec():
    from oracle.unet import DEFAULT_MODEL_CONFIG, unet_param_spec
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet, param_spec
    for ims in (64, 128):
        cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = ims
        a, b = param_spec(cfg), unet_param_spec(cfg)
        assert set(a) == set(b)
        assert all(tuple(a[k]) == tuple(b[k][0]) for k in a)
    m = Unet(cfg)
    sd = m.state_dict()
    assert len(sd) == 382 and sum(v.numel() for v in sd.values()) == 110638339
    assert list(sd.keys()) == list(param_spec(cfg).keys())


def test_scheduler_tables_and_coefficients(golden):
    from oracle.scheduler import OracleScheduler
    from weatherconverter_b200.diffusion_model.scheduler.linear_noise_scheduler import LinearNoiseScheduler
    g = golden("scheduler.pt")
    for T in (1000, 50):
        s = LinearNoiseScheduler(T, 1e-4, 0.02)
        for k, v in g[f"tables_{T}"].items():
            assert torch.equal(getattr(s, k).cpu(), v), k
    s, o = LinearNoiseScheduler(1000, 1e-4, 0.02), OracleScheduler(1000, 1e-4, 0.02)
    for t in range(1, 1000):   # vectorised host coefficients == the reference's per-step 0-d tensor arithmetic
        var = (1 - o.alpha_cum_prod[t - 1]) / (1.0 - o.alpha_cum_prod[t])
        var = var * o.betas[t]
        assert s._coef["sigma"][t] == float(var ** 0.5), t
        assert s._coef["sqrt_alpha"][t] == float(torch.sqrt(o.alphas[t]))


def test_sharding_ranges():
    from weatherconverter_b200.sharding import initial_noise, shard_range
    for gb, ws in ((256, 8), (32, 1), (10, 4), (7, 8)):
        spans = [shard_range(gb, ws, r) for r in range(ws)]
        assert spans[0][0] == 0 and spans[-1][1] == gb
        assert all(spans[i][1] == spans[i + 1][0] for i in range(ws - 1))
    full = initial_noise((3, 4, 4), 0, 6)
    parts = torch.cat([initial_noise((3, 4, 4), *shard_range(6, 2, r)) for r in range(2)])
    assert torch.equal(full, parts)


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["WC_ROOT"])
from weatherconverter_b200.sharding import shard_range, initial_noise, gather_images
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
a, b = shard_range(6, w, r)
local = initial_noise((3, 4, 4), a, b)
parts = gather_images(local, w)
t = torch.tensor([float(r + 1)]); dist.all_reduce(t, op=dist.ReduceOp.MAX)   # bench.py's max-over-ranks timing
a7, b7 = shard_range(7, w, r)            # uneven shards (4 + 3): padded gather, sliced on rank 0
parts7 = gather_images(initial_noise((3, 4, 4), a7, b7), w, global_batch=7)
if r == 0:
    assert torch.equal(torch.cat(parts), initial_noise((3, 4, 4), 0, 6)) and float(t) == w
    assert [p.shape[0] for p in parts7] == [4, 3] and torch.equal(torch.cat(parts7), initial_noise((3, 4, 4), 0, 7))
    print("GLOO_OK")
dist.destroy_process_group()
"""


def test_sharding_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, WC_ROOT=ROOT, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                         env=env, capture_output=True, text=True, timeout=300)
    assert "GLOO_OK" in out.stdout, out.stdout + out.stderr


def test_legacy_unet_state_dict_matches_reference_layout():
    """The legacy UNet module exposes the reference's state_dict keys / shapes / dtypes in registration order."""
    import torch
    from oracle.legacy_unet import legacy_param_spec
    from weatherconverter_b200.diffusion_model.models.old_modules import UNet, legacy_param_spec as spec2
    m = UNet()
    sd = m.state_dict()
    ref = legacy_param_spec()
    assert list(sd.keys()) == list(ref.keys()) == list(spec2().keys())
    for k, (shape, dt) in ref.items():
        assert tuple(sd[k].shape) == tuple(shape) and sd[k].dtype == dt, k
    # head-dim padding helper: 24 -> 32 keeps q.k products and the projected output
    w = {"a.mha.in_proj_weight": torch.randn(288, 96), "a.mha.in_proj_bias": torch.randn(288), "a.mha.out_proj.weight": torch.randn(96, 96)}
    wp, bp, wop = UNet._pad_attention(w, "a", 96)
    assert wp.shape == (384, 96) and bp.shape == (384,) and wop.shape == (96, 128)
    x = torch.randn(5, 96)
    qkv = (x @ w["a.mha.in_proj_weight"].T + w["a.mha.in_proj_bias"]).view(5, 3, 4, 24)
    qkvp = (x @ wp.T + bp).view(5, 3, 4, 32)
    assert torch.allclose(qkvp[..., :24], qkv, atol=1e-5) and float(qkvp[..., 24:].abs().max()) == 0.0
    o = torch.randn(5, 4, 24)
    op = torch.zeros(5, 4, 32); op[..., :24] = o
    assert torch.allclose(op.reshape(5, 128) @ wop.T, o.reshape(5, 96) @ w["a.mha.out_proj.weight"].T, atol=1e-4)


def test_bench_roofline_traffic_comes_from_the_committed_ncu_capture():
    """bench.py's roofline.traffic is the DRAM bytes per igemm launch of the committed ncu launch list of the same command."""
    import json
    sys.path.insert(0, ROOT)
    import bench
    import glob
    t, src = bench._dram_traffic_per_launch("c3")
    newest = max(glob.glob(os.path.join(ROOT, "profiles", "r*_dram_traffic_c3.json")),
                 key=lambda f: int(re.match(r"r(\d+)_", os.path.basename(f)).group(1)))
    assert src == os.path.basename(newest)          # the NEWEST round's capture is the one reported (and named in the line)
    meta = json.load(open(newest))
    assert t == pytest.approx(meta["dram_bytes_per_launch"]) and t > 1e6
    assert os.path.exists(os.path.join(ROOT, meta["source"]))
    assert bench._dram_traffic_per_launch("no_such_workload") == (None, None)


def test_launch_traffic_tool_parses_an_ncu_log(tmp_path, monkeypatch):
    """tools/launch_traffic.py: keeps the last N launches of an ncu metric log, sums time / DRAM bytes per kernel."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import launch_traffic
    hdr = '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"'
    rows = [hdr]
    def add(i, name, ns, rd_mb, wr_kb):
        base = f'"{i}","1","python","h","{name}","1","7","(320, 1, 1)","(148, 1, 1)","0","10.0","Command line profiler metrics"'
        rows.append(base + f',"dram__bytes_read.sum","Mbyte","{rd_mb}"')
        rows.append(base + f',"dram__bytes_write.sum","Kbyte","{wr_kb}"')
        rows.append(base + f',"gpu__time_duration.sum","us","{ns}"')
    add(0, "void wc::<unnamed>::pack_kernel(int)", "5.0", "1.0", "1.0")                       # setup launch: dropped
    add(1, "void wc::<unnamed>::igemm_kernel<(bool)0, (bool)1, (bool)0>(wc::IgemmMaps, wc::IgemmArgs)", "40.0", "10.0", "500.0")
    add(2, "void wc::<unnamed>::igemm_kernel<(bool)0, (bool)1, (bool)0>(wc::IgemmMaps, wc::IgemmArgs)", "60.0", "30.0", "1,500.0")
    add(3, "void wc::<unnamed>::gn_apply_kernel(const __nv_bfloat16 *, int)", "10.0", "2.0", "0.0")
    log = tmp_path / "ncu.csv"
    log.write_text("==PROF== Connected\n" + "\n".join(rows) + "\n")
    (tmp_path / "profiles").mkdir()
    monkeypatch.chdir(tmp_path)
    launch_traffic.main(str(log), 3, str(tmp_path / "profiles" / "x"), "zz", 7)    # round number -> profiles/r7_dram_traffic_zz.json
    import json
    meta = json.load(open(tmp_path / "profiles" / "r7_dram_traffic_zz.json"))
    assert meta["launches_per_step"] == 2
    assert meta["dram_bytes_per_launch"] == pytest.approx((10e6 + 30e6 + 0.5e6 + 1.5e6) / 2)
    summary = (tmp_path / "profiles" / "x_summary.txt").read_text()
    assert "igemm_kernel<0, 1, 0>" in summary and "pack_kernel" not in summary


def test_mma_issue_is_warp_uniform_in_sass():
    """The tcgen05.mma issue loops must stay in warp-uniform control flow with one elected lane (DESIGN 3.1): inside
    `if (lane == 0)` the compiler wraps every UTCHMMA in an ELECT / PLOP3 / BRA.U.ANY loop plus R2UR moves (~13 SASS
    instructions per MMA), which made the issuing thread the limiter of the narrow layers.  Checked on the built objects."""
    import shutil
    import __graft_entry__ as ge
    ge.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    build = os.path.join(ROOT, "weatherconverter_b200", "csrc", "build")
    for obj in ("igemm.o", "attention.o", "attention_small.o", "attention_bwd.o", "wgrad.o"):
        sass = subprocess.run([cuobjdump, "-sass", os.path.join(build, obj)], capture_output=True, text=True, check=True).stdout
        lines = [l for l in sass.splitlines() if re.search(r"/\*[0-9a-f]{4,5}\*/\s+\S", l)]
        n_mma = sum("UTCHMMA" in l for l in lines)
        assert n_mma > 0, obj
        wrapped = sum(1 for i, l in enumerate(lines) if "BRA.U.ANY" in l and any("UTCHMMA" in p for p in lines[max(0, i - 4):i]))
        assert wrapped == 0, f"{obj}: {wrapped} of {n_mma} UTCHMMA are issued from divergent code (ELECT/BRA.U.ANY wrapper)"


def test_tma_epilogue_quadrant_boxes_cover_the_tile_in_lane_order():
    """igemm TMA epilogue (csrc/igemm.cu, conv.cu): the 32 pixels of a TMEM lane quadrant (tile pixels 32q .. 32q+31 in x-fastest
    order) must be exactly the TMA box (qw, qh, qb) at (qx0, qy0, qb0), enumerated in the box's own x-fastest order - that is
    what lets lane i stage row i of the box.  Checked for every power-of-two tile shape with tb*th*tw == 128."""
    shapes = [(tb, th, tw) for tb in (1, 2, 4, 8, 16, 32, 64, 128) for th in (1, 2, 4, 8, 16, 32, 64, 128)
              for tw in (1, 2, 4, 8, 16, 32, 64, 128) if tb * th * tw == 128]
    assert len(shapes) == 36
    for tb, th, tw in shapes:
        qw = min(tw, 32)                      # conv.cu: finish_plan
        qh = min(th, 32 // qw)
        qb = 32 // (qw * qh)
        if qb > tb:                           # such a plan keeps the per-lane stores
            continue
        for quad in range(4):
            q_pix = quad * 32                 # igemm_kernel: epilogue warps
            qx0, qy0, qb0 = q_pix % tw, (q_pix // tw) % th, q_pix // (tw * th)
            for lane in range(32):
                row = q_pix + lane
                bb, rem = divmod(row, th * tw)
                yy, xx = divmod(rem, tw)
                # position of box row `lane`: x fastest, then y, then b
                bx, by, bz = lane % qw, (lane // qw) % qh, lane // (qw * qh)
                assert (xx, yy, bb) == (qx0 + bx, qy0 + by, qb0 + bz), (tb, th, tw, quad, lane)


def test_load_model_reads_reference_checkpoint_formats(tmp_path):
    """The three reference-named load_model functions ingest the reference's checkpoint dictionaries (sample_ddpm.py:56-61
    'model_state_dict'; srgan_model/inference.py:9-16 'model'; seg_model/inference.py:27-33 'model_state_dict' + config name)
    and leave the module in eval mode with exactly the saved values.  (Host-side part; the GPU forward after loading is
    tests/test_gpu_parity_rows.py.)"""
    import torch
    from oracle import deeplab
    from oracle.unet import DEFAULT_MODEL_CONFIG
    from oracle.weights import synth_state_dict
    from weatherconverter_b200.diffusion_model.config.models import ModelConfig
    from weatherconverter_b200.diffusion_model.models.unet_base import param_spec
    from weatherconverter_b200.diffusion_model import sample_ddpm
    from weatherconverter_b200.seg_model import inference as seg_inference
    from weatherconverter_b200.srgan_model import inference as srgan_inference
    from weatherconverter_b200.srgan_model.models import Generator
    cfg = dict(DEFAULT_MODEL_CONFIG)
    sd = synth_state_dict({k: (v, torch.float32) for k, v in param_spec(cfg).items()}, 5)
    torch.save({"model_state_dict": sd, "optimizer_state_dict": {}, "epoch": 7}, tmp_path / "u.ckpt")
    m = sample_ddpm.load_model(str(tmp_path / "u.ckpt"), ModelConfig(**cfg))
    got = m.state_dict()
    assert not m.training and list(got) == list(sd) and all(torch.equal(got[k].cpu(), sd[k]) for k in sd)
    sdg = synth_state_dict(Generator(upscale_factor=4).state_dict(), 6)
    torch.save({"model": sdg}, tmp_path / "g.pth.tar")
    G = srgan_inference.load_model(str(tmp_path / "g.pth.tar"))
    got = G.state_dict()
    assert not G.training and all(torch.equal(got[k].cpu(), sdg[k]) for k in sdg)
    with pytest.raises(KeyError):     # a diffusion-style file is not an SRGAN checkpoint
        srgan_inference.load_model(str(tmp_path / "u.ckpt"))
    sds = synth_state_dict(deeplab.deeplab_param_spec("resnet101"), 8)
    torch.save({"model_state_dict": sds, "epoch": 40, "loss": 0.0}, tmp_path / "s.pth")
    S = seg_inference.load_model(str(tmp_path / "s.pth"), {"name": "deeplabv3plus_resnet101", "num_classes": 19, "output_stride": 16})
    got = S.state_dict()
    assert not S.training and set(got) == set(sds) and all(torch.equal(got[k].cpu(), sds[k]) for k in sds)
