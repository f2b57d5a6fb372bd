"""GroupNorm(8)[+SiLU], its backward and the bias column sums (csrc/norm.cu) at the UNet's launch geometries against a float64
reference, plus exact identities and bitwise checks that need no reference.

Launch geometry (``walk_unet`` in csrc/unet_plan.cuh with DEFAULT_MODEL_CONFIG; ``test_plans_launch_only_tabled_shapes``
checks the tables below against the launch records).  Per UNet level the pixel count HW is that of the level's map:

  C3    64x128 latent, inference, batch 32:  HW 8192, 2048, 512, 128.
  C2    128x256, inference, batch 16:        HW 32768, 8192, 2048, 512.
  C5    128x256, training, batch 64:         the C2 forward shapes, the backward and the bias column sums.

GroupNorm forward (HW of the level, C, ldx; the output is a fresh contiguous buffer, ldy = C):

  level 0   (64, 128)  (128, 128)  (64, 64)                  first down ResNet reads the conv_in slice of the concat
  level 1   (128, 256) (256, 256)  (64, 64)                  buffer: ldx = 2C; up blocks read the whole concat buffer
  level 2   (256, 512) (512, 512)  (128, 128)
  level 3   (512, 1024) (768, 768) (512, 512) (1024, 1024) (256, 256)     (mid blocks included)

The backward (C5) runs at the same (HW, C, ldx); dy is contiguous, dx has the layout of x (ldo = ldx: the gradient of a slice
is the same slice of a shadow buffer), ``add1`` is the attention's identity branch and ``add2 == dx`` accumulates in place
where the residual 1x1 convolution wrote the gradient first.  ``BWD_PLAN`` lists the exact strides.  The column sums add
every conv / linear bias gradient (C up to 2304 = 3 x 768, the mid blocks' QKV projection) and the per-sample t-embedding
gradient (``out_rows`` with ldo = 8192, the width of the concatenated t-embedding projection); ``COLSUM_PLAN`` lists them.

Split counts (``stats_splits``, ``apply_splits``, ``bwd_splits`` mirror the host code; SM count from the device):

  ========================  ===============================================  ===========================================
  pass                      blocks per sample                                regimes reached (``test_split_coverage``)
  ========================  ===============================================  ===========================================
  forward statistics        HW <= 2048: largest power of two <= ceil(HW/128)  1 (HW <= 128), 2, 4, 8; the 32 cap (HW >
                            capped at 8; else min(32, ceil(HW/128)).  A       4096); ragged slabs (HW % splits != 0)
                            function of HW only: batch invariance
  forward apply             min(ceil(8 SMs / B), ceil(HW / 32))              the HW/32 cap; more than one wave
  backward stats / reduce   min(ceil(8 SMs / B), ceil(HW / 32), 32)          ragged: 32768 / 19 at batch 64; the caps
  backward apply            min(ceil(8 SMs / B), ceil(HW / 32))
  colsum                    as backward stats; threads = C/8 rounded up to   C/8 >= 256 (C = 2304: one pixel row)
                            32 when C/8 >= 256, else (256 / (C/8)) * C/8
  ========================  ===============================================  ===========================================

The backward split counts depend on the batch, so the backward is deterministic (a repeated launch is bit-identical) but
NOT batch-invariant: image b of a batch-64 backward differs in the last bits from the same image alone.  The forward is
batch-invariant and is checked bit for bit.

Reference: float64 on the device from the same bf16 inputs, two-pass variance.  Forward: every element of every sample.
Backward: dx per element for the first, the last and two random samples; dgamma / dbeta over the whole batch; with SiLU off
and no additive inputs, sum(dx) = 0 and sum(dx * xhat) = 0 for every (sample, group).

Bounds were calibrated on an NVIDIA B200 (power limit 1000 W): each is 1.5-2x the worst value measured over its case
family, which is written beside it.
"""
import math
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

EPS = 1e-5
GROUPS = 8
U8 = 2.0 ** -8     # unit roundoff of bf16

# ---- bounds (NVIDIA B200, 1000 W power limit; measured worst value of the family in the comment)
# forward: max |y - ref| / (2^-8 |ref| + 2^-12 |z| + 2^-16); the 2^-12 |z| term is silu_fast's tanh.approx error on the negative
# tail (h * tanh(h) with |h| = |z|/2 and relative error 2^-11).  "dc": the fp32 partial sums put an absolute error of a few
# 2^-24 |mean| on the mean, which shows where z is near 0 (worst at HW 128, C >= 256)
FWD_ERR = {"plain": 1.5, "dc": 2.5, "wide": 1.5, "flat": 1.5}   # measured 0.937 / 1.654 / 0.937 / 0.937
BWD_DX = 1.6           # max |dx - ref| / (2^-8 |ref| + 2^-12 rms(ref of the sample)); measured 0.980
BWD_DGAMMA = 4e-5      # ||got - ref|| / ||ref|| over the channels; measured 2.48e-5 (C 2048, HW 1000, DC offsets), 3e-7 plain
BWD_DBETA = 6e-7       # measured 3.10e-7
# |sum over a (sample, group)| / (2^-8 sqrt(n) rms(term)), worst over the batch; measured 10.99 (sum dx) / 8.73 (sum dx xhat)
# at HW 32768.  Not a random walk: dx ~ rstd gamma_c dy with dy on the bf16 grid, so its rounding errors are correlated; the
# exact dx rounded once to bf16 reaches 7.3 over 8 samples of that shape.
BWD_SUM = 18.0
COLSUM_REL = 1.5e-7    # max |got - ref| / (sum |x| over the summed elements), per output; measured 7.82e-8


def stats_splits(HW):
    n = -(-HW // 128)
    if HW <= 2048:
        c = 1
        while c * 2 <= n and c < 8:
            c *= 2
        return c
    return max(1, min(n, 32))


def apply_splits(B, HW, sms):
    return max(1, min(-(-8 * sms // B), -(-HW // 32)))


def bwd_splits(B, HW, sms):
    return max(1, min(-(-8 * sms // B), -(-HW // 32), 32))


def gn_threads(C):
    vpp = C // 8
    return (256 // vpp) * vpp


def _level_shapes(hw0):
    """(HW, C, ldx) of the GroupNorm launches of one plan, level 0 at hw0 pixels."""
    h = [hw0, hw0 // 4, hw0 // 16, hw0 // 64]
    return [(h[0], 64, 128), (h[0], 128, 128), (h[0], 64, 64),
            (h[1], 128, 256), (h[1], 256, 256), (h[1], 64, 64),
            (h[2], 256, 512), (h[2], 512, 512), (h[2], 128, 128),
            (h[3], 512, 1024), (h[3], 768, 768), (h[3], 512, 512), (h[3], 1024, 1024), (h[3], 256, 256)]


PLAN_BATCH = {"C3": 32, "C2": 16, "C5": 64}
PLAN_SHAPES = {"C3": _level_shapes(8192), "C2": _level_shapes(32768), "C5": _level_shapes(32768)}

# (HW, C, ldx, ldd, ldo, lda1, lda2) of the C5 backward; 0: no such input
BWD_PLAN = sorted({
    (32768, 64, 128, 64, 128, 0, 128), (32768, 128, 128, 128, 128, 0, 0), (32768, 128, 128, 128, 128, 0, 128),
    (32768, 64, 64, 64, 64, 0, 0), (32768, 64, 64, 64, 64, 0, 64),
    (8192, 128, 256, 128, 256, 0, 256), (8192, 256, 256, 256, 256, 0, 0), (8192, 256, 256, 256, 256, 256, 0),
    (8192, 256, 256, 256, 256, 0, 256), (8192, 64, 64, 64, 64, 0, 0), (8192, 64, 64, 64, 64, 64, 0),
    (8192, 64, 64, 64, 64, 0, 64),
    (2048, 256, 512, 256, 512, 0, 512), (2048, 512, 512, 512, 512, 0, 0), (2048, 512, 512, 512, 512, 512, 0),
    (2048, 512, 512, 512, 512, 0, 512), (2048, 128, 128, 128, 128, 0, 0), (2048, 128, 128, 128, 128, 128, 0),
    (2048, 128, 128, 128, 128, 0, 128),
    (512, 512, 1024, 512, 1024, 0, 1024), (512, 768, 768, 768, 768, 0, 0), (512, 768, 768, 768, 768, 768, 0),
    (512, 768, 768, 768, 768, 0, 768), (512, 512, 512, 512, 512, 0, 0), (512, 512, 512, 512, 512, 512, 0),
    (512, 512, 512, 512, 512, 0, 512), (512, 1024, 1024, 1024, 1024, 0, 1024), (512, 256, 256, 256, 256, 0, 0),
    (512, 256, 256, 256, 256, 256, 0), (512, 256, 256, 256, 256, 0, 256),
})

# (HW, C, ldx, ldo) of the C5 bias column sums; ldo 0: no per-sample rows
COLSUM_PLAN = sorted({
    (32768, 128, 128, 8192), (32768, 128, 128, 0), (32768, 64, 64, 8192), (32768, 64, 64, 0), (32768, 64, 128, 0),
    (8192, 128, 256, 0), (8192, 256, 256, 8192), (8192, 256, 256, 0), (8192, 768, 768, 0), (8192, 64, 64, 8192),
    (8192, 64, 64, 0), (8192, 192, 192, 0), (8192, 128, 256, 0),
    (2048, 256, 512, 0), (2048, 512, 512, 8192), (2048, 512, 512, 0), (2048, 1536, 1536, 0), (2048, 128, 128, 8192),
    (2048, 128, 128, 0), (2048, 384, 384, 0),
    (512, 512, 1024, 0), (512, 768, 768, 8192), (512, 768, 768, 0), (512, 2304, 2304, 0), (512, 512, 512, 8192),
    (512, 512, 512, 0), (512, 1536, 1536, 0), (512, 256, 256, 8192), (512, 256, 256, 0), (512, 768, 768, 0),
})

# forward cases (B, HW, C, ldx, plan): every table geometry at the plan's batch, then the shapes that reach the remaining
# split regimes, and the former op-level cases (batch 3 at HW 32 .. 512)
FWD_CASES = [(PLAN_BATCH[p], hw, c, ld, p) for p in ("C3", "C2", "C5") for hw, c, ld in PLAN_SHAPES[p]]
FWD_CASES += [
    (8, 256, 128, 256, None),      # two statistics slabs, strided
    (4, 2600, 256, 256, None),     # 21 statistics slabs, ragged (2600 % 21 != 0)
    (2, 4096, 64, 64, None),       # 32 slabs exactly
    (1, 1000, 2048, 2048, None),   # C at the limit, 8 slabs of 125 pixels (HW % 8 == 0 but not % 16: ragged apply)
    (3, 256, 64, 64, None), (3, 256, 128, 128, None), (3, 32, 768, 768, None), (3, 512, 1024, 1024, None),
]
FAMILIES = ("plain", "dc", "wide", "flat")

# backward cases (B, HW, C, ldx, silu): every C5 geometry at batch 64, SiLU on (+add1 +add2, in place where ldx == 2C as
# the plan does) and off (no adds: the identities); then ragged / small shapes and the former op-level cases
BWD_CASES = [(64, hw, c, ld, s) for hw, c, ld in PLAN_SHAPES["C5"] for s in (True, False)]
BWD_CASES += [(64, 2600, 256, 512, True), (5, 1000, 2048, 2048, False), (2, 256, 64, 64, True), (3, 256, 128, 128, False),
              (2, 32, 768, 768, True), (1, 512, 1024, 1024, True)]

# colsum cases (B, HW, C, ldx, ldo): the plan's bias-gradient shapes at batch 64 (ldo 8192: the t-embedding rows), plus the
# former op-level case (3 x 128 pixels x 2304)
COLSUM_CASES = [(64, hw, c, ld, ldo) for hw, c, ld, ldo in COLSUM_PLAN]
COLSUM_CASES += [(3, 128, 2304, 2304, 2304 + 64), (8, 2600, 136, 144, 200)]


def _id(case):
    return "-".join(str(c) for c in case if c is not None)


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _lib():
    from weatherconverter_b200._lib import check, lib, ptr, stream_ptr
    return check, lib(), ptr, stream_ptr


def _ld(t):
    """Pixel stride of a [B, HW, C] view whose pixels are evenly spaced."""
    assert t.stride(2) == 1 and t.stride(0) == t.shape[1] * t.stride(1), t.stride()
    return t.stride(1)


def _strided(B, HW, C, ld, dev, fill):
    """A [B, HW, C] view into a [B, HW, ld] buffer filled with `fill` (the view starts at channel ld - C)."""
    buf = torch.full((B, HW, ld), fill, device=dev, dtype=torch.bfloat16)
    return buf[:, :, ld - C:], buf


def _canary_ws(nbytes, dev):
    ws = torch.full((nbytes + 4096,), 0xFF, device=dev, dtype=torch.uint8)
    ws[nbytes:] = 0xA5
    return ws


def _canary_ok(ws, nbytes):
    return bool((ws[nbytes:] == 0xA5).all())


def gn_fwd(x, gamma, beta, silu, y, ws=None):
    """One wc_groupnorm_silu launch on [B, HW, C] views; returns the workspace (canary checked)."""
    check, L, ptr, stream_ptr = _lib()
    B, HW, C = x.shape
    nbytes = L.wc_groupnorm_workspace_bytes(B)
    if ws is None:
        ws = _canary_ws(nbytes, x.device)
    check(L.wc_groupnorm_silu(ptr(x), ptr(y), B, HW, C, _ld(x), _ld(y), ptr(gamma), ptr(beta), EPS, int(silu), ptr(ws),
                              stream_ptr()))
    assert _canary_ok(ws, nbytes)
    return ws


def gn_bwd(x, dy, dx, gamma, beta, silu, stats, add1=None, add2=None):
    """One wc_groupnorm_silu_bwd launch; returns (dgamma, dbeta)."""
    check, L, ptr, stream_ptr = _lib()
    B, HW, C = x.shape
    dg = torch.full((C,), float("nan"), device=x.device)
    db = torch.full((C,), float("nan"), device=x.device)
    nbytes = L.wc_groupnorm_bwd_workspace_bytes(B, C)
    ws = _canary_ws(nbytes, x.device)
    check(L.wc_groupnorm_silu_bwd(ptr(x), ptr(dy), ptr(dx), B, HW, C, _ld(x), _ld(dy), _ld(dx), ptr(gamma), ptr(beta), EPS,
                                  int(silu), ptr(stats), ptr(add1), _ld(add1) if add1 is not None else 8, ptr(add2),
                                  _ld(add2) if add2 is not None else 8, ptr(dg), ptr(db), ptr(ws), stream_ptr()))
    assert _canary_ok(ws, nbytes)
    return dg, db


def colsum(x, rows=None, total=None):
    check, L, ptr, stream_ptr = _lib()
    B, HW, C = x.shape
    nbytes = L.wc_groupnorm_bwd_workspace_bytes(B, C)
    ws = _canary_ws(nbytes, x.device)
    check(L.wc_colsum(ptr(x), B, HW, C, _ld(x), ptr(rows), rows.stride(0) if rows is not None else C, ptr(total), ptr(ws),
                      stream_ptr()))
    assert _canary_ok(ws, nbytes)


def _inputs(B, HW, C, family, seed, dev):
    """x [B, HW, C] (float32, to be rounded to bf16), gamma, beta [C] for an input family."""
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(B, HW, C, device=dev, generator=g)
    gamma = 1 + 0.2 * torch.randn(C, device=dev, generator=g)
    beta = 0.2 * torch.randn(C, device=dev, generator=g)
    cpg = C // GROUPS
    if family == "plain":
        x = x * 2 + 0.5
    elif family == "dc":       # per-group DC offset up to 32 standard deviations: E[x^2] - mean^2 cancels to 1 part in 1025
        ratio = torch.tensor([0.0, 1.0, -4.0, 8.0, -16.0, 24.0, -32.0, 32.0], device=dev)
        x = x + ratio.repeat_interleave(cpg)
    elif family == "wide":     # |z| up to ~13: SiLU's negative tail
        gamma = 5 * torch.rand(C, device=dev, generator=g) - 2.5
        beta = torch.randn(C, device=dev, generator=g)
    elif family == "flat":     # group 0 constant (variance 0), group 1 constant but one element (variance near 0)
        x[:, :, :cpg] = 0.1
        x[:, :, cpg:2 * cpg] = -0.3
        x[:, HW // 2, cpg + 1] = 3.7
    return x, gamma, beta


def _ref_stats(xb):
    """xb [n, HW, C] bf16 -> mean, rstd [n, 1, 8, 1] float64 (two-pass variance)."""
    n, HW, C = xb.shape
    x = xb.double().view(n, HW, GROUPS, C // GROUPS)
    mean = x.mean(dim=(1, 3), keepdim=True)
    var = (x - mean).pow(2).mean(dim=(1, 3), keepdim=True)
    return mean, 1.0 / torch.sqrt(var + EPS)


def _xhat(xb, mean, rstd):
    n, HW, C = xb.shape
    return ((xb.double().view(n, HW, GROUPS, C // GROUPS) - mean) * rstd).view(n, HW, C)


def _silu(z):
    return z * torch.sigmoid(z)


def _chunks(B, HW, C):
    per = max(1, (1 << 24) // (HW * C))
    return [(i, min(B, i + per)) for i in range(0, B, per)]


@pytest.mark.parametrize("B,HW,C,ld,plan", FWD_CASES, ids=[_id(c) for c in FWD_CASES])
def test_forward_vs_float64(B, HW, C, ld, plan):
    dev = _dev()
    for fi, family in enumerate(FAMILIES):
        seed = HW * 31 + C * 7 + B + fi
        x32, gamma, beta = _inputs(B, HW, C, family, seed, dev)
        x, _ = _strided(B, HW, C, ld, dev, 3.0)
        x.copy_(x32)
        del x32
        for silu in (True, False) if family != "wide" else (True,):
            y = torch.full((B, HW, C), float("nan"), device=dev, dtype=torch.bfloat16)
            gn_fwd(x, gamma, beta, silu, y)
            worst = 0.0
            for a, b in _chunks(B, HW, C):
                mean, rstd = _ref_stats(x[a:b])
                z = _xhat(x[a:b], mean, rstd) * gamma.double() + beta.double()
                ref = _silu(z) if silu else z
                got = y[a:b].double()
                assert not torch.isnan(got).any(), "an output pixel was not written"
                err = (got - ref).abs() / (U8 * ref.abs() + 2.0 ** -12 * z.abs() + 2.0 ** -16)
                worst = max(worst, float(err.max()))
            print(f"[gn] fwd {family} silu={int(silu)} {_id((B, HW, C, ld))}: {worst:.3f}")
            assert worst < FWD_ERR[family], (family, silu, worst)


def _bwd_run(B, HW, C, ld, silu, seed, dev, family):
    """Inputs at the plan's layout and one forward + backward launch.  SiLU on: add1 contiguous, add2 = dx in place (dx is
    pre-filled with the add2 values, as the plan accumulates); off: no additive inputs and dx NaN-filled."""
    x32, gamma, beta = _inputs(B, HW, C, family, seed, dev)
    x, _ = _strided(B, HW, C, ld, dev, 3.0)
    x.copy_(x32)
    del x32
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    dy = torch.randn(B, HW, C, device=dev, generator=g).bfloat16()
    y = torch.empty(B, HW, C, device=dev, dtype=torch.bfloat16)
    stats = gn_fwd(x, gamma, beta, silu, y)
    dx, _ = _strided(B, HW, C, ld, dev, float("nan"))
    add1 = add2 = None
    if silu:
        add1 = torch.randn(B, HW, C, device=dev, generator=g).bfloat16()
        dx.copy_(torch.randn(B, HW, C, device=dev, generator=g))
        add2 = dx.clone()          # the reference's copy; the launch reads add2 from dx itself
    dg, db = gn_bwd(x, dy, dx, gamma, beta, silu, stats, add1, dx if silu else None)
    return x, dy, dx, gamma, beta, add1, add2, dg, db


@pytest.mark.parametrize("B,HW,C,ld,silu", BWD_CASES, ids=[_id(c) for c in BWD_CASES])
def test_backward_vs_float64(B, HW, C, ld, silu):
    dev = _dev()
    seed = HW * 17 + C * 3 + B + int(silu)
    x, dy, dx, gamma, beta, add1, add2, dg, db = _bwd_run(B, HW, C, ld, silu, seed, dev, "plain" if silu else "dc")
    assert not torch.isnan(dx).any(), "a dx pixel was not written"
    gd, bd = gamma.double(), beta.double()
    rng = random.Random(seed)
    check = {0, B - 1, rng.randrange(B), rng.randrange(B)}
    ref_dg = torch.zeros(C, dtype=torch.float64, device=dev)
    ref_db = torch.zeros_like(ref_dg)
    dx_err, sum0, sum1 = 0.0, 0.0, 0.0
    cpg = C // GROUPS
    n = HW * cpg
    for a, b in _chunks(B, HW, C):
        mean, rstd = _ref_stats(x[a:b])
        xh = _xhat(x[a:b], mean, rstd)
        z = xh * gd + bd
        d = dy[a:b].double()
        if silu:
            s = torch.sigmoid(z)
            d = d * s * (1 + z * (1 - s))
        ref_dg += (d * xh).sum(dim=(0, 1))
        ref_db += d.sum(dim=(0, 1))
        k = b - a
        gdz = (gd * d).view(k, HW, GROUPS, cpg)
        m1 = gdz.mean(dim=(1, 3), keepdim=True)
        m2 = (gdz * xh.view(k, HW, GROUPS, cpg)).mean(dim=(1, 3), keepdim=True)
        ref = ((gdz - m1 - xh.view(k, HW, GROUPS, cpg) * m2) * rstd).view(k, HW, C)
        got = dx[a:b].double()
        if add1 is not None:
            ref = ref + add1[a:b].double() + add2[a:b].double()
        for i in range(a, b):
            if i in check:
                r = ref[i - a]
                e = (got[i - a] - r).abs() / (U8 * r.abs() + 2.0 ** -12 * r.pow(2).mean().sqrt())
                dx_err = max(dx_err, float(e.max()))
        if not silu:     # sum dx = 0 and sum dx * xhat = 0 per (sample, group)
            gg = got.view(k, HW, GROUPS, cpg)
            t1 = gg * xh.view(k, HW, GROUPS, cpg)
            unit = U8 * math.sqrt(n)
            sum0 = max(sum0, float((gg.sum(dim=(1, 3)).abs() / (unit * gg.pow(2).mean(dim=(1, 3)).sqrt())).max()))
            sum1 = max(sum1, float((t1.sum(dim=(1, 3)).abs() / (unit * t1.pow(2).mean(dim=(1, 3)).sqrt())).max()))
    e_dg = float((dg.double() - ref_dg).norm() / ref_dg.norm())
    e_db = float((db.double() - ref_db).norm() / ref_db.norm())
    print(f"[gn] bwd silu={int(silu)} {_id((B, HW, C, ld))}: dx {dx_err:.3f} dgamma {e_dg:.2e} dbeta {e_db:.2e} "
          f"sums {sum0:.3f} {sum1:.3f}")
    assert dx_err < BWD_DX, dx_err
    assert e_dg < BWD_DGAMMA and e_db < BWD_DBETA, (e_dg, e_db)
    assert sum0 < BWD_SUM and sum1 < BWD_SUM, (sum0, sum1)


@pytest.mark.parametrize("B,HW,C,ld,ldo", COLSUM_CASES, ids=[_id(c) for c in COLSUM_CASES])
def test_colsum_vs_float64(B, HW, C, ld, ldo):
    dev = _dev()
    g = torch.Generator(device=dev).manual_seed(HW + C + ld)
    x, _ = _strided(B, HW, C, ld, dev, 3.0)
    x.copy_(torch.randn(B, HW, C, device=dev, generator=g) + 0.25)
    sentinel = 7.0
    rows_buf = torch.full((B, max(ldo, C)), sentinel, device=dev)
    rows = rows_buf[:, :C] if ldo else None
    total = torch.full((C,), float("nan"), device=dev)
    colsum(x, rows, total)
    xd = x.double()
    ref_rows, ref_tot = xd.sum(1), xd.sum((0, 1))
    mass_rows, mass_tot = xd.abs().sum(1), xd.abs().sum((0, 1))
    err = float(((total.double() - ref_tot).abs() / mass_tot).max())
    if ldo:
        err = max(err, float(((rows.double() - ref_rows).abs() / mass_rows).max()))
        assert bool((rows_buf[:, C:] == sentinel).all()), "colsum wrote past channel C of a row"
    print(f"[gn] colsum {_id((B, HW, C, ld, ldo))}: {err:.2e}")
    assert err < COLSUM_REL, err


BIT_CASES = [(4, 2600, 128), (8, 512, 256), (2, 8192, 64), (64, 512, 64), (3, 32, 768), (16, 2048, 1024)]


@pytest.mark.parametrize("B,HW,C", BIT_CASES, ids=[_id(c) for c in BIT_CASES])
def test_bitwise(B, HW, C):
    """Without a reference: a strided launch (ld = 2C, sentinel-filled gaps) equals the contiguous launch bit for bit and leaves
    the gaps alone - y, dx, dgamma, dbeta and the column sums; add2 == dx in place equals out of place; image b of the forward
    equals the batch-1 launch of image b; a repeated backward is bit-identical."""
    dev = _dev()
    x32, gamma, beta = _inputs(B, HW, C, "dc", B * HW + C, dev)
    g = torch.Generator(device=dev).manual_seed(C)
    xc = x32.bfloat16()
    dyc = torch.randn(B, HW, C, device=dev, generator=g).bfloat16()
    a1c = torch.randn(B, HW, C, device=dev, generator=g).bfloat16()
    a2c = torch.randn(B, HW, C, device=dev, generator=g).bfloat16()
    sentinel = -5.0

    def run(ld):
        views = []
        for t in (xc, dyc, a1c, a2c):
            v, _ = _strided(B, HW, C, ld, dev, sentinel)
            v.copy_(t)
            views.append(v)
        x, dy, a1, a2 = views
        y, ybuf = _strided(B, HW, C, ld, dev, sentinel)
        st = gn_fwd(x, gamma, beta, True, y)
        dx, dxbuf = _strided(B, HW, C, ld, dev, sentinel)
        dg, db = gn_bwd(x, dy, dx, gamma, beta, True, st, a1, a2)
        rows_buf = torch.full((B, 2 * C), sentinel, device=dev)
        total = torch.empty(C, device=dev)
        colsum(dy, rows_buf[:, :C], total)
        return ybuf, dxbuf, dg, db, rows_buf, total, (x, dy, a1, a2, st)

    base = run(C)
    wide = run(2 * C)
    for i in (0, 1):
        assert torch.equal(wide[i][..., C:], base[i]), i
        assert bool((wide[i][..., :C].float() == sentinel).all()), ("gap written", i)
    for i in (2, 3, 5):
        assert torch.equal(wide[i], base[i]), i
    assert torch.equal(wide[4][:, :C], base[4][:, :C]) and bool((wide[4][:, C:] == sentinel).all())

    # add2 == dx in place, as the plan accumulates, equals the out-of-place launch
    x, dy, a1, a2, st = base[6]
    inplace = a2.clone()
    dg2, db2 = gn_bwd(x, dy, inplace, gamma, beta, True, st, a1, inplace)
    assert torch.equal(inplace, base[1]) and torch.equal(dg2, base[2]) and torch.equal(db2, base[3])

    # the backward repeats bit for bit (it is not batch-invariant: its split counts depend on the batch)
    dx3 = torch.empty_like(xc)
    dg3, db3 = gn_bwd(x, dy, dx3, gamma, beta, True, st, a1, a2)
    assert torch.equal(dx3, base[1]) and torch.equal(dg3, base[2]) and torch.equal(db3, base[3])

    # forward batch invariance: image b alone gives the same bits
    for b in sorted({0, B // 2, B - 1}):
        y1 = torch.empty(1, HW, C, device=dev, dtype=torch.bfloat16)
        gn_fwd(xc[b:b + 1], gamma, beta, True, y1)
        assert torch.equal(y1[0], base[0][b]), b


@pytest.mark.parametrize("C,ld", [(96, 96), (2112, 2112), (128, 132)])
def test_guard_rails(C, ld):
    """C % 64 != 0, C > 2048 or a pixel stride that is not a multiple of 8: every GroupNorm entry point returns the library's
    error and writes nothing."""
    check, L, ptr, stream_ptr = _lib()
    dev = _dev()
    B, HW = 2, 64
    x = torch.ones(B, HW, ld, device=dev, dtype=torch.bfloat16)
    gamma, beta = torch.ones(C, device=dev), torch.zeros(C, device=dev)
    sentinel = 7.0
    y = torch.full((B, HW, ld), sentinel, device=dev, dtype=torch.bfloat16)
    dx = torch.full((B, HW, ld), sentinel, device=dev, dtype=torch.bfloat16)
    dg, db = torch.full((C,), sentinel, device=dev), torch.full((C,), sentinel, device=dev)
    ws = torch.zeros(L.wc_groupnorm_workspace_bytes(B), device=dev, dtype=torch.uint8)
    ws2 = torch.zeros(L.wc_groupnorm_bwd_workspace_bytes(B, max(C, 64)), device=dev, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="C % 64|multiples of 8"):
        check(L.wc_groupnorm_silu(ptr(x), ptr(y), B, HW, C, ld, ld, ptr(gamma), ptr(beta), EPS, 1, ptr(ws), stream_ptr()))
    with pytest.raises(RuntimeError, match="C % 64|multiples of 8"):
        check(L.wc_groupnorm_silu_bwd(ptr(x), ptr(x), ptr(dx), B, HW, C, ld, ld, ld, ptr(gamma), ptr(beta), EPS, 1, ptr(ws),
                                      None, 8, None, 8, ptr(dg), ptr(db), ptr(ws2), stream_ptr()))
    torch.cuda.synchronize()
    for t in (y, dx, dg, db):
        assert bool((t.float() == sentinel).all())


@pytest.mark.parametrize("C,ld", [(100, 104), (4104, 4104), (64, 68)])
def test_colsum_guard_rails(C, ld):
    """colsum: C % 8 != 0, C > 4096 or a stride that is not a multiple of 8 returns the library's error and writes nothing."""
    check, L, ptr, stream_ptr = _lib()
    dev = _dev()
    B, HW = 2, 64
    x = torch.ones(B, HW, ld, device=dev, dtype=torch.bfloat16)
    sentinel = 7.0
    rows, total = torch.full((B, C), sentinel, device=dev), torch.full((C,), sentinel, device=dev)
    ws = torch.zeros(L.wc_groupnorm_bwd_workspace_bytes(B, C), device=dev, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="colsum"):
        check(L.wc_colsum(ptr(x), B, HW, C, ld, ptr(rows), C, ptr(total), ptr(ws), stream_ptr()))
    torch.cuda.synchronize()
    assert bool((rows == sentinel).all()) and bool((total == sentinel).all())


def test_ops_wrappers_take_channel_slices():
    """ops.groupnorm_silu_fwd_bwd and ops.colsum pass the views' real strides: a channel slice of a concat buffer gives the
    bits of its contiguous copy."""
    from weatherconverter_b200 import ops
    dev = _dev()
    B, H, W, C = 2, 16, 32, 128
    g = torch.Generator(device=dev).manual_seed(3)
    buf = [torch.randn(B, H, W, 2 * C, device=dev, generator=g).bfloat16() for _ in range(4)]
    gamma, beta = 1 + 0.2 * torch.randn(C, device=dev, generator=g), 0.2 * torch.randn(C, device=dev, generator=g)
    sl = [t[..., C:] for t in buf]
    co = [t.contiguous() for t in sl]
    a = ops.groupnorm_silu_fwd_bwd(sl[0], gamma, beta, sl[1], add1=sl[2], add2=sl[3])
    b = ops.groupnorm_silu_fwd_bwd(co[0], gamma, beta, co[1], add1=co[2], add2=co[3])
    for p, q in zip(a, b):
        assert torch.equal(p, q)
    assert torch.equal(ops.groupnorm_silu(sl[0], gamma, beta), b[0])
    for p, q in zip(ops.colsum(sl[1]), ops.colsum(co[1])):
        assert torch.equal(p, q)


def _profiled(run):
    """Launch records of run(): (class, work, info[6])."""
    import ctypes as C
    from weatherconverter_b200._lib import lib
    L = lib()
    L.wc_profile_begin()
    try:
        run()
        torch.cuda.synchronize()
    finally:
        cap = 1 << 15
        cls, ms, work, info = (C.c_int * cap)(), (C.c_double * cap)(), (C.c_double * cap)(), (C.c_int * (cap * 6))()
        n = L.wc_profile_detail(cap, cls, ms, work, info)
        L.wc_profile_end((C.c_double * 8)(), (C.c_longlong * 8)(), (C.c_double * 8)())
    assert 0 < n <= cap
    return [(cls[i], work[i], tuple(info[i * 6: i * 6 + 6])) for i in range(n)]


def _plan_shapes(records, B):
    """GroupNorm forward / backward and colsum shapes of the launch records; checks the noted split counts and the work."""
    sms = _sms()
    fwd, bwd, cs = set(), set(), set()
    for cls, work, (hw, c, f2, f3, f4, f5) in records:
        if cls == 2 and hw and work == 6.0 * B * hw * c:
            assert (f4, f5) == (stats_splits(hw), apply_splits(B, hw, sms)), (hw, c, f4, f5)
            assert f3 == c
            fwd.add((hw, c, f2))
        elif cls == 2 and hw:
            assert work == 10.0 * B * hw * c
            assert (f5 & 0xFFFF, f5 >> 16) == (bwd_splits(B, hw, sms), apply_splits(B, hw, sms))
            bwd.add((hw, c, f2 & 0xFFFF, f2 >> 16, f3 & 0xFFFF, f3 >> 16, f4))
        elif cls == 5 and f5 & 1:
            assert f4 == bwd_splits(B, hw, sms) and f5 & 4, (hw, c, f4, f5)
            cs.add((hw, c, f2, f3))
    return fwd, bwd, cs


def test_plans_launch_only_tabled_shapes():
    """The inference plans at 64x128 and 128x256 and the training plan at 128x256, forward and backward, launch GroupNorm and
    colsum at exactly the tabled (HW, C, strides), with the split counts of the mirror."""
    from oracle.unet import DEFAULT_MODEL_CONFIG
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet
    dev = _dev()
    t = torch.tensor([17], device=dev)
    models = {}
    for ims in (64, 128):
        cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = ims
        torch.manual_seed(ims)
        models[ims] = Unet(cfg).to(dev).eval()
    x3, x2 = torch.randn(1, 3, 64, 128, device=dev), torch.randn(1, 3, 128, 256, device=dev)
    got3 = _plan_shapes(_profiled(lambda: models[64](x3, t)), 1)
    got2 = _plan_shapes(_profiled(lambda: models[128](x2, t)), 1)
    models[128].differentiable = True
    got5 = _plan_shapes(_profiled(lambda: models[128](x2, t).backward(torch.ones_like(x2))), 1)
    print("[gn] plan C3", sorted(got3[0]))
    print("[gn] plan C2", sorted(got2[0]))
    print("[gn] plan C5 fwd", sorted(got5[0]))
    print("[gn] plan C5 bwd", sorted(got5[1]))
    print("[gn] plan C5 colsum", sorted(got5[2]))
    assert got3 == (set(PLAN_SHAPES["C3"]), set(), set())
    assert got2 == (set(PLAN_SHAPES["C2"]), set(), set())
    assert got5[0] == set(PLAN_SHAPES["C5"])
    assert got5[1] == set(BWD_PLAN)
    assert got5[2] == set(COLSUM_PLAN)


def test_split_coverage():
    """The case lists reach every split regime of the mirror: 1, 2, 4 and 8 statistics slabs, the 32-slab cap, ragged slabs in
    the forward and the backward, the HW/32 cap of the apply grids, grids of more than one wave, colsum's C/8 >= 256 path."""
    _dev()
    sms = _sms()
    reach = set()

    def waves(blocks, threads):
        return blocks > sms * (2048 // threads)

    for B, HW, C, _, _ in FWD_CASES:
        ns, na = stats_splits(HW), apply_splits(B, HW, sms)
        reach.add(f"stats-{ns}" if ns <= 8 else "stats-many")
        reach |= {"stats-cap"} if -(-HW // 128) > 32 else set()
        reach |= {"fwd-ragged"} if HW % ns else set()
        reach |= {"fwd-apply-cap"} if na == -(-HW // 32) < -(-8 * sms // B) else set()
        reach |= {"fwd-waves"} if waves(ns * B, gn_threads(C)) or waves(na * B, gn_threads(C)) else set()
    for B, HW, C, _, _ in BWD_CASES:
        nb, na = bwd_splits(B, HW, sms), apply_splits(B, HW, sms)
        reach |= {"bwd-ragged"} if HW % nb else set()
        reach |= {"bwd-cap"} if nb == -(-HW // 32) < -(-8 * sms // B) else set()
        reach |= {"bwd-waves"} if waves(nb * B, gn_threads(C)) else set()
    for B, HW, C, _, _ in COLSUM_CASES:
        reach |= {"colsum-wide"} if C // 8 >= 256 else set()
        reach |= {"colsum-ragged"} if HW % bwd_splits(B, HW, sms) else set()
    need = {"stats-1", "stats-2", "stats-4", "stats-8", "stats-cap", "fwd-ragged", "fwd-apply-cap", "fwd-waves", "bwd-ragged",
            "bwd-cap", "bwd-waves", "colsum-wide", "colsum-ragged"}
    assert need <= reach, need - reach
