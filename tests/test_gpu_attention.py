"""Every attention kernel at the UNet's launch geometries against a float64 reference, plus exact identities and bitwise
independence checks that need no reference.

Dispatch (a pure function of head_dim, N and whether the log2-domain softmax scale is exactly 1, i.e. Q prescaled):
``attention_forward`` (csrc/attention.cu), ``small_forward`` (csrc/attention_small.cu), ``attention_backward``
(csrc/attention_bwd.cu).  ``fwd_kernel`` / ``bwd_kernels`` below write the same map down; ``test_dispatch_table_coverage``
checks that the case lists reach every instantiation at a plan shape, at a ragged N (N % 64 != 0: the last query tile and
the last KV tile are both partial) and with a grid of more than one wave (148 SMs; the head_dim <= 64 backward holds two
CTAs per SM, so there more than 296 CTAs).  Cases are (head_dim, N, batch); 4 heads throughout.

=================================================  ======================  ===================  =================  ==================
instantiation                                      selected when           plan shape           ragged N           multi-wave
=================================================  ======================  ===================  =================  ==================
attention_small_kernel<16,12,false>  (3 groups)    hd 16, N < 2048         legacy (16,1024,16)  (16,2040,16)       (16,8,64): 256
attention_small_kernel<32,8,true>    (3 groups)    hd 32, N < 2048         C3 (32,512,32)       (32,520,32)        (32,520,32): 256
attention_small4_kernel<16,true>     (4 groups)    hd 16, N >= 2048, Q'    C3 (16,8192,32)      (16,2056,16)       (16,8192,32): 2048
attention_small4_kernel<16,false>                  hd 16, N >= 2048        C5 (16,8192,4)       (16,8184,2)        (16,2176,16): 320
attention_small4_kernel<32,true>                   hd 32, N >= 2048, Q'    C3 (32,8192,32)      (32,8184,4)        (32,8192,32): 2048
attention_small4_kernel<32,false>                  hd 32, N >= 2048        C5 (32,2048,16)      (32,2056,16)       (32,2056,16): 320
attention_kernel<64,128,2>                         hd 64                   C3 (64,2048,8)       (64,2056,8)        (64,2056,8): 288
attention_kernel<128,64,2>                         hd 128                  C5 (128,2048,8)      (128,8184,2)       (128,8184,2): 256
attention_kernel<192,64,1>                         hd 192                  C2 (192,512,16)      (192,2056,4)       (192,2056,4): 272
attention_bwd_kernel<16,64,2,KV|dQ,1>  (2 / SM)    hd 16                   C5 (16,8192,2)       (16,200,40)        (16,200,40): 320
attention_bwd_kernel<32,64,2,KV|dQ,1>  (2 / SM)    hd 32                   C5 (32,2048,8)       (32,520,20)        (32,520,20): 400
attention_bwd_kernel<64,64,2,KV|dQ,1>  (2 / SM)    hd 64                   C5 (64,8192,64)      (64,2056,8)        (64,8192,64): 16384
attention_bwd_kernel<128,128,1,KV|dQ,2>            hd 128                  C5 (128,2048,4)      (128,8184,1)       (128,2048,4): 256
attention_bwd_kernel<192,64,{1,2},KV|dQ,2>         hd 192                  C5 (192,512,16)      (192,2056,4)       (192,2056,4): 272
=================================================  ======================  ===================  =================  ==================

(Q' = Q prescaled by log2(e)/sqrt(hd), scale < 0; the backward runs two kernels per head_dim, a KV pass and a dQ pass, with
the same grid.)  Those are nineteen kernels in all; the table names one case of each kind, the lists hold more.

Plan shapes (``walk_unet`` in csrc/unet_plan.cuh with DEFAULT_MODEL_CONFIG; ``test_plans_launch_only_tabled_shapes`` checks
them against the launch records):
  C3    64x128 latent, inference, Q prescaled: (32,8192) (16,8192) (64,2048) (16,2048) (128,512) (32,512) (192,128)
        (128,128) (64,128).
  C2    128x256, inference, Q prescaled: (64,8192) (16,8192) (128,2048) (32,2048) (192,512) (128,512) (64,512).
  C5    128x256, training: the same shapes with unscaled Q, ``attention_lse`` and the backward.
  legacy UNet (128x128, csrc/legacy.cu): explicit scale 1/sqrt(C/4); head_dim 24 zero-padded to 32 at N 1024 and 256,
        head_dim 16 at 1024, 32 at 256, 64 at 64.

Reference: float64 on the device from the same bf16 inputs.  For each case a few (batch, head) pairs are checked - always
the first and the last, which shows a batch / head index mix-up - and within a pair every query row, so every CTA's first
and last row and the ragged tail are among them.  The backward reference is exact per pair: log-sum-exp, O and
D = rowsum(dO * O) over all queries, then dQ, dK, dV for all rows, in chunks of query rows.

Bounds were calibrated on an NVIDIA B200 (power limit 1000 W): each is 1.5-2x the worst value measured over its case
family, which is written beside it.
"""
import math
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

HEADS = 4
SMS = 148
LN2 = math.log(2.0)
LOG2E = 1.0 / LN2
PRE = "pre"      # Q prescaled by log2(e)/sqrt(hd), scale < 0: the inference plans (UNIT kernels at head_dim 16/32, N >= 2048)
LSE = "lse"      # unscaled Q through attention_lse (scale 1/sqrt(hd), log-sum-exp saved): the training plan
LEGACY_SCALE = {24: 1 / math.sqrt(24), 16: 0.25, 32: 1 / math.sqrt(32), 64: 0.125}

# ---- bounds (NVIDIA B200, 1000 W power limit; measured worst value of the family in the comment)
FWD_RMS = {"small3": 4e-3, "small4": 4e-3, "general": 4e-3}    # rms-rel over the checked rows; measured 2.54e-3 / 2.38e-3 / 2.34e-3
FWD_ROW = {"small3": 9e-3, "small4": 1.2e-2, "general": 7e-3}   # worst single row, relative; measured 5.88e-3 / 7.97e-3 / 4.63e-3
# log-sum-exp, log2 units, absolute.  The small-head kernels sum l from the bf16-rounded P (row sums on the tensor core), so a
# row dominated by one key carries that term's rounding, up to 2^-8 / ln 2 = 5.6e-3 ("peaked": big / grow / shrink logits).
LSE_ABS = {"general": 4e-4,        # measured 2.03e-4
           "small": 4e-3,          # plain logits; measured 2.75e-3 (N = 8, one tile of eight keys), 7.3e-4 at N >= 136
           "small-peaked": 8.5e-3}  # measured 5.61e-3
BWD_RMS = {"dq": 1.1e-2, "dk": 1e-2, "dv": 4e-3}   # rms-rel against float64; measured 7.29e-3 / 6.15e-3 / 2.61e-3 (dQ, dK at
                                                    # "grow" logits: D from the bf16 O cancels against the dominant dP; 2.8e-3 else)
BWD_SUM = {"dv": 5.0, "dk": 10.0}   # |sum of rows| / (2^-8 sqrt(N) rms(row)), worst component; measured 3.34 / 6.47
ONE_TOL = 2.0 ** -8                  # V = 1: |o - 1|, exact up to the bf16 rounding of the output


def fwd_kernel(hd, N, scale):
    """The forward instantiation that attention_forward launches for (head_dim, N, scale)."""
    if hd == 24:
        hd = 32
    if hd in (16, 32):
        if N >= 2048:
            return f"attention_small4_kernel<{hd},{'true' if scale == PRE else 'false'}>"
        return {16: "attention_small_kernel<16,12,false>", 32: "attention_small_kernel<32,8,true>"}[hd]
    return {64: "attention_kernel<64,128,2>", 128: "attention_kernel<128,64,2>", 192: "attention_kernel<192,64,1>"}[hd]


def fwd_family(hd, N, scale):
    k = fwd_kernel(hd, N, scale)
    return "small4" if "small4" in k else "small3" if "small" in k else "general"


def fwd_ctas(hd, N, B):
    hd = 32 if hd == 24 else hd
    span = (512 if N >= 2048 else 384) if hd <= 32 else (128 if hd == 192 else 256)
    return B * HEADS * -(-N // span)


def bwd_kernels(hd):
    bt, skv, sq, nsw = {16: (64, 2, 2, 1), 32: (64, 2, 2, 1), 64: (64, 2, 2, 1), 128: (128, 1, 1, 2), 192: (64, 1, 2, 2)}[hd]
    return [f"attention_bwd_kernel<{hd},{bt},{skv},true,{nsw}>", f"attention_bwd_kernel<{hd},{bt},{sq},false,{nsw}>"]


def bwd_ctas(hd, N, B):
    return B * HEADS * -(-N // 128)


def bwd_wave(hd):
    return 2 * SMS if hd <= 64 else SMS


# (head_dim, N, batch, scale, logit mode, plan).  scale: PRE, LSE or an explicit float.
FWD_CASES = [
    # C3: 64x128 latent, Q prescaled (full batch 32 at N 8192)
    (32, 8192, 32, PRE, "plain", "C3"), (16, 8192, 32, PRE, "plain", "C3"), (64, 2048, 8, PRE, "plain", "C3"),
    (16, 2048, 16, PRE, "plain", "C3"), (128, 512, 32, PRE, "plain", "C3"), (32, 512, 32, PRE, "plain", "C3"),
    (192, 128, 64, PRE, "plain", "C3"), (128, 128, 64, PRE, "plain", "C3"), (64, 128, 64, PRE, "plain", "C3"),
    # C2: 128x256, Q prescaled
    (64, 8192, 2, PRE, "plain", "C2"), (16, 8192, 4, PRE, "plain", "C2"), (128, 2048, 8, PRE, "plain", "C2"),
    (32, 2048, 16, PRE, "plain", "C2"), (192, 512, 16, PRE, "plain", "C2"), (128, 512, 32, PRE, "plain", "C2"),
    (64, 512, 32, PRE, "plain", "C2"),
    # C5: 128x256 training, unscaled Q and the log-sum-exp rows
    (64, 8192, 2, LSE, "plain", "C5"), (16, 8192, 4, LSE, "plain", "C5"), (128, 2048, 8, LSE, "plain", "C5"),
    (32, 2048, 16, LSE, "plain", "C5"), (192, 512, 16, LSE, "plain", "C5"), (128, 512, 32, LSE, "plain", "C5"),
    (64, 512, 32, LSE, "plain", "C5"),
    # legacy UNet at 128x128: explicit scale, head_dim 24 zero-padded to 32
    (24, 1024, 16, LEGACY_SCALE[24], "plain", "legacy"), (24, 256, 48, LEGACY_SCALE[24], "plain", "legacy"),
    (16, 1024, 16, LEGACY_SCALE[16], "plain", "legacy"), (32, 256, 48, LEGACY_SCALE[32], "plain", "legacy"),
    (64, 64, 64, LEGACY_SCALE[64], "plain", "legacy"),
    # ragged N: 8 (one tile, first and ragged), 120 / 136, either side of the three / four-group switch, a four-group tail
    # of 8 tokens (2056), a last four-group CTA with one populated group (2176), 8184; logit extremes
    (16, 8, 64, LSE, "plain", None), (16, 120, 64, PRE, "plain", None), (16, 136, 64, LSE, "grow", None),
    (16, 1016, 16, LSE, "shrink", None), (16, 2040, 16, PRE, "grow", None), (16, 2056, 16, PRE, "plain", None),
    (16, 2176, 16, LSE, "plain", None), (16, 8184, 4, PRE, "big", None), (16, 8184, 2, LSE, "shrink", None),
    (32, 8, 64, PRE, "plain", None), (32, 136, 64, LSE, "plain", None), (32, 520, 32, LSE, "grow", None),
    (32, 2040, 16, LSE, "big", None), (32, 2056, 16, LSE, "plain", None), (32, 2176, 16, PRE, "plain", None),
    (32, 8184, 4, PRE, "grow", None), (32, 8184, 4, LSE, "shrink", None),
    (64, 8, 64, PRE, "plain", None), (64, 200, 64, LSE, "plain", None), (64, 520, 32, PRE, "big", None),
    (64, 2056, 8, LSE, "grow", None), (64, 8184, 2, PRE, "shrink", None),
    (128, 8, 64, LSE, "plain", None), (128, 200, 64, PRE, "grow", None), (128, 520, 32, LSE, "big", None),
    (128, 2056, 8, PRE, "plain", None), (128, 8184, 2, LSE, "grow", None),
    (192, 8, 64, PRE, "plain", None), (192, 200, 32, LSE, "grow", None), (192, 520, 16, PRE, "shrink", None),
    (192, 2056, 4, LSE, "big", None), (192, 8184, 1, PRE, "grow", None),
    # explicit scale > 0 at N >= 2048: the non-UNIT four-group kernel
    (16, 2048, 16, 0.3, "grow", None), (16, 8192, 4, 0.3, "plain", None), (32, 2048, 16, 0.2, "plain", None),
    (32, 8192, 4, 0.3, "big", None),
]

# (head_dim, N, batch, logit mode, plan); the backward runs unscaled Q (training)
BWD_CASES = [
    (64, 8192, 64, "plain", "C5"), (16, 8192, 2, "plain", "C5"), (128, 2048, 4, "plain", "C5"), (32, 2048, 8, "plain", "C5"),
    (192, 512, 16, "plain", "C5"), (128, 512, 16, "plain", "C5"), (64, 512, 32, "plain", "C5"),
    (16, 200, 40, "plain", None), (16, 8184, 2, "grow", None), (32, 520, 20, "plain", None), (32, 2056, 8, "grow", None),
    (32, 136, 64, "plain", None), (64, 8, 64, "plain", None), (64, 200, 40, "grow", None), (64, 2056, 8, "plain", None),
    (128, 520, 16, "plain", None), (128, 8184, 1, "plain", None), (192, 200, 40, "plain", None), (192, 2056, 4, "grow", None),
]


def _id(case):
    return "-".join(str(round(c, 4)) if isinstance(c, float) else str(c) for c in case if c is not None)


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.device("cuda")


def _inputs(hd, N, B, scale, mode, seed, dev):
    """bf16 q, k, v [B,heads,N,hd] (head_dim 24: zero-padded to 32) and the natural-log softmax scale the kernel applies."""
    hdr = 32 if hd == 24 else hd
    g = torch.Generator(device=dev).manual_seed(seed)
    q, k, v = (torch.randn(B, HEADS, N, hdr, device=dev, generator=g) for _ in range(3))
    if hd == 24:
        for t in (q, k, v):
            t[..., 24:] = 0
    if mode == "grow":      # key norms grow with the index: every later tile raises the row maximum
        k = k * torch.linspace(0.25, 14.0, N, device=dev)[:, None]
    elif mode == "big":     # logits of several hundred (log2 units)
        q, k = q * 6.0, k * 6.0
    elif mode == "shrink":  # the largest logits are all in the first tile
        k = k * torch.linspace(14.0, 0.05, N, device=dev)[:, None]
    if scale == PRE:
        q, c = q * (LOG2E / math.sqrt(hd)), LN2
    else:
        c = 1 / math.sqrt(hd) if scale == LSE else scale
    return q.bfloat16(), k.bfloat16(), v.bfloat16(), c


def _run_fwd(q, k, v, scale):
    from weatherconverter_b200 import ops
    vt = v.transpose(2, 3).contiguous()
    if scale == LSE:
        return ops.attention_lse(q, k, vt)
    return ops.attention(q, k, vt, scale=-1.0 if scale == PRE else scale), None


def _pairs(BH, seed):
    """First and last (batch, head) pair plus two random ones."""
    rng = random.Random(seed)
    return sorted({0, BH - 1, rng.randrange(BH), rng.randrange(BH)})


def _chunk(N):
    return max(8, (1 << 24) // N)


def _ref_fwd(q, k, v, c):
    """One (batch, head): q, k, v [N, hd] float64 -> O [N, hd], log-sum-exp [N] in log2 units."""
    N = q.shape[0]
    o, lse = torch.empty_like(q), torch.empty(N, dtype=q.dtype, device=q.device)
    for i in range(0, N, _chunk(N)):
        s = (q[i:i + _chunk(N)] @ k.T) * c
        m = s.amax(1, keepdim=True)
        p = torch.exp(s - m)
        l = p.sum(1, keepdim=True)
        o[i:i + _chunk(N)] = (p @ v) / l
        lse[i:i + _chunk(N)] = (m + l.log()).squeeze(1) / LN2
    return o, lse


def _ref_bwd(q, k, v, do, c):
    """One (batch, head), float64: exact dQ, dK, dV of softmax(c q k^T) v for the output gradient do."""
    N = q.shape[0]
    dq, dk, dv = torch.empty_like(q), torch.zeros_like(k), torch.zeros_like(v)
    for i in range(0, N, _chunk(N)):
        qc, doc = q[i:i + _chunk(N)], do[i:i + _chunk(N)]
        s = (qc @ k.T) * c
        p = torch.exp(s - s.amax(1, keepdim=True))
        p = p / p.sum(1, keepdim=True)
        D = (doc * (p @ v)).sum(1, keepdim=True)
        ds = p * (doc @ v.T - D)
        dq[i:i + _chunk(N)] = (ds @ k) * c
        dk += (ds.T @ qc) * c
        dv += p.T @ doc
    return dq, dk, dv


def _head(t, B, N, hd, b, h, off=0):
    """Rows of head h of image b from a [B, N, x] tensor whose head h occupies columns off + h*hd .. off + h*hd + hd."""
    return t[b, :, off + h * hd: off + (h + 1) * hd]


@pytest.mark.parametrize("hd,N,B,scale,mode,plan", FWD_CASES, ids=[_id(c) for c in FWD_CASES])
def test_forward_vs_float64(hd, N, B, scale, mode, plan):
    dev = _dev()
    seed = hd * 100003 + N * 7 + B
    q, k, v, c = _inputs(hd, N, B, scale, mode, seed, dev)
    o, lse = _run_fwd(q, k, v, scale)
    hdr = q.shape[-1]
    assert torch.isfinite(o.float()).all()
    num = den = 0.0
    worst_row = lse_err = 0.0
    for bh in _pairs(B * HEADS, seed):
        b, h = divmod(bh, HEADS)
        ro, rl = _ref_fwd(q[b, h].double(), k[b, h].double(), v[b, h].double(), c)
        got = _head(o, B, N, hdr, b, h).double()
        d = got - ro
        num += float((d * d).sum())
        den += float((ro * ro).sum())
        worst_row = max(worst_row, float((d.norm(dim=1) / ro.norm(dim=1)).max()))
        if lse is not None:
            lse_err = max(lse_err, float((lse[bh].double() - rl).abs().max()))
    rms = math.sqrt(num / den)
    fam = fwd_family(hd, N, scale)
    print(f"[attn] fwd {fam} {_id((hd, N, B, scale, mode))}: rms-rel {rms:.3e} worst row {worst_row:.3e} lse {lse_err:.3e}")
    assert rms < FWD_RMS[fam], rms
    assert worst_row < FWD_ROW[fam], worst_row
    lse_fam = "general" if fam == "general" else "small" if mode == "plain" else "small-peaked"
    assert lse_err < LSE_ABS[lse_fam], lse_err


@pytest.mark.parametrize("hd,N,B,mode,plan", BWD_CASES, ids=[_id(c) for c in BWD_CASES])
def test_backward_vs_float64(hd, N, B, mode, plan):
    from weatherconverter_b200 import ops
    dev = _dev()
    seed = hd * 100019 + N * 3 + B
    q, k, v, c = _inputs(hd, N, B, LSE, mode, seed, dev)
    C = HEADS * hd
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    do = torch.randn(B, N, C, device=dev, generator=g).bfloat16()
    o, lse = ops.attention_lse(q, k, v.transpose(2, 3).contiguous())
    dqkv = ops.attention_bwd(q, k, v, o, do, lse)
    assert torch.isfinite(dqkv.float()).all()
    errs = {}
    acc = {n: [0.0, 0.0] for n in ("dq", "dk", "dv")}
    for bh in _pairs(B * HEADS, seed):
        b, h = divmod(bh, HEADS)
        ref = _ref_bwd(q[b, h].double(), k[b, h].double(), v[b, h].double(), _head(do, B, N, hd, b, h).double(), c)
        for i, n in enumerate(("dq", "dk", "dv")):
            d = _head(dqkv, B, N, hd, b, h, i * C).double() - ref[i]
            acc[n][0] += float((d * d).sum())
            acc[n][1] += float((ref[i] * ref[i]).sum())
    for n, (num, den) in acc.items():
        errs[n] = math.sqrt(num / den)
    # exact identities over every (batch, head): sum_j dV_j = sum_i dO_i (rows of P sum to 1), sum_j dK_j = 0 (softmax is
    # invariant under a common shift of the keys), in units of 2^-8 sqrt(N) rms(row)
    t = dqkv.double().view(B, N, 3, HEADS, hd)
    unit = 2.0 ** -8 * math.sqrt(N)
    dv_sum, do_sum = t[:, :, 2].sum(1), do.double().view(B, N, HEADS, hd).sum(1)
    sums = {"dv": float(((dv_sum - do_sum).abs() / (unit * t[:, :, 2].pow(2).mean(dim=(1, 3)).sqrt()[..., None])).max()),
            "dk": float((t[:, :, 1].sum(1).abs() / (unit * t[:, :, 1].pow(2).mean(dim=(1, 3)).sqrt()[..., None])).max())}
    print(f"[attn] bwd {_id((hd, N, B, mode))}: rms-rel dq {errs['dq']:.3e} dk {errs['dk']:.3e} dv {errs['dv']:.3e}; "
          f"sums dv {sums['dv']:.3f} dk {sums['dk']:.3f}")
    for n in ("dq", "dk", "dv"):
        assert errs[n] < BWD_RMS[n], (n, errs[n])
    for n in ("dv", "dk"):
        assert sums[n] < BWD_SUM[n], (n, sums[n])


ONES_GEOMS = [(136, LSE), (2040, PRE), (2056, LSE), (8184, PRE)]


@pytest.mark.parametrize("mode", ["big", "grow", "shrink"])
@pytest.mark.parametrize("N,scale", ONES_GEOMS, ids=[f"{n}-{s}" for n, s in ONES_GEOMS])
@pytest.mark.parametrize("hd", [16, 32, 64, 128, 192])
def test_forward_v_ones(hd, N, scale, mode):
    """V = 1: every output is a ratio of the numerator and the row sum, so it is 1 up to the bf16 rounding of the output.  A
    tile lost from l, a masked key counted on one side only, or an offset that rescales O and not l moves it."""
    dev = _dev()
    q, k, _, _ = _inputs(hd, N, 2, scale, mode, hd + N, dev)
    v = torch.ones_like(q)
    o, _ = _run_fwd(q, k, v, scale)
    err = float((o.float() - 1).abs().max())
    assert err <= ONE_TOL, err


BIT_CASES = [(16, 1032, 16, PRE), (16, 2056, 16, PRE), (16, 8184, 4, LSE), (32, 520, 16, LSE), (32, 2176, 8, PRE),
             (32, 2056, 8, 0.3), (64, 2056, 8, LSE), (128, 520, 16, LSE), (192, 200, 32, LSE)]


@pytest.mark.parametrize("hd,N,B,scale", BIT_CASES, ids=[_id(c) for c in BIT_CASES])
def test_bitwise_independence(hd, N, B, scale):
    """Without a reference: slice b of a batch-B launch equals a batch-1 launch of image b, permuting the heads permutes the
    outputs, and a second launch repeats the first bit for bit - output, log-sum-exp and (training cases) dQKV.  Catches
    index mix-ups and interference between CTAs (two backward CTAs per SM, the head-fastest grid, CTAs that skip groups)."""
    from weatherconverter_b200 import ops
    dev = _dev()
    q, k, v, _ = _inputs(hd, N, B, scale, "plain", 5 * hd + N, dev)
    g = torch.Generator(device=dev).manual_seed(N)
    do = torch.randn(B, N, HEADS * hd, device=dev, generator=g).bfloat16()

    def run(q, k, v, do):
        o, lse = _run_fwd(q, k, v, scale)
        return o, lse, (ops.attention_bwd(q, k, v, o, do, lse) if scale == LSE else None)

    def heads_view(t, B):
        return t.view(B, N, -1, HEADS, hd) if t.dim() == 3 else t.view(B, HEADS, N)

    base = run(q, k, v, do)
    again = run(q, k, v, do)
    for x, y in zip(base, again):
        assert x is None or torch.equal(x, y)
    for b in (0, B - 1):
        one = run(q[b:b + 1], k[b:b + 1], v[b:b + 1], do[b:b + 1])
        for x, y in zip(base, one):
            assert x is None or torch.equal(heads_view(x, B)[b], heads_view(y, 1)[0]), b
    perm = [2, 0, 3, 1]
    dop = do.view(B, N, HEADS, hd)[:, :, perm].reshape(B, N, HEADS * hd)
    permuted = run(q[:, perm].contiguous(), k[:, perm].contiguous(), v[:, perm].contiguous(), dop)
    for x, y in zip(base, permuted):
        if x is None:
            continue
        xv, yv = heads_view(x, B), heads_view(y, B)
        for i, p in enumerate(perm):
            assert torch.equal(yv[..., i, :] if x.dim() == 3 else yv[:, i], xv[..., p, :] if x.dim() == 3 else xv[:, p]), i


@pytest.mark.parametrize("hd,N", [(64, 100), (16, 2052), (24, 128), (48, 128), (256, 128)])
def test_guard_rails(hd, N):
    """Unsupported head_dim or N % 8 != 0: every entry point returns the library's error and writes nothing."""
    from weatherconverter_b200._lib import check, lib, ptr, stream_ptr
    dev = _dev()
    B, C = 1, HEADS * hd
    q = torch.randn(B, HEADS, N, hd, device=dev).bfloat16()
    vt = q.transpose(2, 3).contiguous()
    sentinel = 7.0
    out = torch.full((B, N, C), sentinel, device=dev, dtype=torch.bfloat16)
    lse = torch.full((B * HEADS, N), sentinel, device=dev)
    dqkv = torch.full((B, N, 3 * C), sentinel, device=dev, dtype=torch.bfloat16)
    o, do = torch.ones(B, N, C, device=dev).bfloat16(), torch.ones(B, N, C, device=dev).bfloat16()
    scratch = torch.empty(B * HEADS * N, device=dev)
    L = lib()
    with pytest.raises(RuntimeError, match="head_dim|multiple of 8"):
        check(L.wc_attention(ptr(q), ptr(q), ptr(vt), ptr(out), B, HEADS, N, hd, C, stream_ptr()))
    with pytest.raises(RuntimeError, match="head_dim|multiple of 8"):
        check(L.wc_attention_scaled(ptr(q), ptr(q), ptr(vt), ptr(out), B, HEADS, N, hd, C, -1.0, stream_ptr()))
    with pytest.raises(RuntimeError, match="head_dim|multiple of 8"):
        check(L.wc_attention_lse(ptr(q), ptr(q), ptr(vt), ptr(out), ptr(lse), B, HEADS, N, hd, C, stream_ptr()))
    with pytest.raises(RuntimeError, match="head_dim|multiples of 8"):
        check(L.wc_attention_bwd(ptr(q), ptr(q), ptr(q), ptr(o), ptr(do), ptr(lse), ptr(scratch), ptr(dqkv), B, HEADS, N, hd,
                                 stream_ptr()))
    torch.cuda.synchronize()
    assert bool((out.float() == sentinel).all()) and bool((lse == sentinel).all()) and bool((dqkv.float() == sentinel).all())


def _profiled(run):
    """Class-1 (attention) launch records of run(): (work, (BH, N, head_dim) noted by the launcher)."""
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
    return [(work[i], tuple(info[i * 6: i * 6 + 3])) for i in range(n) if cls[i] == 1]


def _shapes(records, B):
    """(head_dim, N) of the forward records; checks each record's work and BH."""
    out = set()
    for w, (bh, N, hd) in records:
        assert bh == B * HEADS and w == 4.0 * bh * N * N * hd, (w, bh, N, hd)
        out.add((hd, N))
    return out


def test_plans_launch_only_tabled_shapes():
    """The inference plans (Q prescaled) at 64x128 and 128x256, the training plan (unscaled Q) forward and backward at 128x256
    and the legacy UNet launch exactly the shapes FWD_CASES / BWD_CASES list for them."""
    from oracle.unet import DEFAULT_MODEL_CONFIG
    from oracle.legacy_unet import legacy_param_spec
    from oracle.weights import synth_state_dict
    from weatherconverter_b200.diffusion_model.models.old_modules import UNet
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet
    dev = _dev()
    tabled = {p: {(32 if hd == 24 else hd, N) for hd, N, _, _, _, plan in FWD_CASES if plan == p} for p in ("C3", "C2", "C5", "legacy")}
    t = torch.tensor([17], device=dev)
    models = {}
    for ims in (64, 128):
        cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = ims
        torch.manual_seed(ims)
        models[ims] = Unet(cfg).to(dev).eval()
    x3, x2 = torch.randn(1, 3, 64, 128, device=dev), torch.randn(1, 3, 128, 256, device=dev)
    assert _shapes(_profiled(lambda: models[64](x3, t)), 1) == tabled["C3"]
    assert _shapes(_profiled(lambda: models[128](x2, t)), 1) == tabled["C2"]

    models[128].differentiable = True
    fwd = _profiled(lambda: models[128](x2, t).backward(torch.ones_like(x2)))
    noted = [r for r in fwd if r[1] != (0, 0, 0)]
    assert _shapes(noted, 1) == tabled["C5"]
    # the backward launchers note nothing: their work is 8 (KV pass) and 6 (dQ pass) x BH N^2 hd of a training forward
    bwd = sorted(w for w, info in fwd if info == (0, 0, 0))
    expect = sorted(f * bh * N * N * hd for _, (bh, N, hd) in noted for f in (8.0, 6.0))
    assert bwd == expect
    assert _shapes(noted, 1) == {(hd, N) for hd, N, _, _, plan in BWD_CASES if plan == "C5"}

    legacy = UNet().to(dev).eval()
    legacy.load_state_dict(synth_state_dict(legacy_param_spec(), 5))
    xl = torch.randn(1, 3, 128, 128, device=dev)
    assert _shapes(_profiled(lambda: legacy(xl, torch.full((1, 1, 1, 1), 0.5, device=dev))), 1) == tabled["legacy"]


def test_dispatch_table_coverage():
    """Every instantiation is reached by a float64-checked case at a plan shape, at a ragged N and with a multi-wave grid."""
    kernels = {fwd_kernel(hd, N, s) for hd in (16, 32, 64, 128, 192) for N in (1024, 4096) for s in (PRE, LSE)}
    kernels |= {k for hd in (16, 32, 64, 128, 192) for k in bwd_kernels(hd)}
    assert len(kernels) == 19
    reach = {k: set() for k in kernels}
    for hd, N, B, scale, _, plan in FWD_CASES:
        kern = fwd_kernel(hd, N, scale)
        reach[kern] |= {"plan"} if plan else set()
        reach[kern] |= {"ragged"} if N % 64 else set()
        reach[kern] |= {"waves"} if fwd_ctas(hd, N, B) > SMS else set()
    for hd, N, B, _, plan in BWD_CASES:
        for kern in bwd_kernels(hd):
            reach[kern] |= {"plan"} if plan else set()
            reach[kern] |= {"ragged"} if N % 64 else set()
            reach[kern] |= {"waves"} if bwd_ctas(hd, N, B) > bwd_wave(hd) else set()
    missing = {k: {"plan", "ragged", "waves"} - r for k, r in reach.items() if r != {"plan", "ragged", "waves"}}
    assert not missing, missing
