"""The stem's BatchNorm handling kernel by kernel, against float64 references at the shapes the model runs.

Two code paths carry the stem's BatchNorms (engine.py:147-262):
  * eval mode folds every BN into the convolutions: pack_weights multiplies each output channel's weights by the BN
    scale (fp16 product, clamped to +-65504), conv_fwd adds the shift as an epilogue bias (+ ReLU, + the block's skip
    connection in conv2);
  * train mode runs the batch statistics (conv_fwd(stats=...) partials -> bn_finalize) and the two-pass BN backward
    (bn_bwd: reduce -> apply; bn_bwd_apply on sums produced elsewhere), plus the max-pool with fused BN + ReLU.

Every reference is a float64 computation on the exact 16-bit operands the kernel consumed, and every comparison is
per element (or per channel for statistics) with a bound derived from the formats:

    |out - ref| <= u_out * |ref| + eta_out + (1 + u_out) * u_acc * mag

where `mag` is the same computation on the magnitudes the kernel's fp32 arithmetic saw.  The older files
(test_gpu_norm_stem.py, test_gpu_gemm.py) compare with `_rel`: the largest error over the largest reference value of
the whole tensor, at 1e-2 .. 3e-2.  That cannot see an error confined to a channel whose values are small (a channel
with gamma 1e-3, a wrong shift of one channel, the Cc term of the BN backward); test_helpers_catch_injected_faults
below shows which injected faults `_rel` lets through and the bounds here do not.
"""
import math
from importlib import import_module

import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu
F16, BF16 = torch.float16, torch.bfloat16

# ---- constants of the bounds ---------------------------------------------------------------------------------------
# unit roundoff of round-to-nearest into the 16-bit output format (half an ulp, relative): 11 / 8 significand bits
U_OUT = {F16: 2.0 ** -11, BF16: 2.0 ** -8}
# absolute floor of that rounding: half the smallest subnormal (fp16 2^-24, bf16 2^-133)
ETA_OUT = {F16: 2.0 ** -25, BF16: 2.0 ** -134}
# fp32 unit roundoff: one IEEE round-to-nearest fp32 operation (the build uses no fast-math)
U32 = 2.0 ** -24
# smallest positive normal fp16: products below it land in the subnormal range
F16_MIN_NORMAL = 2.0 ** -14


def u_mma(K):
    """Accumulation bound of the tcgen05 tap-GEMM over K products, relative to sum |x||w|: the products of 16-bit
    operands are exact in fp32; each kind::f16 MMA step sums k = 16 of them (alignment may truncate: one fp32 ulp,
    2^-23, per addition, <= 16 additions) and adds the block into the fp32 accumulator once (K / 16 steps)."""
    return (K // 16 + 16) * 2.0 ** -23


def out_tol(ref, fmt, err):
    """Per-element bound of a 16-bit store of a value that is within `err` of `ref` before rounding."""
    return U_OUT[fmt] * ref.abs() + ETA_OUT[fmt] + (1 + U_OUT[fmt]) * err


def excess(out, ref, tol):
    """|out - ref| / tol per element (> 1: outside the bound; a non-finite output always is)."""
    out = out.double()
    r = (out - ref.double()).abs() / tol.double().clamp_min(1e-300)     # (a zero bound: only 0 / 0 is inside)
    return torch.where(torch.isfinite(out), r, torch.full_like(r, math.inf))


def assert_within(out, ref, tol, what):
    r = excess(out, ref, tol)
    worst = float(r.max())
    if not worst <= 1.0:
        i = int(r.flatten().argmax())
        idx = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), r.shape))
        raise AssertionError("%s: %d of %d elements outside the bound; worst at %s: out %r ref %r tol %r (x%.3g)" % (
            what, int((r > 1).sum()), r.numel(), idx, float(out.double().flatten()[i]),
            float(ref.double().flatten()[i]), float(tol.double().flatten()[i]), worst))


def _rel_old(a, b):
    """The comparison of test_gpu_norm_stem.py / test_gpu_gemm.py (kept here only to show what it misses)."""
    return float((a.float() - b.float()).abs().max() / (b.float().abs().max() + 1e-12))


def ops():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200.ops")


def nchw(t):
    return t.permute(0, 3, 1, 2)


def nhwc(t):
    return t.permute(0, 2, 3, 1)


def conv64(x_nhwc, w_oihw, ks, sh, sw):
    """float64 convolution of NHWC data (zero padding ks // 2) -> NHWC float64."""
    return nhwc(F.conv2d(nchw(x_nhwc).double(), w_oihw.double(), None, (sh, sw), ks // 2))


def pack_ref(w, scale, fmt):
    """What pack_weights must write for a 'conv' item: torch's fp32 product w * scale[co], clamped to the fp16 range
    when the destination is fp16, rounded once to the destination format, in the [Cout, taps, Cin] layout."""
    p = w * scale.view(-1, 1, 1, 1) if scale is not None else w.clone()
    if fmt == F16:
        p = p.clamp(-65504.0, 65504.0)
    Cout, Cin, kh, kw = w.shape
    return p.to(fmt).permute(0, 2, 3, 1).reshape(Cout, kh * kw, Cin).contiguous()


# ---- BatchNorm backward: the closed form and its bound ------------------------------------------------------------
def bn_bwd_reduce_depth(P, C):
    """fp32 additions on the longest path of bn_bwd's column sums (stem.cu:345-410): a thread sums its rows of one
    CTA (ceil(rows / R)), the CTA sums its R row lanes in shared memory, the CTAs meet in one atomicAdd each; the fma
    g' * (x - mean) adds one more rounding.  CTA count and rows per CTA mirror htrvt_bn_bwd_ctas."""
    G = C // 8
    R = 256 // G
    ctas = min(max((P + 63) // 64, 1), 592)
    rows = -(-P // ctas)
    return -(-rows // R) + R + ctas + 2


def bn_bwd_closed_form(gm, raw, mean, rstd, gamma):
    """float64 d_raw of BN(train) given the masked gradient g' (rows = pixels): gamma rstd (g' - k1 - xhat k2)."""
    P = gm.shape[0]
    xhat = (raw - mean) * rstd
    k1 = gm.sum(0) / P
    k2 = (gm * xhat).sum(0) / P
    return gamma * rstd * (gm - k1 - xhat * k2)


def bn_bwd_tol(gm, raw, mean, rstd, gamma, u_red, ref):
    """Per-element bound of the kernel's d_raw = A g' + Bc raw + Cc (stem.cu:412-415, 437-451, 485).

    gm, raw: float64 [P, C] of the exact 16-bit operands; mean, rstd: float64 [C] of the fp32 statistics the kernel
    was given (the reference graph uses the exact batch statistics, whose fp32 rounding is one U32 of each).
      * coefficients: each of A, Bc, Cc carries at most 6 fp32 roundings (including those of mean, rstd, k1 = s0 / N,
        k2 = s1 / N), the apply's two fmas add 2: 8 U32 on |A g'| + |Bc raw| + |Cc| (Bc raw + Cc cancel when raw is
        near the mean, so the bound is on the terms, not on their sum);
      * column sums: s0 and s1 carry u_red * sum |g'| and u_red * sum |g' xhat| (u_red = reduce depth x U32); s1 also
        sees the fp32 rounding of mean / rstd: U32 (|s1| + |mean| rstd sum |g'|);  d moves by |A| (ds0 + |xhat| ds1) / N."""
    P = gm.shape[0]
    A = (gamma * rstd).abs()
    xhat = (raw - mean) * rstd
    s0, s1 = gm.sum(0), (gm * xhat).sum(0)
    s0a, s1a = gm.abs().sum(0), (gm * xhat).abs().sum(0)
    k1, k2 = s0.abs() / P, s1.abs() / P
    coef = A * (gm.abs() + k1 + (raw.abs() + mean.abs()) * rstd * k2)
    mr = mean.abs() * rstd
    ds0 = u_red * s0a
    ds1 = u_red * (s1a + mr * s0a) + U32 * (s1.abs() + mr * s0a)
    return out_tol(ref, BF16, 8 * U32 * coef + A * (ds0 + xhat.abs() * ds1) / P)


def bn_bwd_stat_tols(gm, raw, mean, rstd, u_red):
    """Per-channel bounds of dbeta = sum g' and dgamma = sum g' xhat (same terms as above, one final fp32 store)."""
    xhat = (raw - mean) * rstd
    s0a, s1a = gm.abs().sum(0), (gm * xhat).abs().sum(0)
    mr = mean.abs() * rstd
    return (u_red + U32) * s0a, (u_red + 2 * U32) * (s1a + mr * s0a)


def pack_mask(m):
    """bool [P, C] -> the ReLU mask bytes bn_act_fwd writes: uint8 [P, C / 8], bit k = channel 8 g + k."""
    P, C = m.shape
    bits = m.view(P, C // 8, 8).to(torch.int32) << torch.arange(8, device=m.device, dtype=torch.int32)
    return bits.sum(-1).to(torch.uint8)


# =====================================================================================================================
# A. the helpers themselves (CPU)
# =====================================================================================================================
def _fault_data():
    """Synthetic outputs of a correct kernel (the float64 value rounded once to the output format) for the 1x1
    downsample conv with its folded shift (K = 192) on two image rows of a 200-pixel line (the second 128-pixel tile of
    each row is ragged: 72 pixels), and for the BN backward at P = 1000, C = 16 with one channel at gamma = 1e-3."""
    g = torch.Generator().manual_seed(0)
    W, K, Co = 200, 192, 32
    x = torch.randn(2 * W, K, generator=g).to(F16).double()
    w = (torch.randn(Co, K, generator=g) / K ** 0.5).to(F16).double()
    bias = torch.randn(Co, generator=g, dtype=torch.float64)
    conv = dict(ref=x @ w.t() + bias, mag=x.abs() @ w.abs().t() + bias.abs(), bias=bias, K=K, W=W)
    P, C = 1000, 16
    raw = (torch.randn(P, C, generator=g, dtype=torch.float64) + 1.0).to(F16).double()   # conv outputs: mean ~ std
    gm = torch.randn(P, C, generator=g, dtype=torch.float64).to(BF16).double()
    gm = gm * (torch.rand(P, C, generator=g, dtype=torch.float64) > 0.5)          # the ReLU mask
    gamma = torch.rand(C, generator=g, dtype=torch.float64) + 0.5
    gamma[7] = 1e-3
    mean, rstd = raw.mean(0), raw.var(0, unbiased=False).add(1e-5).rsqrt()
    ref = bn_bwd_closed_form(gm, raw, mean, rstd, gamma)
    bn = dict(ref=ref, gm=gm, raw=raw, mean=mean, rstd=rstd, gamma=gamma,
              tol=bn_bwd_tol(gm, raw, mean, rstd, gamma, bn_bwd_reduce_depth(P, C) * U32, ref))
    return conv, bn


def test_helpers_catch_injected_faults():
    """Each injected fault must fail the new bound; the table records whether the old `_rel` check at its threshold
    (1e-2 for conv outputs, 3e-2 for the BN-backward d_raw) would have caught it."""
    conv, bn = _fault_data()
    ref, K, W = conv["ref"], conv["K"], conv["W"]
    tol = out_tol(ref, F16, u_mma(K) * conv["mag"])
    good = ref.to(F16)
    assert float(excess(good, ref, tol).max()) <= 1.0
    c = int(conv["bias"].abs().argmax())
    faults = {}
    shifted = ref.clone()
    shifted[:, c] += 1e-3 * conv["bias"][c]                          # one channel's shift off by 1e-3 relative
    faults["shift_1e-3"] = (shifted.to(F16), ref, tol, 1e-2)
    swapped = good.clone()
    swapped[:, [3, 4]] = swapped[:, [4, 3]]                            # two channels swapped
    faults["swap"] = (swapped, ref, tol, 1e-2)
    zeroed = good.clone()
    zeroed[W - 1] = 0                                                  # last row of the ragged tile of image row 0
    faults["ragged_row"] = (zeroed, ref, tol, 1e-2)
    bref, btol = bn["ref"], bn["tol"]
    bgood = bref.to(BF16)
    assert float(excess(bgood, bref, btol).max()) <= 1.0
    small = bref.clone()
    small[:, 7] *= 1.01                                                # 1 % error in the gamma = 1e-3 channel
    faults["small_gamma_1pct"] = (small.to(BF16), bref, btol, 3e-2)
    gm, raw, mean, rstd, gamma = bn["gm"], bn["raw"], bn["mean"], bn["rstd"], bn["gamma"]
    P = gm.shape[0]
    A = gamma * rstd
    k2 = (gm * (raw - mean) * rstd).sum(0) / P
    no_cc = A * gm - A * rstd * k2 * raw                               # A g' + Bc raw, the Cc term dropped
    faults["cc_dropped"] = (no_cc.to(BF16), bref, btol, 3e-2)
    old_caught = {}
    for name, (out, r, t, thr) in faults.items():
        assert float(excess(out, r, t).max()) > 1.0, name
        old_caught[name] = _rel_old(out, r) >= thr
    # recorded: the old check sees the swap and the zeroed row (errors of the tensor's own size) and misses the rest
    assert old_caught == {"shift_1e-3": False, "swap": True, "ragged_row": True, "small_gamma_1pct": False,
                          "cc_dropped": False}, old_caught


# =====================================================================================================================
# B. the eval-mode fold
# =====================================================================================================================
@gpu
@pytest.mark.parametrize("fmt", [F16, BF16])
@pytest.mark.parametrize("ks", [1, 3])
def test_pack_weights_scale_bit_exact(ks, fmt):
    o = ops()
    torch.manual_seed(20 + ks)
    Cout, Cin = 96, 64
    w = torch.randn(Cout, Cin, ks, ks, device="cuda") * 0.05
    scale = torch.randn(Cout, device="cuda") * 3                       # negative scales throughout
    scale[:8] = torch.tensor([2e-6, -2e-6, 1e-5, -3e-4, 1e-7, 4e-6, -6e-6, 8e-5])   # fp16 subnormal products
    w[9].fill_(3.0)
    scale[9] = 4e4                                                     # 1.2e5: beyond the fp16 range (clamped)
    w[10].fill_(-2.5)
    scale[10] = 3e4                                                    # -7.5e4: clamped to -65504
    out = o.pack_weights([(w, "conv", scale)], conv_dtype=fmt)[0]
    ref = pack_ref(w, scale, fmt)
    assert out.dtype == fmt and out.shape == ref.shape
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))
    if fmt == F16:
        sub = (ref.float().abs() < F16_MIN_NORMAL) & (ref != 0)
        assert int(sub.sum()) > 100                                    # the subnormal range was exercised
        assert float(ref[9].float().min()) == 65504.0 and float(ref[10].float().max()) == -65504.0


@gpu
def test_pack_weights_many_tensors_and_reuse():
    """70 tensors (> kMaxPack = 64: the host splits the call into two launches), mixing 'cast' with pad_rows, 'conv'
    with and without a scale and 'convT'; then the reuse= path overwrites the same tensors in place."""
    o = ops()
    torch.manual_seed(21)
    items, names, want = [], [], []

    def fill():
        items.clear(); names.clear()
        for i in range(70):
            kind = ("cast", "conv", "convT", "conv")[i % 4]
            if kind == "cast":
                t = torch.randn(20 + i % 5, 48, device="cuda")
                items.append((t, kind))
            else:
                ks = 3 if i % 3 else 1
                t = torch.randn(16 + 8 * (i % 3), 64, ks, ks, device="cuda") * 0.1
                sc = (torch.randn(t.shape[0], device="cuda") * 4) if (kind == "conv" and i % 8 == 1) else None
                items.append((t, kind, sc) if sc is not None else (t, kind))
            names.append("t%d" % i)

    def expect():
        out = []
        for name, it in zip(names, items):
            t, kind = it[0], it[1]
            if kind == "cast":
                e = t.bfloat16()
                if name in pad:
                    e = torch.cat([e, torch.zeros(pad[name] - t.shape[0], t.shape[1], dtype=BF16, device="cuda")])
            elif kind == "conv":
                e = pack_ref(t, it[2] if len(it) > 2 else None, F16)
            else:
                Co, Ci, kh, kw = t.shape
                e = t.permute(1, 2, 3, 0).reshape(Ci, kh * kw, Co).bfloat16()
            out.append(e)
        return out

    fill()
    pad = {n: 32 for n, it in zip(names, items) if it[1] == "cast" and int(n[1:]) % 8 == 0}
    packed = o.pack_weights(items, pad_rows=pad, names=names)
    for i, (p, e) in enumerate(zip(packed, expect())):
        assert p.dtype == e.dtype and torch.equal(p.view(torch.int16), e.view(torch.int16)), names[i]
    for it in items:                                                   # new parameter values, same tensors
        it[0].copy_(torch.randn_like(it[0]) * 0.2)
        if len(it) > 2:
            it[2].copy_(torch.randn_like(it[2]) * 4)
    again = o.pack_weights(items, pad_rows=pad, names=names, reuse=packed)
    for i, (p, q, e) in enumerate(zip(packed, again, expect())):
        assert q is p and torch.equal(q.view(torch.int16), e.view(torch.int16)), names[i]


# Shapes of conv_fwd: (NB, H, W, Cin, Cout, ks, sh, sw) -> (BN, cluster, reuse) from pick_bn / pick_cluster /
# use_window_reuse (gemm.cu:818-844): BN = 128 for Cout <= 128, 256 when Cout % 256 == 0, else 192 when Cout % 192 == 0;
# CTA pairs (cluster 2) when the M tiles (ceil(Wo / 128) * Ho * NB) are even and >= 4 tiles in all; the window-reuse
# kernel for ks 3, sw 1, cluster 2, BN 192 / 256.
CONV_SHAPES = [
    # every stem conv of the 64 x 512 model (B = 2): layer1 at 16 x 512 -> 8 x 512, layer2 -> 4 x 256, layer3 -> 2 x 128
    (2, 16, 512, 192, 192, 3, 2, 1),   # layer1.0.conv1   64 M tiles: BN 192, cluster 2, reuse
    (2, 16, 512, 192, 192, 1, 2, 1),   # layer1.0 ds      64:        BN 192, cluster 2
    (2, 8, 512, 192, 192, 3, 1, 1),    # layer1.x.conv2   64:        BN 192, cluster 2, reuse
    (2, 8, 512, 192, 384, 3, 2, 2),    # layer2.0.conv1   16:        BN 192, cluster 2
    (2, 8, 512, 192, 384, 1, 2, 2),    # layer2.0 ds      16:        BN 192, cluster 2
    (2, 4, 256, 384, 384, 3, 1, 1),    # layer2.x.conv2   16:        BN 192, cluster 2, reuse
    (2, 4, 256, 384, 768, 3, 2, 2),    # layer3.0.conv1    4:        BN 256, cluster 2
    (2, 4, 256, 384, 768, 1, 2, 2),    # layer3.0 ds       4:        BN 256, cluster 2
    (2, 2, 128, 768, 768, 3, 1, 1),    # layer3.x.conv2    4:        BN 256, cluster 2, reuse
    # the same convs on a 1000-pixel line (outputs 8 x 1000, 4 x 500, 2 x 250: the last M tile of a row is ragged)
    (1, 16, 1000, 192, 192, 3, 2, 1),  # 64 M tiles (last 104 rows): BN 192, cluster 2, reuse
    (1, 16, 1000, 192, 192, 1, 2, 1),  # 64:                         BN 192, cluster 2
    (1, 8, 1000, 192, 192, 3, 1, 1),   # 64:                         BN 192, cluster 2, reuse
    (1, 8, 1000, 192, 384, 3, 2, 2),   # 16 (last 116 rows):         BN 192, cluster 2
    (1, 8, 1000, 192, 384, 1, 2, 2),   # 16:                         BN 192, cluster 2
    (1, 4, 500, 384, 384, 3, 1, 1),    # 16:                         BN 192, cluster 2, reuse
    (1, 4, 500, 384, 768, 3, 2, 2),    # 4 (last 122 rows):          BN 256, cluster 2
    (1, 4, 500, 384, 768, 1, 2, 2),    # 4:                          BN 256, cluster 2
    (1, 2, 250, 768, 768, 3, 1, 1),    # 4:                          BN 256, cluster 2, reuse
    # Cout = 128
    (2, 8, 200, 64, 128, 3, 1, 1),     # 32 M tiles:                 BN 128, cluster 2
    (2, 8, 200, 128, 128, 1, 2, 2),    # 8:                          BN 128, cluster 2
    # an odd number of M tiles: the single-CTA kernel
    (3, 1, 128, 192, 192, 3, 1, 1),    # 3 M tiles:                  BN 192, cluster 1 (no reuse without pairs)
    (1, 3, 300, 384, 768, 3, 1, 1),    # 9:                          BN 256, cluster 1
    (1, 5, 100, 64, 128, 3, 1, 1),     # 5:                          BN 128, cluster 1
    (1, 6, 250, 192, 384, 1, 2, 2),    # 3:                          BN 192, cluster 1
]


@gpu
@pytest.mark.parametrize("fmt", [F16, BF16])
@pytest.mark.parametrize("NB,H,W,Cin,Cout,ks,sh,sw", CONV_SHAPES)
def test_conv_fwd_epilogues(NB, H, W, Cin, Cout, ks, sh, sw, fmt):
    """conv_fwd with no epilogue, bias, bias + ReLU and bias + residual + ReLU (conv2 of a folded block), per element
    against float64: the bias is the folded BN shift (fp32), the residual a 16-bit tensor like y."""
    o = ops()
    torch.manual_seed(NB * 1000 + W + Cout + ks)
    K = ks * ks * Cin
    x = torch.randn(NB, H, W, Cin, device="cuda").to(fmt)
    w = (torch.randn(Cout, Cin, ks, ks, device="cuda") / K ** 0.5).to(fmt)
    wk = w.permute(0, 2, 3, 1).reshape(Cout, ks * ks, Cin).contiguous()
    conv = conv64(x, w, ks, sh, sw)
    mag = conv64(x.abs(), w.abs(), ks, sh, sw)
    Ho, Wo = conv.shape[1:3]
    bias = torch.randn(Cout, device="cuda") * 2
    bias[::5] *= 1e-3                                                 # shifts much smaller than the conv output too
    res = torch.randn(NB, Ho, Wo, Cout, device="cuda").to(fmt)
    b64, r64 = bias.double(), res.double()
    cases = [("none", {}, conv, mag),
             ("bias", dict(bias=bias), conv + b64, mag + b64.abs()),
             ("bias_relu", dict(bias=bias, relu=True), (conv + b64).clamp_min(0), mag + b64.abs()),
             ("bias_res_relu", dict(bias=bias, res=res, relu=True), (conv + b64 + r64).clamp_min(0),
              mag + b64.abs() + r64.abs())]
    for name, kw, ref, m in cases:
        y = torch.full((NB, Ho, Wo, Cout), 7.0, device="cuda", dtype=fmt)
        y = o.conv_fwd(x, wk, ks, sh, sw, y=y, **kw)
        assert y.dtype == fmt and y.shape == ref.shape
        # u_mma covers the K-term accumulation; the fp32 adds of bias and residual are 2 U32 <= u_mma(K) of |bias| + |res|
        assert_within(y, ref, out_tol(ref, fmt, u_mma(K) * m), "%s %s" % (name, fmt))


# (Cin, Cout, stride, H, W of the block's input, downsample): both blocks of each stem layer
FOLD_BLOCKS = [
    (192, 192, (2, 1), 16, 256, True),    # layer1.0
    (192, 192, (1, 1), 8, 256, False),    # layer1.1
    (192, 384, (2, 2), 8, 256, True),     # layer2.0
    (384, 384, (1, 1), 4, 128, False),    # layer2.1
    (384, 768, (2, 2), 4, 128, True),     # layer3.0
    (768, 768, (1, 1), 2, 64, False),     # layer3.1
]


def _hostile_bn(C, gen_seed):
    """BatchNorm parameters spanning realistic and hostile values: running_var from 1e-4 to 10 (log-uniform), gamma
    of both signs with every seventh channel near zero, running_mean and beta of order one."""
    g = torch.Generator(device="cuda").manual_seed(gen_seed)
    rv = 10.0 ** (torch.rand(C, device="cuda", generator=g) * 5 - 4)
    gamma = torch.randn(C, device="cuda", generator=g)
    gamma[::7] = torch.randn(gamma[::7].shape, device="cuda", generator=g) * 1e-3
    beta = torch.randn(C, device="cuda", generator=g) * 0.5
    rm = torch.randn(C, device="cuda", generator=g) * 0.5
    return gamma, beta, rm, rv


def _fold_stage(xabs, xerr, w_oihw, scale64, ks, s, extra_abs):
    """float64 magnitude and error bound (before the output rounding) of one folded conv: input magnitude / error
    per element, weights w * scale rounded once to fp16 (u + 8 U32 relative: the fp32 BN scale carries 5.5 U32 - see
    test_bn_finalize_eval - and the fp32 product one more; + ETA absolute for subnormal products), the accumulation (u_mma) and the fp32 shift / residual."""
    wabs = (w_oihw.double() * scale64.view(-1, 1, 1, 1)).abs()
    dw = (U_OUT[F16] + 8 * U32) * wabs + ETA_OUT[F16]
    K = ks * ks * w_oihw.shape[1]
    mag = conv64(xabs, wabs, ks, *s)
    err = conv64(xerr, wabs + dw, ks, *s) + conv64(xabs, dw, ks, *s) + u_mma(K) * (mag + extra_abs)
    return mag, err


@gpu
@pytest.mark.parametrize("Cin,Cout,stride,H,W,ds", FOLD_BLOCKS)
def test_folded_basic_block(Cin, Cout, stride, H, W, ds):
    """The three launches engine.forward makes for one eval-mode BasicBlock (engine.py:225-230: conv1 + shift + ReLU,
    the 1x1 downsample + shift, conv2 + shift + skip + ReLU) against a float64 F.batch_norm(training=False) graph of the
    block.  The bound propagates per element: each stage's error goes through the next convolution's |w'|."""
    o = ops()
    torch.manual_seed(Cin + Cout + H)
    eps = 1e-5
    x = torch.relu(torch.randn(1, H, W, Cin, device="cuda")).to(F16)          # a post-ReLU activation
    w1 = torch.randn(Cout, Cin, 3, 3, device="cuda") / (9 * Cin) ** 0.5
    wd = torch.randn(Cout, Cin, 1, 1, device="cuda") / Cin ** 0.5
    bns = [_hostile_bn(Cout, 100 * i + Cout) for i in range(3)]
    # conv2's weights are scaled to the rms of what bn1 produces (as training would leave them): bn1's scales of up to
    # ~300 (running_var 1e-4) would otherwise push bn2's output past the fp16 range - a format limit, not a kernel error
    g1, b1, rm1, rv1 = bns[0]
    a1_rms = float(torch.relu(conv64(x, w1, 3, *stride) * (g1 / (rv1 + 1e-5).sqrt()).double() +
                              (b1 - rm1 * g1 / (rv1 + 1e-5).sqrt()).double()).square().mean().sqrt())
    w2 = torch.randn(Cout, Cout, 3, 3, device="cuda") / (9 * Cout) ** 0.5 / max(a1_rms, 1e-3)
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    st = [o.bn_finalize(None, 1, g, b, rm, rv, nbt, False) for g, b, rm, rv in bns]
    assert int(nbt) == 0
    items = [(w1, "conv", st[0][2]), (w2, "conv", st[1][2])] + ([(wd, "conv", st[2][2])] if ds else [])
    wp = o.pack_weights(items)
    a1 = o.conv_fwd(x, wp[0], 3, stride[0], stride[1], relu=True, bias=st[0][3])
    skip = o.conv_fwd(x, wp[2], 1, stride[0], stride[1], bias=st[2][3]) if ds else x
    y = o.conv_fwd(a1, wp[1], 3, 1, 1, relu=True, bias=st[1][3], res=skip)

    def bn64(z, p):
        g, b, rm, rv = (t.double() for t in p)
        return nhwc(F.batch_norm(nchw(z), rm, rv, g, b, False, 0.0, eps))

    def fold(p):                                                     # float64 scale / shift, |shift| bound terms
        g, b, rm, rv = (t.double() for t in p)
        sc = g / (rv + eps).sqrt()
        sh = b - rm * sc
        return sc, sh, U32 * (b.abs() + 8 * (rm * sc).abs())          # test_bn_finalize_eval's shift bound

    x64 = x.double()
    a1_ref = torch.relu(bn64(conv64(x64, w1, 3, *stride), bns[0]))
    sc1, sh1, dsh1 = fold(bns[0])
    _, e1 = _fold_stage(x64.abs(), torch.zeros_like(x64), w1, sc1, 3, stride, sh1.abs())
    tol1 = out_tol(a1_ref, F16, e1 + dsh1)
    assert_within(a1, a1_ref, tol1, "conv1 + bn1 + relu")
    if ds:
        skip_ref = bn64(conv64(x64, wd, 1, *stride), bns[2])
        scd, shd, dshd = fold(bns[2])
        _, ed = _fold_stage(x64.abs(), torch.zeros_like(x64), wd, scd, 1, stride, shd.abs())
        tol_s = out_tol(skip_ref, F16, ed + dshd)
        assert_within(skip, skip_ref, tol_s, "downsample + bn")
    else:
        skip_ref, tol_s = x64, torch.zeros_like(x64)
    y_ref = torch.relu(bn64(conv64(a1_ref, w2, 3, 1, 1), bns[1]) + skip_ref)
    sc2, sh2, dsh2 = fold(bns[1])
    _, e2 = _fold_stage(a1_ref.abs(), tol1, w2, sc2, 3, (1, 1), sh2.abs() + skip_ref.abs() + tol_s)
    assert_within(y, y_ref, out_tol(y_ref, F16, e2 + dsh2 + tol_s), "conv2 + bn2 + skip + relu")


@gpu
@pytest.mark.parametrize("C", [13, 192, 2048])
def test_bn_finalize_eval(C):
    """Running-statistics coefficients: mean = running_mean exactly; rstd = rsqrtf(var + eps) within rsqrtf's 2 ulp
    (4 U32) plus the rounding of var + eps (U32 / 2); scale one more U32; shift = beta - mean scale two more."""
    o = ops()
    gamma, beta, rm, rv = _hostile_bn(C, C)
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    st = o.bn_finalize(None, 1, gamma, beta, rm, rv, nbt, False)
    assert int(nbt) == 0
    g, b, m, v = (t.double() for t in (gamma, beta, rm, rv))
    rstd = 1 / (v + 1e-5).sqrt()
    sc = g * rstd
    assert torch.equal(st[0], rm)
    assert_within(st[1], rstd, 4.5 * U32 * rstd, "rstd")
    assert_within(st[2], sc, 5.5 * U32 * sc.abs(), "scale")
    shift = b - m * sc
    assert_within(st[3], shift, U32 * shift.abs() + 7.5 * U32 * (m * sc).abs(), "shift")


# =====================================================================================================================
# C. the train-mode kernels at ragged splits
# =====================================================================================================================
# (P, C): reduce grid = ceil(P / 64) CTAs (<= 592) of `rows` rows, R = 256 / (C / 8) row lanes of 4-row groups; the
# apply pass walks n8 = P C / 8 groups in pairs of 256-group runs over <= 592 CTAs
BN_BWD_SHAPES = [
    (37, 192),       # one CTA; G = 24, R = 10: 256 % G != 0 (240 threads)
    (1000, 64),      # 16 CTAs x 63 rows (rows do not divide P: last CTA 55); n8 % 512 = 320
    (4099, 8),       # G = 1, R = 256: 65 CTAs, last holds 3 rows (< 4R = 1024); n8 % 512 = 3 (< 256)
    (3001, 384),     # G = 48, R = 5: last CTA 57 rows (not a multiple of 4R = 20); n8 % 512 = 176 (< 256)
    (9999, 768),     # G = 96, R = 2: last CTA 15 rows (< 2 x 4R); n8 % 512 = 416; 4 apply iterations
    (1531, 2048),    # G = 256 (the ABI limit), R = 1: last CTA 59 rows; 2 apply iterations
    (100003, 64),    # 592 CTAs x 169 rows, last 124 (< 4R = 128); n8 = 800024 > 592 x 512: 3 apply iterations
]


def _bn_bwd_check(o, P, C, mode, fmt, seed):
    torch.manual_seed(seed)
    dev = "cuda"
    eps = 1e-5

    def make_raw():
        mu = torch.randn(C, device=dev) * 3                        # non-zero channel means (raw conv outputs)
        sd = torch.rand(C, device=dev) * 2 + 0.1
        return (torch.randn(P, C, device=dev) * sd + mu).to(fmt)

    def stats(raw):                                                # what bn_finalize hands the backward: fp32
        r = raw.double()
        m, v = r.mean(0), r.var(0, unbiased=False)
        return torch.stack([m.float(), (v + eps).rsqrt().float()])

    def gammas():
        g = torch.randn(C, device=dev)
        g[::5] = 1e-3 * torch.sign(g[::5])                          # small-gamma channels, both signs
        return g

    raw_a, ga = make_raw(), gammas()
    sa, ba = stats(raw_a), torch.randn(C, device=dev)
    raw_b = make_raw() if mode == "ds" else None
    gb = gammas() if mode == "ds" else None
    sb = stats(raw_b) if mode == "ds" else None
    xres = torch.randn(P, C, device=dev).to(fmt) if mode == "gz" else None
    g = torch.randn(P, C, device=dev).bfloat16()

    # float64 autograd graph: BN(train) [+ BN(train) | + residual] -> ReLU
    ra = raw_a.double().requires_grad_(True)
    ga64 = ga.double().requires_grad_(True)
    ba64 = ba.double().requires_grad_(True)
    pre = F.batch_norm(ra, None, None, ga64, ba64, True, 0.0, eps)
    if mode == "ds":
        rb = raw_b.double().requires_grad_(True)
        gb64 = gb.double().requires_grad_(True)
        bb64 = torch.zeros(C, dtype=torch.float64, device=dev, requires_grad=True)
        pre = pre + F.batch_norm(rb, None, None, gb64, bb64, True, 0.0, eps)
    elif mode == "gz":
        pre = pre + xres.double()
    mask = pre.detach() > 0
    torch.relu(pre).backward(g.double())
    km = pack_mask(mask)
    gm = g.double() * mask

    dga, dba = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    dgb, dbb = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    if mode == "ds":
        d_a, d_b, gz = o.bn_bwd(g, km, raw_a, sa, ga, dga, dba, raw_b=raw_b, st_b=sb, gamma_b=gb, dgamma_b=dgb,
                                dbeta_b=dbb)
    else:
        d_a, d_b, gz = o.bn_bwd(g, km, raw_a, sa, ga, dga, dba, want_gz=(mode == "gz"))
    u_red = bn_bwd_reduce_depth(P, C) * U32
    for name, d, raw, st, gam, ref, dgam, dbet, gref, bref in (
            [("a", d_a, raw_a, sa, ga, ra.grad, dga, dba, ga64.grad, ba64.grad)] +
            ([("b", d_b, raw_b, sb, gb, rb.grad, dgb, dbb, gb64.grad, bb64.grad)] if mode == "ds" else [])):
        r64, m64, s64 = raw.double(), st[0].double(), st[1].double()
        assert d.dtype == BF16 and d.shape == raw.shape
        assert_within(d, ref, bn_bwd_tol(gm, r64, m64, s64, gam.double(), u_red, ref), "d_%s %s" % (name, mode))
        tb, tg = bn_bwd_stat_tols(gm, r64, m64, s64, u_red)
        assert_within(dbet, bref, tb, "dbeta_%s" % name)
        assert_within(dgam, gref, tg, "dgamma_%s" % name)
    if mode == "gz":
        assert torch.equal(gz, (g.float() * mask).bfloat16())
    else:
        assert gz is None

    # bn_bwd_apply on sums produced elsewhere (the fused dgrad epilogue): fp32 [3, C] of the float64 sums
    r64, m64, s64 = raw_a.double(), sa[0].double(), sa[1].double()
    sums = torch.stack([gm.sum(0), (gm * (r64 - m64) * s64).sum(0), torch.zeros_like(m64)]).float().contiguous()
    dg2, db2 = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
    d2 = o.bn_bwd_apply(gm.bfloat16(), raw_a, sa, ga, dg2, db2, sums.view(-1))
    assert torch.equal(dg2, sums[1]) and torch.equal(db2, sums[0])
    # the sums reach the apply pass rounded once to fp32 (u_red = U32) and already hold the fp32 mean / rstd
    assert_within(d2, ra.grad, bn_bwd_tol(gm, r64, m64, s64, ga.double(), U32, ra.grad), "bn_bwd_apply")


@gpu
@pytest.mark.parametrize("fmt", [F16, BF16])
@pytest.mark.parametrize("mode", ["single", "ds", "gz"])
@pytest.mark.parametrize("P,C", BN_BWD_SHAPES)
def test_bn_bwd_ragged(P, C, mode, fmt):
    """bn_bwd alone, with the downsample branch (raw_b) and with want_gz, then bn_bwd_apply on the same data: d_a,
    d_b per element, gz exactly, dgamma / dbeta per channel, against float64 autograd of BN(train) -> add -> ReLU."""
    _bn_bwd_check(ops(), P, C, mode, fmt, P + C)


@gpu
def test_bn_bwd_full_size():
    """layer1's BatchNorm at B = 128 of 64 x 512 lines: P = 524288, C = 192 (592 CTAs of 886 rows, last 662; n8 =
    12582912, 42 iterations of the apply pass), with the downsample branch."""
    _bn_bwd_check(ops(), 524288, 192, "ds", F16, 7)


def _finalize_bounds(part, count, R):
    """float64 reference and per-channel bounds of bn_finalize(training=True) on fp32 partials [R, 2, C].

    The kernel sums each channel's rows in fp32 (four accumulators per lane, ceil(R / 512) + 3 additions at most,
    stem.cu:131-146) and the rest in float64: the sums carry u_red = (ceil(R / 512) + 4) U32 of sum |s_r| and of sum
    q_r.  var = Q / N - mean^2 in float64 then inherits dQ / N + 2 |mean| dS / N; rstd = rsqrtf(var + eps) adds 4 U32
    (rsqrtf's 2 ulp) and U32 for each fp32 rounding of var, var + eps."""
    p = part.double()
    S, Q = p[:, 0].sum(0), p[:, 1].sum(0)
    Sa = p[:, 0].abs().sum(0)
    u_red = (-(-R // 512) + 4) * U32
    mean = S / count
    var = Q / count - mean * mean
    dmean = u_red * Sa / count
    dvar = u_red * Q / count + 2 * mean.abs() * dmean + dmean * dmean
    ve = var + 1e-5
    t = (dvar + 2 * U32 * ve) / ve                                   # relative error of var + eps as the kernel sees it
    rstd = ve.rsqrt()
    return mean, var, rstd, dmean + U32 * mean.abs(), dvar + U32 * var.abs(), t, rstd * (t + 4 * U32)


@gpu
@pytest.mark.parametrize("C", [13, 192])
@pytest.mark.parametrize("R", [1, 127, 128, 129, 384, 385, 512, 513, 2000])
def test_bn_finalize_train(R, C):
    """Batch statistics from R partial rows (the four-way unrolled loop engages at R > 384), C = 13 (not a multiple
    of 8), three consecutive calls: mean / rstd / scale / shift and the momentum update of running_mean and the
    unbiased running_var, per channel against float64; num_batches_tracked counts the calls."""
    o = ops()
    torch.manual_seed(R * 7 + C)
    n = 64                                                           # pixels behind each partial row
    count = R * n
    gamma, beta, rm0, rv0 = _hostile_bn(C, R + C)
    rm, rv = rm0.clone(), rv0.clone()
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    rm64, rv64 = rm0.double(), rv0.double()
    drm = torch.zeros(C, dtype=torch.float64, device="cuda")
    drv = torch.zeros_like(drm)
    mom = 0.1
    for call in range(3):
        mu = torch.randn(C, device="cuda", dtype=torch.float64) * 2
        data = torch.randn(R, n, C, device="cuda", dtype=torch.float64) * (torch.rand(C, device="cuda") + 0.2) + mu
        part = torch.stack([data.sum(1), (data * data).sum(1)], 1).float().contiguous()
        st = o.bn_finalize(part, count, gamma, beta, rm, rv, nbt, True, momentum=mom)
        assert int(nbt) == call + 1
        mean, var, rstd, dmean, dvar, t, drstd = _finalize_bounds(part, count, R)
        assert float(t.max()) < 0.5                   # |1 / sqrt(1 + t) - 1| <= |t| needs |t| <= 1/2 (see _finalize_bounds)
        assert_within(st[0], mean, dmean, "mean (call %d)" % call)
        assert_within(st[1], rstd, drstd, "rstd (call %d)" % call)
        g64, b64 = gamma.double(), beta.double()
        sc = g64 * rstd
        assert_within(st[2], sc, g64.abs() * drstd + U32 * sc.abs() * 2, "scale")
        dsc = g64.abs() * drstd + 2 * U32 * sc.abs()
        sh = b64 - mean * sc
        assert_within(st[3], sh, dmean * sc.abs() + mean.abs() * dsc + 3 * U32 * (b64.abs() + (mean * sc).abs()),
                      "shift")
        # momentum update in fp32: (1 - m) r + m x, three roundings on each term's magnitude
        m32 = float(torch.tensor(mom, dtype=torch.float32))
        unb = var * count / (count - 1)
        rm64 = (1 - m32) * rm64 + m32 * mean
        rv64 = (1 - m32) * rv64 + m32 * unb
        drm = (1 - m32) * drm + m32 * dmean + 3 * U32 * rm64.abs() + U32 * mean.abs()
        drv = (1 - m32) * drv + m32 * dvar * count / (count - 1) + 3 * U32 * rv64.abs() + U32 * unb.abs()
        assert_within(rm, rm64, drm, "running_mean (call %d)" % call)
        assert_within(rv, rv64, drv, "running_var (call %d)" % call)
    o.bn_finalize(None, 1, gamma, beta, rm, rv, nbt, False)
    assert int(nbt) == 3                                             # eval mode counts nothing


@gpu
@pytest.mark.parametrize("ratio", [0.0, 3.0, 25.0, 100.0, 300.0])
def test_bn_finalize_large_mean(ratio):
    """The variance comes from E[x^2] - E[x]^2 over fp32 partial sums (stem.cu:158-160): it cancels when |mean| is
    large against the std.  With every row of the partials an exact fp32 value, the derived bound holds at any ratio;
    for R = 2000 rows it keeps rstd within 1e-3 relative up to |mean| / std = 25 (dvar / var ~ 3 u_red ratio^2 with
    u_red = 8 U32), and it stops holding at all (dvar / var > 1/2: the computed variance may be 0 and rstd 1 / sqrt(eps))
    from |mean| / std ~ 590.  The ratios above 25 are run to show that the kernel stays inside the wider bound, which
    is then asserted only where it is meaningful."""
    o = ops()
    torch.manual_seed(int(ratio) + 1)
    R, n, C = 2000, 64, 64
    std = torch.rand(C, device="cuda", dtype=torch.float64) + 0.5
    mu = std * ratio * torch.sign(torch.randn(C, device="cuda", dtype=torch.float64))
    data = torch.randn(R, n, C, device="cuda", dtype=torch.float64) * std + mu
    part = torch.stack([data.sum(1), (data * data).sum(1)], 1).float().contiguous()
    gamma, beta = torch.ones(C, device="cuda"), torch.zeros(C, device="cuda")
    st = o.bn_finalize(part, R * n, gamma, beta, None, None, None, True)
    mean, var, rstd, dmean, dvar, t, drstd = _finalize_bounds(part, R * n, R)
    assert_within(st[0], mean, dmean, "mean")
    ok = t < 0.5
    assert_within(st[1][ok], rstd[ok], drstd[ok], "rstd")
    if ratio <= 25.0:
        assert bool(ok.all()) and float((drstd / rstd).max()) <= 1e-3


# (NB, H, W, Cin, Cout, ks, sh, sw): widths whose last M tile is ragged, so rows past Wo exist in the tile
STATS_SHAPES = [
    (2, 8, 200, 64, 128, 3, 1, 1),      # Wo 200 = 128 + 72: BN 128, cluster 2
    (1, 16, 1000, 192, 192, 3, 2, 1),   # Wo 1000, last tile 104 rows: BN 192, cluster 2, reuse
    (1, 8, 1000, 192, 384, 1, 2, 2),    # Wo 500, last tile 116 rows: BN 192, cluster 2
    (1, 4, 500, 384, 768, 3, 2, 2),     # Wo 250, last tile 122 rows: BN 256, cluster 2
    (3, 1, 100, 64, 128, 3, 1, 1),      # Wo 100 < one tile, 3 M tiles: BN 128, cluster 1
]


@gpu
@pytest.mark.parametrize("fmt", [F16, BF16])
@pytest.mark.parametrize("NB,H,W,Cin,Cout,ks,sh,sw", STATS_SHAPES)
def test_conv_stats_partials_ragged(NB, H, W, Cin, Cout, ks, sh, sw, fmt):
    """conv_fwd(stats=...): per-channel sum and sum of squares of what is stored, against float64 of the stored
    output.  Inputs and weights have non-zero means, so a row past Wo that leaked into the sums would move them far
    outside the bound.  Each value enters one 32-row warp sum and then the CTA's running sum over the tiles it owns:
    the CTA's row of the partials gets one more addition per change of n-tile: (32 + 2 x M tiles + 1) fp32
    additions bound the error, on sum |y| and sum y^2."""
    o = ops()
    torch.manual_seed(W + Cout)
    K = ks * ks * Cin
    x = (torch.randn(NB, H, W, Cin, device="cuda") + 1.5).to(fmt)
    w = (torch.randn(Cout, Cin, ks, ks, device="cuda") / K ** 0.5 + 0.02).to(fmt)
    wk = w.permute(0, 2, 3, 1).reshape(Cout, ks * ks, Cin).contiguous()
    stats = torch.zeros(o.conv_stats_rows(NB, H, W, ks, sh, sw), 2, Cout, device="cuda")
    y = o.conv_fwd(x, wk, ks, sh, sw, stats=stats)
    Ho, Wo = y.shape[1:3]
    tiles_m = -(-Wo // 128) * Ho * NB
    y64 = y.double().reshape(-1, Cout)
    S, Q = stats.double().sum(0)
    u = (32 + 2 * tiles_m + 1) * U32
    assert_within(S, y64.sum(0), u * y64.abs().sum(0), "column sums")
    assert_within(Q, (y64 * y64).sum(0), u * (y64 * y64).sum(0), "column sums of squares")


# (B, H, W, C): odd H (Ho = (H - 1) / 2 + 1), W = 1 and 2, C = 8
POOL_SHAPES = [(2, 7, 1, 8), (3, 5, 2, 8), (2, 9, 33, 8), (1, 8, 2, 16), (2, 1, 5, 8)]


def _round_to(v32, fmt):
    return v32.to(fmt).double()


@gpu
@pytest.mark.parametrize("fmt", [F16, BF16])
@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("B,H,W,C", POOL_SHAPES)
def test_pool_fwd_bwd_edges(B, H, W, C, fused, fmt):
    """max-pool 3x3, stride (2, 1), pad 1, optionally over relu(raw scale + shift) (the stem head's fused BN + ReLU):
    the forward equals the reference bit for bit, arg-max codes included (first maximum in kh * 3 + kw order: many
    ReLU zeros and quantised raw values make ties); the backward sums at most 6 gradient terms (2 rows x 3 columns of
    windows) in fp32 and rounds once to bf16: bound u_bf16 |ref| + 6 U32 sum |terms|."""
    o = ops()
    torch.manual_seed(B * 100 + H * 10 + W + int(fused))
    raw = (torch.randint(-3, 4, (B, H, W, C), device="cuda").float() * 0.5).to(fmt)
    st = None
    a = raw.double()
    if fused:
        raw = (torch.randn(B, H, W, C, device="cuda") * 2).to(fmt)
        scale = torch.randn(C, device="cuda")
        scale[0] = -1.5
        shift = torch.randn(C, device="cuda") * 0.5
        st = (None, None, scale, shift)
        v = raw.double() * scale.double() + shift.double()            # exact fma value; the kernel rounds it to fp32
        a = _round_to(v.float().clamp_min(0), fmt)                   # then applies ReLU and rounds to the 16-bit format
    Ho = (H - 1) // 2 + 1
    ap = F.pad(a, (0, 0, 1, 1, 1, 1), value=-math.inf)               # [B, H + 2, W + 2, C]
    win = torch.stack([ap[:, kh:kh + 2 * Ho - 1:2, kw:kw + W] for kh in range(3) for kw in range(3)])
    ref_out, ref_idx = win.max(0).values, win.argmax(0)               # argmax: the first maximal value
    out, idx = o.pool_fwd(raw, st, True)
    assert out.dtype == fmt and out.shape == (B, Ho, W, C)
    assert torch.equal(out.double(), ref_out)
    assert torch.equal(idx.long(), ref_idx)
    for gtype in (torch.float32, BF16):
        gout = torch.randn(B, Ho, W, C, device="cuda").to(gtype)
        gin = o.pool_bwd(gout, idx, (B, H, W, C), raw=raw if fused else None, st=st)
        acc = torch.zeros(B, H + 2, W + 2, C, dtype=torch.float64, device="cuda")
        mag = torch.zeros_like(acc)
        for k in range(9):
            kh, kw = divmod(k, 3)
            sel = gout.double() * (ref_idx == k)
            acc[:, kh:kh + 2 * Ho - 1:2, kw:kw + W] += sel
            mag[:, kh:kh + 2 * Ho - 1:2, kw:kw + W] += sel.abs()
        ref, mag = acc[:, 1:H + 1, 1:W + 1], mag[:, 1:H + 1, 1:W + 1]
        if fused:
            keep = v > 0
            ref, mag = ref * keep, mag * keep
        assert gin.dtype == BF16
        assert_within(gin, ref, out_tol(ref, BF16, 6 * U32 * mag), "pool_bwd %s" % gtype)
