"""The transformer's normalisation, token, GELU, column-sum and v1 attention kernels one by one, against float64.

Kernels: csrc/norm.cu (row and whole-sample LayerNorm, tokens, GELU, mul_bf16, colsum_bf16, cast_colsum_bf16), the
GELU pieces of common.cuh as the tap-GEMM epilogues use them, csrc/attention.cu (v1 attention) and the fp32 twins in
csrc/exact.cu (row_ln_f32, tokens_f32, attention_f32).  Every reference is float64 on the exact fp32 / 16-bit values
the kernel read; every comparison is per element (per row or column for statistics) against a bound built from the
formats (fp_bounds.py): the output format's half ulp, fp32 roundings along the longest summation path of the kernel
(its "depth", counted from the code), and the documented error of the approximations it uses.  Constants:

  * U32 = 2^-24 per fp32 operation (no fast-math);
  * rsqrtf: 2 ulp = 4 U32 (CUDA C Programming Guide, mathematical functions appendix);
  * rcp.approx.f32 (1 ulp) and ex2.approx.f32 (2^-22.5 relative), PTX ISA: both taken as 4 U32;
  * __logf: 2^-21.41 absolute on [0.5, 2], 3 ulp elsewhere (CUDA C Programming Guide, intrinsic functions);
  * Abramowitz & Stegun 7.1.26: |erf error| <= 1.5e-7 (so 7.5e-8 on Phi = (1 + erf(u / sqrt 2)) / 2);
  * u_mma(K): the tcgen05 accumulation over K products (fp_bounds.py).

test_helpers_catch_injected_faults shows, on synthetic outputs, that the bounds catch faults the older `_rel` check
(largest error over largest reference value of the whole tensor, at 1e-2 .. 1.5e-2) lets through.
"""
import math
from importlib import import_module

import pytest
import torch
import torch.nn.functional as F

from fp_bounds import BF16, F16, U32, U_OUT, assert_within, bf16_tol, excess, out_tol, u_mma

gpu = pytest.mark.gpu
F64 = torch.float64
SQRT1_2 = 0.7071067811865476
AS_ERF = 1.5e-7                      # A&S 7.1.26
EPS_APPROX = 4 * U32                 # rcp.approx / ex2.approx (PTX ISA), rounded up to 4 U32
SUB32 = 2.0 ** -146                  # absolute floor of a few fp32 operations whose result is subnormal (2^-150 each)


def _rel_old(a, b):
    """The comparison of test_gpu_norm_stem.py / test_gpu_attention.py (kept here only to show what it misses)."""
    return float((a.float() - b.float()).abs().max() / (b.float().abs().max() + 1e-12))


def ops():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200.ops")


def cdiv(a, b):
    return -(-a // b)


# =====================================================================================================================
# bounds
# =====================================================================================================================
def ln_stats(v, depth, eps):
    """float64 mean / rstd of the rows of v (the exact fp32 values the kernel normalised) and their bounds.

    The kernel sums in fp32 along a path of `depth` additions: dmean = depth U32 sum|v| / D, plus the rounding of
    S / D (two: 1/D need not be exact).  The variance is two-pass around the computed mean: sum (v - mean')^2 =
    Q + D dmean^2 exactly, the subtraction, the square and the sum add (depth + 3) U32 of it; Q / D and + eps two more.
    rstd = rsqrtf(var + eps): relative t / 2 from var + eps (t its relative error, <= t for t <= 1/2), 4 U32 rsqrtf."""
    D = v.shape[-1]
    mu = v.mean(-1)
    d = v - mu.unsqueeze(-1)
    Q = (d * d).sum(-1)
    var = Q / D
    dmean = depth * U32 * v.abs().sum(-1) / D + 2 * U32 * mu.abs()
    dQ = D * dmean ** 2 + (depth + 3) * U32 * (Q + D * dmean ** 2)
    ve = var + eps
    t = (dQ / D + 3 * U32 * ve) / ve
    assert float(t.max()) < 0.5
    rstd = ve.rsqrt()
    return mu, rstd, dmean, rstd * (t + 4 * U32)


def ln_y_err(v, mu, rstd, dmean, drstd, g, b):
    """Bound of (v - mean') rstd' g + b in fp32 before the output rounding: the centred value is off by dmean plus
    its rounding, rstd' by drstd; * rstd, * g, + b round three times."""
    dv = (v - mu.unsqueeze(-1)).abs()
    a = g.abs() * rstd.unsqueeze(-1) * dv
    dc = dmean.unsqueeze(-1) + U32 * (dv + dmean.unsqueeze(-1))
    err = g.abs() * ((rstd + drstd).unsqueeze(-1) * dc + dv * drstd.unsqueeze(-1))
    return err + 3 * U32 * (a + b.abs())


def gelu64(u):
    """float64 erf-GELU, its derivative, 1 - Phi(|u|) and |u| phi(u) on finite u."""
    cdf = 0.5 * torch.special.erfc(-u * SQRT1_2)
    tail = 0.5 * torch.special.erfc(u.abs() * SQRT1_2)
    uphi = u * torch.exp(-0.5 * u * u) / math.sqrt(2 * math.pi)
    return u * cdf, cdf + uphi, tail, uphi.abs(), cdf


def gelu_errs(u):
    """Bounds (before the bf16 store) of gelu_parts (common.cuh) for gelu(u) and gelu'(u), float64 u.

    h = 1 - Phi(|u|) = 0.5 p(t) t e with t = rcp(1 + 0.3275911 z), z = |u| / sqrt 2, e = ex2(-u^2 log2(e) / 2):
      * the formula: |h_AS - h| <= AS_ERF / 2 (absolute);
      * its fp32 evaluation, relative rho = (64 + u^2) U32: t carries 4 U32 (z, the fma, two constants) + rcp (4 U32)
        and the polynomial's sensitivity to t is <= 1 + 2.45 (|t Q'/Q| <= 2.45 on (0, 1]); Horner in four fmas with
        fp32 coefficients, 5 U32 times sum|a_i| t^i / Q(t) <= 4.48; two products; e: u^2 is exact for bf16 u, the
        argument carries 2 U32 (u^2 U32 relative on e) + ex2 (4 U32).  3.45 x 8 + 4.48 x 5 + 2 + 4 = 56 <= 64.
    gelu = u c with c = 1 - h or h: + U32 for 1 - h, + U32 for the product.
    gelu' = fma(u * (1 / sqrt(2 pi)), e, c): the density term carries e's relative error and two more roundings.
    Where ex2.approx.ftz flushes e to 0 (its fp32 argument fl(u^2 * -0.7213475) below -126; |u| > 13.2, including
    u^2 = inf) the kernel's h is exactly 0: c is exactly 1 or 0, gelu exactly u or 0 and gelu' exactly c.  There the
    errors are exactly what is lost, h and |u| phi, and the u^2 growth of rho does not apply.  Arguments within 0.01
    of -126 keep the general bound, which is larger than h + |u| phi there."""
    val, grad, tail, uphi, cdf = gelu64(u)
    u32 = u.float()
    arg = (u32 * u32 * torch.tensor(-0.72134752044448170, dtype=torch.float32, device=u.device)).double()
    flushed = arg < -126.01
    rho = (64 + u * u) * U32
    dh = AS_ERF / 2 + rho * (tail + AS_ERF / 2)
    e_val = u.abs() * dh + 2 * U32 * val.abs() + SUB32
    e_grad = dh + U32 * cdf + uphi * (u * u + 8) * U32 + U32 * grad.abs() + SUB32
    e_val = torch.where(flushed, u.abs() * tail + SUB32, e_val)
    e_grad = torch.where(flushed, tail + uphi + SUB32, e_grad)
    return val, grad, e_val, e_grad


def test_gelu_bound_is_tight_on_every_bf16():
    """gelu_errs never allows more than the bf16 half ulp (2^-8 relative) plus 4e-6 absolute (A&S and the fp32
    evaluation: 2.05e-6 at most, near u = 0) on every finite bf16 value.  Beyond |u| = 13.3 it allows only the
    rounding of the exact u, 0 or 1, and 2^-125 absolute for gelu (the lost |u| h < 2^-126 of the flushed range): a
    bound that grew with |u| would accept any output of the large values."""
    u = _finite_bf16().double()
    val, grad, e_val, e_grad = gelu_errs(u)
    assert bool((bf16_tol(val, e_val) <= 2.0 ** -8 * val.abs() + 4e-6).all())
    assert bool((bf16_tol(grad, e_grad) <= 2.0 ** -8 * grad.abs() + 4e-6).all())
    far = u.abs() > 13.3
    assert int(far.sum()) > 30000
    assert bool((bf16_tol(val, e_val)[far] <= 2.0 ** -8 * val.abs()[far] + 2.0 ** -125).all())
    assert bool((bf16_tol(grad, e_grad)[far] <= 2.0 ** -8).all())


def attn_fwd_bounds(q, k, v, scale):
    """float64 reference and bounds of attn_fwd_kernel for one [.., T, hd] set of heads (bf16 values as float64).

    s = q k^T on tcgen05 (u_mma(128) of sum|q||k|); p = ex2((s - m) * fl(scale log2 e)): relative error eta <=
    scale (ds_j + ds_max) + 4 U32 scale |s_j - m| (subtraction, product, the two constants) + ex2's 4 U32.  P is
    stored as bf16 (2^-8) and P V accumulated by tcgen05 (u_mma(128)); the row sum is fp32 over 128 terms, its
    reciprocal __fdividef (2 ulp = 4 U32), the final scaling one more: |out' - out| <= (2 eta + 2^-8 + u_mma) sum_j
    P|v| + (128 + 6) U32 |out|.  lse = m scale + __logf(sum): the sum's log moves by eta + 128 U32, __logf by
    2^-21.41 + 6 U32 |log sum| (3 ulp), the product and the sum round once each."""
    S = q @ k.transpose(-2, -1)
    A = q.abs() @ k.abs().transpose(-2, -1)
    Ssc = S * scale
    lse = torch.logsumexp(Ssc, -1)
    P = torch.softmax(Ssc, -1)
    out = P @ v
    um = u_mma(128)
    ds = um * A
    rng = Ssc.amax(-1) - Ssc.amin(-1)
    eta = scale * 2 * ds.amax(-1) + 4 * U32 * rng + EPS_APPROX
    mag = P @ v.abs()
    e_out = (2 * eta + U_OUT[BF16] + um).unsqueeze(-1) * mag + 134 * U32 * out.abs()
    m = Ssc.amax(-1)
    logsum = lse - m
    e_lse = (scale * ds.amax(-1) + U32 * m.abs() + U32 * lse.abs() + eta + 128 * U32 + 2.0 ** -21.41
             + 6 * U32 * logsum.abs())
    return dict(S=S, A=A, Ssc=Ssc, lse=lse, P=P, out=out, e_out=e_out, e_lse=e_lse)


def attn_bwd_bounds(q, k, v, do, o_k, lse_k, f, scale):
    """float64 gradients and bounds of attn_bwd_kernel; o_k / lse_k: the forward's stored out and lse it reads.

    delta = sum o_k dO in fp32 (products exact, 128 additions); dP = dO V^T (u_mma); p = ex2(s sl2 - lse_k log2 e):
    relative scale ds + |lse_k - lse| + 3 U32 scale|s| + 2 U32 |lse_k| + U32 |arg| + 4 U32; ds = p (dp - delta)
    scale: three roundings.  P and dS are stored as bf16 (2^-8) and the three products accumulate on tcgen05 over 128
    rows (u_mma(128))."""
    um = u_mma(128)
    P, Ssc = f["P"], f["Ssc"]
    delta = (o_k * do).sum(-1)
    dP = do @ v.transpose(-2, -1)
    dS = P * (dP - delta.unsqueeze(-1)) * scale
    dV = P.transpose(-2, -1) @ do
    dK = dS.transpose(-2, -1) @ q
    dQ = dS @ k
    e_delta = 128 * U32 * (o_k.abs() * do.abs()).sum(-1)
    e_dp = um * (do.abs() @ v.abs().transpose(-2, -1))
    lk = lse_k.unsqueeze(-1)
    eta = (scale * um * f["A"] + (lse_k - f["lse"]).abs().unsqueeze(-1) + 3 * U32 * Ssc.abs() + 2 * U32 * lk.abs()
           + U32 * (lk - Ssc).abs() + EPS_APPROX)
    Pm = P * (1 + eta)
    e_ds = Pm * scale * ((dP - delta.unsqueeze(-1)).abs() * (eta + 3 * U32) + e_dp + e_delta.unsqueeze(-1))
    E_ds = e_ds + U_OUT[BF16] * (dS.abs() + e_ds)
    M_ds = dS.abs() + E_ds
    E_p = P * eta + U_OUT[BF16] * Pm
    e_dv = E_p.transpose(-2, -1) @ do.abs() + um * (Pm + E_p).transpose(-2, -1) @ do.abs()
    e_dk = E_ds.transpose(-2, -1) @ q.abs() + um * M_ds.transpose(-2, -1) @ q.abs()
    e_dq = E_ds @ k.abs() + um * M_ds @ k.abs()
    return dict(dQ=dQ, dK=dK, dV=dV, e_dq=e_dq, e_dk=e_dk, e_dv=e_dv)


def colsum_depth_bf16(M):
    """fp32 additions on the longest path of colsum_bf16 (norm.cu): a thread sums ceil(rows / 2) rows of its CTA, the
    two row lanes meet once, the gy CTAs of a column and the old value meet in atomics."""
    gy = min(cdiv(M, 256), 128)
    return cdiv(cdiv(M, gy), 2) + 1 + gy + 1


def colsum_depth_cast(M, N):
    """cast_colsum_kernel: a row lane sums ceil(rows / R) rows, the R lanes meet in shared memory, the CTAs and the
    old value in atomics (R = 256 / (N / 8), ctas = min(ceil(M / 32), 1184))."""
    R = 256 // (N // 8)
    ctas = min(cdiv(M, 32), 148 * 8)
    return cdiv(cdiv(M, ctas), R) + R + ctas + 1


# =====================================================================================================================
# A. the bounds themselves (CPU)
# =====================================================================================================================
def _attn_case(T, seed, peak):
    g = torch.Generator().manual_seed(seed)
    q, k, v = ((torch.randn(1, 1, T, 128, generator=g) * s).bfloat16().double() for s in (peak, 0.7, 0.7))
    return q, k, v


def test_helpers_catch_injected_faults():
    """Each injected fault must fail the new bound; the table records whether the old `_rel` check at its threshold
    would have caught it.  Correct outputs are the float64 references rounded once to the output format."""
    g = torch.Generator().manual_seed(0)
    faults = {}
    # one wrong LayerNorm row among 16384 (its rstd 1 % off), D = 256, rows spanning 10^-2 .. 10^2 in scale
    M, D = 16384, 256
    sd = 10.0 ** (torch.rand(M, 1, generator=g, dtype=F64) * 4 - 2)
    v = (torch.randn(M, D, generator=g, dtype=F64) * sd + sd).float().double()
    gam, bet = torch.rand(D, generator=g, dtype=F64) + 0.5, torch.randn(D, generator=g, dtype=F64) * 0.1
    mu, rstd, dmean, drstd = ln_stats(v, 2 + 7, 1e-6)
    y = (v - mu[:, None]) * rstd[:, None] * gam + bet
    tol = out_tol(y, BF16, ln_y_err(v, mu, rstd, dmean, drstd, gam, bet))
    assert float(excess(y.to(BF16), y, tol).max()) <= 1.0
    bad = y.clone()
    bad[5000] = (v[5000] - mu[5000]) * rstd[5000] * 1.01 * gam + bet
    faults["ln_row"] = (bad.to(BF16), y, tol, 1e-2)
    # a dropped odd last column of a column sum: N = 80, columns scaled 1, 1e-1, 1e-2, 1e-3
    M, N = 16384, 80
    a = (torch.randn(M, N, generator=g) * 10.0 ** -(torch.arange(N) % 4).double()).bfloat16().double()
    cs = a.sum(0)
    tol = colsum_depth_bf16(M) * U32 * a.abs().sum(0)
    assert float(excess(cs.float(), cs, tol).max()) <= 1.0
    bad = cs.clone()
    bad[N - 1] = 0.0
    faults["colsum_last_col"] = (bad.float(), cs, tol, 1e-2)
    # a GELU error confined to u < -3 (1 % there), over every finite bf16 value
    u = _finite_bf16().double()
    val, grad, e_val, e_grad = gelu_errs(u)
    tol = bf16_tol(val, e_val)
    assert float(excess(val.to(BF16), val, tol).max()) <= 1.0
    bad = torch.where(u < -3, val * 1.01, val)
    faults["gelu_tail"] = (bad.to(BF16), val, tol, 1e-2)
    # one wrong attention row at T = 125 (3 % off), peaked attention
    q, k, v = _attn_case(125, 1, 2.0)
    f = attn_fwd_bounds(q, k, v, _scale())
    ref = f["out"]
    tol = out_tol(ref, BF16, f["e_out"])
    assert float(excess(ref.to(BF16), ref, tol).max()) <= 1.0
    bad = ref.clone()
    bad[..., 60, :] *= 1.03
    faults["attn_row"] = (bad.to(BF16), ref, tol, 1.5e-2)
    old_caught = {}
    for name, (out, r, t, thr) in faults.items():
        assert float(excess(out, r, t).max()) > 1.0, name
        old_caught[name] = _rel_old(out, r) >= thr
    # recorded: the old check misses all four (each fault is small next to the largest value of its tensor)
    assert old_caught == {"ln_row": False, "colsum_last_col": False, "gelu_tail": False, "attn_row": False}, old_caught


def test_gelu_bound_covers_fp32_evaluation():
    """The fp32 evaluation of gelu_parts restated on the CPU (exact fp32 roundings of every step; exact reciprocal and
    exponential, whose approximation error the bound adds separately) stays inside gelu_errs for every finite bf16 u:
    the derivation of rho is not short of the arithmetic it describes."""
    u32 = _finite_bf16().float()
    f32 = torch.float32

    def fma(a, b, c):                       # fp32 fma: the float64 product of two fp32 values is exact
        return (a.double() * b.double() + c.double()).to(f32)

    c = lambda x: torch.tensor(x, dtype=f32)  # noqa: E731
    z = u32.abs() * c(0.70710678118654752)
    t = (1.0 / fma(c(0.3275911), z, c(1.0)).double()).to(f32)
    e = torch.exp2((u32 * u32 * c(-0.72134752044448170)).double()).to(f32)
    e = torch.where(e.abs() < 2.0 ** -126, torch.zeros_like(e), e)          # ftz of ex2.approx.ftz
    p = fma(t, c(1.061405429), c(-1.453152027))
    p = fma(p, t, c(1.421413741))
    p = fma(p, t, c(-0.284496736))
    p = fma(p, t, c(0.254829592))
    h = c(0.5) * p * t * e
    cdf = torch.where(u32 >= 0, c(1.0) - h, h)
    val32 = u32 * cdf
    grad32 = fma(u32 * c(0.3989422804014327), e, cdf)
    u = u32.double()
    val, grad, e_val, e_grad = gelu_errs(u)
    assert_within(val32, val, e_val, "gelu fp32 restatement")
    assert_within(grad32, grad, e_grad, "gelu' fp32 restatement")


def _finite_bf16():
    bits = torch.arange(-32768, 32768, dtype=torch.int32).to(torch.int16)
    u = bits.view(BF16)
    return u[torch.isfinite(u.float())]


def _scale():
    return float(torch.tensor(128 ** -0.5, dtype=torch.float32))    # the fp32 scale the kernels receive


# =====================================================================================================================
# B. row LayerNorm (row_ln_fwd / row_ln_bwd / row_ln_f32)
# =====================================================================================================================
def _ln_rows(M, D, seed, dev="cuda"):
    """Rows of scale 10^-2 .. 10^2 whose |mean| / std cycles through 0, 1, 10, 100, 1000 (a one-pass E[x^2] - E[x]^2
    variance loses everything at 1000)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    sd = 10.0 ** (torch.rand(M, 1, device=dev, generator=g) * 4 - 2)
    ratio = torch.tensor([0.0, 1.0, 10.0, 100.0, 1000.0], device=dev)[torch.arange(M, device=dev) % 5].view(M, 1)
    sign = torch.where(torch.rand(M, 1, device=dev, generator=g) < 0.5, -1.0, 1.0)
    x = torch.randn(M, D, device=dev, generator=g) * sd + sign * ratio * sd
    addend = (torch.randn(M, D, device=dev, generator=g) * sd * 0.5).bfloat16()
    gamma = torch.rand(D, device=dev, generator=g) + 0.5
    gamma[::7] = 1e-3
    beta = torch.randn(D, device=dev, generator=g) * 0.5
    return x, addend, gamma, beta


ROW_M = [1, 7, 9, 1003, 16384, 32768, 592 * 65 + 5]


@gpu
@pytest.mark.parametrize("M", ROW_M)
@pytest.mark.parametrize("D", [256, 768])
def test_row_ln_fwd_bwd_f64(D, M):
    """row_ln_fwd with and without the fused residual add, row_ln_bwd with accumulate on and off, row_ln_f32 on the
    same rows.  M = 1, 7, 9, 1003: a last CTA of fewer than 8 rows; 16384 / 32768: the v1 / windowed models at
    B = 128; 38485: above the 592-CTA cap of the backward (66 rows per CTA; the last CTAs get none)."""
    o = ops()
    eps = 1e-6
    x, addend, gamma, beta = _ln_rows(M, D, M + D)
    g64, b64 = gamma.double(), beta.double()
    V = D // 128
    for ad in (None, addend):
        y, mean, rstd, xn = o.row_ln_fwd(x, gamma, beta, eps, addend=ad)
        if ad is not None:
            assert torch.equal(xn, x + ad.float())                  # one fp32 add
        else:
            assert xn is x
        v = xn.double()
        mu, rs, dmean, drstd = ln_stats(v, V + 7, eps)             # per lane: (a + b) + (c + d), V groups; 5 shuffles
        assert_within(mean, mu, dmean, "mean")
        assert_within(rstd, rs, drstd, "rstd")
        yref = (v - mu[:, None]) * rs[:, None] * g64 + b64
        assert_within(y, yref, out_tol(yref, BF16, ln_y_err(v, mu, rs, dmean, drstd, g64, b64)), "y")
    # backward on the last forward (with addend): the reference uses the mean / rstd the kernel read
    gen = torch.Generator(device="cuda").manual_seed(M * D + 1)
    dy = torch.randn(M, D, device="cuda", generator=gen).bfloat16()
    d64 = dy.double()
    mk, rk = mean.double()[:, None], rstd.double()[:, None]
    xh = (v - mk) * rk
    gy = d64 * g64
    m1 = gy.mean(-1, keepdim=True)
    m2 = (gy * xh).mean(-1, keepdim=True)
    gref = rk * (gy - m1 - xh * m2)
    dm1 = (V + 8) * U32 * gy.abs().mean(-1, keepdim=True) + 2 * U32 * m1.abs()
    dm2 = (V + 11) * U32 * (gy * xh).abs().mean(-1, keepdim=True) + 2 * U32 * m2.abs()
    e_gx = rk * (dm1 + xh.abs() * dm2 + 4 * U32 * (gy.abs() + m1.abs() + (xh * m2).abs()))
    ctas = min(cdiv(M, 64), 592)
    depth = cdiv(cdiv(M, ctas), 8) + 8 + ctas + 1
    s_dg, s_db = (d64 * xh).sum(0), d64.sum(0)
    m_dg, m_db = (d64 * xh).abs().sum(0), d64.abs().sum(0)
    dg0, db0 = torch.randn(D, device="cuda", generator=gen), torch.randn(D, device="cuda", generator=gen)
    for acc in (False, True):
        g0 = torch.randn(M, D, device="cuda", generator=gen) if acc else torch.full((M, D), math.nan, device="cuda")
        gx = g0.clone()
        dg, db = dg0.clone(), db0.clone()
        o.row_ln_bwd(dy, xn, mean, rstd, gamma, gx, acc, dg, db)
        ref = gref + (g0.double() if acc else 0.0)
        assert_within(gx, ref, e_gx + U32 * ref.abs() + (U32 * g0.double().abs() if acc else 0.0), "gx acc=%d" % acc)
        assert_within(dg, dg0.double() + s_dg, (depth + 3) * U32 * (m_dg + dg0.double().abs()), "dgamma")
        assert_within(db, db0.double() + s_db, depth * U32 * (m_db + db0.double().abs()), "dbeta")
    # fp32 twin (exact.cu): fp32 addend, sequential lane sums of D / 32 terms; its planes sum back to the fp32 value
    planes, xn32 = o.row_ln_f32(x, gamma, beta, eps, addend.float())
    assert torch.equal(xn32, xn)
    mu, rs, dmean, drstd = ln_stats(v, cdiv(D, 32) + 5, eps)
    drstd = drstd + rs * 2 * U32                                    # 1 / sqrtf(): two IEEE roundings, not rsqrtf
    yref = (v - mu[:, None]) * rs[:, None] * g64 + b64
    err = ln_y_err(v, mu, rs, dmean, drstd, g64, b64)
    assert_within(planes.double().sum(0), yref, err + U32 * yref.abs(), "row_ln_f32")


# =====================================================================================================================
# C. whole-sample LayerNorm (sample_ln_fwd / sample_ln_bwd)
# =====================================================================================================================
def _sample_ln_check(o, x, fmt, eps=1e-5):
    B = x.shape[0]
    y, mean, rstd = o.sample_ln_fwd(x, fmt, eps)
    v = x.double().reshape(B, -1)
    N = v.shape[1]
    mu, rs, dmean, drstd = ln_stats(v, cdiv(N, 4096) + 12, eps)   # per thread ceil(N / 4096) float4 groups; 2 x 5
    assert_within(mean, mu, dmean, "mean")
    assert_within(rstd, rs, drstd, "rstd")
    one, zero = torch.ones_like(v[0]), torch.zeros_like(v[0])
    yref = (v - mu[:, None]) * rs[:, None]
    err = ln_y_err(v, mu, rs, dmean, drstd, one, zero)
    tol = out_tol(yref, fmt, err) if fmt != torch.float32 else err
    assert y.dtype == fmt
    assert_within(y.reshape(B, -1), yref, tol, "y %s" % fmt)
    return y, rstd


@gpu
@pytest.mark.parametrize("W", [128, 512, 600, 1000, 1024])
@pytest.mark.parametrize("fmt", [torch.float32, BF16])
def test_sample_ln_image_f64(W, fmt):
    """The input image's LayerNorm over 64 x W: three ordinary samples and one with |mean| / std = 1000."""
    o = ops()
    torch.manual_seed(W)
    x = torch.rand(4, 64, W, device="cuda") * 3 + 1
    x[3] = 100.0 + 0.1 * torch.randn(64, W, device="cuda")
    _sample_ln_check(o, x, fmt)


@gpu
@pytest.mark.parametrize("C", [80, 81, 228])
@pytest.mark.parametrize("T", [32, 100, 128])
def test_sample_ln_logits_f64(T, C):
    """The logits slab's LayerNorm (fp32 out) and its backward into the head's padded bf16 layout (ld = C rounded up
    to 8): dx per element against float64 from the y / rstd the kernel read, the pad columns exactly 0."""
    o = ops()
    torch.manual_seed(T * 1000 + C)
    B = 3
    x = torch.randn(B, T, C, device="cuda") * 3
    x[1] += 500.0
    y, rstd = _sample_ln_check(o, x, torch.float32)
    C8 = cdiv(C, 8) * 8
    dy = torch.randn(B, T, C, device="cuda")
    dx = o.sample_ln_bwd(dy, y, rstd, C, C8)
    assert dx.shape == (B * T, C8) and dx.dtype == BF16
    N = T * C
    g, yy, r = dy.double().reshape(B, N), y.double().reshape(B, N), rstd.double()[:, None]
    m1, m2 = g.mean(-1, keepdim=True), (g * yy).mean(-1, keepdim=True)
    ref = r * (g - m1 - yy * m2)
    depth = cdiv(N, 1024) + 10                                       # per thread ceil(N / 1024) terms; block_sum
    dm1 = (depth + 1) * U32 * g.abs().mean(-1, keepdim=True)
    dm2 = (depth + 2) * U32 * (g * yy).abs().mean(-1, keepdim=True)
    err = r * (dm1 + yy.abs() * dm2 + 3 * U32 * (g.abs() + m1.abs() + (yy * m2).abs())) + U32 * ref.abs()
    dxv = dx.view(B, T, C8)
    assert_within(dxv[:, :, :C].reshape(B, N), ref, out_tol(ref, BF16, err), "dx")
    assert torch.equal(dxv[:, :, C:], torch.zeros_like(dxv[:, :, C:]))


@gpu
def test_sample_ln_refuses_n_not_multiple_of_4():
    o = ops()
    err = import_module("htr-vt_b200._lib").HtrvtError
    with pytest.raises(err):
        o.sample_ln_fwd(torch.randn(2, 7, 81, device="cuda"), torch.float32)


# =====================================================================================================================
# D. tokens (tokens_fwd / tokens_bwd / tokens_f32)
# =====================================================================================================================
@gpu
@pytest.mark.parametrize("fmt", [F16, BF16])
@pytest.mark.parametrize("B", [1, 3, 128])
@pytest.mark.parametrize("T", [1, 7, 128, 250, 256])
def test_tokens_f64(T, B, fmt):
    """x = (m ? tok : mask_token) + pos is one fp32 add for m in {0, 1}: bit exact, as are dtok = bf16(gx m) and the
    fp32 twin.  dmask_token += sum over b, t of gx (1 - m): B additions per token, the finalise's ceil(T / 8) + 8 and
    the old value."""
    o = ops()
    D = 768
    torch.manual_seed(T * 10 + B)
    tok = torch.randn(B, T, D, device="cuda").to(fmt)
    mt = torch.randn(D, device="cuda")
    pos = torch.randn(T, D, device="cuda")
    masks = {"none": None, "zeros": torch.zeros(T, device="cuda"), "ones": torch.ones(T, device="cuda"),
             "random": (torch.rand(T, device="cuda") > 0.4).float()}
    gx = torch.randn(B * T, D, device="cuda")
    for name, mask in masks.items():
        m = (mask if mask is not None else torch.ones(T, device="cuda")).view(1, T, 1)
        for p in (None, pos):
            base = torch.where(m > 0, tok.float(), mt)
            ref = base + p if p is not None else base
            x = o.tokens_fwd(tok, mask, mt, p, B, T, D)
            assert torch.equal(x.view(B, T, D), ref), (name, p is None)
            x32 = o.tokens_f32(tok.float().contiguous(), mask, mt, p, B, T, D)
            assert torch.equal(x32.view(B, T, D), ref), (name, p is None)
        dmt0 = torch.randn(D, device="cuda")
        dmt = dmt0.clone()
        dtok = o.tokens_bwd(gx, mask, dmt, B, T, D)
        assert torch.equal(dtok, (gx.view(B, T, D) * m).bfloat16()), name
        if mask is None:
            assert torch.equal(dmt, dmt0)
            continue
        terms = gx.double().view(B, T, D) * (1 - m.double())
        ref = dmt0.double() + terms.sum((0, 1))
        depth = B + cdiv(T, 8) + 8 + 1
        assert_within(dmt, ref, depth * U32 * (terms.abs().sum((0, 1)) + dmt0.double().abs()), "dmask_token " + name)


# =====================================================================================================================
# E. GELU, exhaustively over every finite bf16 value
# =====================================================================================================================
def _gelu_inputs():
    """Every finite bf16 value (65280) padded with zeros to 65536 = 256 x 256, on the GPU."""
    u = _finite_bf16()
    return torch.cat([u, torch.zeros(65536 - u.numel(), dtype=BF16)]).cuda()


@gpu
def test_gelu_kernels_every_bf16():
    """gelu_fwd / gelu_bwd (da = 1 and random da) against float64 erf-GELU and GELU' (bound: gelu_errs + the bf16
    store's half ulp), and +-inf / NaN as F.gelu and its autograd in fp32 on the same device."""
    o = ops()
    u = _gelu_inputs()
    u64 = u.double()
    val, grad, e_val, e_grad = gelu_errs(u64)
    a = o.gelu_fwd(u)
    assert_within(a, val, bf16_tol(val, e_val), "gelu_fwd")
    torch.manual_seed(3)
    for name, da in (("da=1", torch.ones_like(u)), ("da random", torch.randn(u.shape, device="cuda").bfloat16())):
        d64 = da.double()
        ref = d64 * grad
        err = d64.abs() * e_grad + U32 * ref.abs()
        assert_within(o.gelu_bwd(da, u), ref, bf16_tol(ref, err), "gelu_bwd " + name)
    sp = torch.tensor([math.inf, -math.inf, math.nan, -math.nan, 0.0, -0.0, 1.0, -1.0], device="cuda").bfloat16()
    uf = sp.float().requires_grad_(True)
    want = F.gelu(uf)
    want.backward(torch.ones_like(uf))
    got_a, got_d = o.gelu_fwd(sp).float(), o.gelu_bwd(torch.ones_like(sp), sp).float()
    for got, ref in ((got_a, want.detach().bfloat16().float()), (got_d, uf.grad.bfloat16().float())):
        assert torch.equal(torch.isnan(got), torch.isnan(ref)), (got, ref)
        fin = ~torch.isnan(ref)
        assert torch.equal(got[fin], ref[fin]), (got, ref)


@gpu
def test_gelu_gemm_epilogues_every_bf16():
    """The tap-GEMM's GELU epilogues on every finite bf16 value: x = [256, 256] of the values, w = I, zero bias, so the
    accumulator holds each value exactly (checked first, fp32 out).  Eval gelu; train gelu + the saved gelu'; fc2's
    input-gradient epilogue du = dy * gelu' (a bf16 x bf16 product is exact in fp32: rounded once, bit exact) with
    fc1's bias gradient from the epilogue's column sums (gemm.cu flush_stats)."""
    o = ops()
    x = _gelu_inputs().view(256, 256)
    eye = torch.eye(256, device="cuda").bfloat16()
    zero = torch.zeros(256, device="cuda")
    acc = torch.empty(256, 256, device="cuda")
    o.gemm_tn(x, eye, acc)
    assert torch.equal(acc, x.float())
    u64 = x.double()
    val, grad, e_val, e_grad = gelu_errs(u64)
    a1 = torch.full((256, 256), 7.0, device="cuda", dtype=BF16)
    o.gemm_tn(x, eye, a1, bias=zero, gelu=True)
    assert_within(a1, val, bf16_tol(val, e_val), "gemm_tn gelu (eval)")
    a2 = torch.full_like(a1, 7.0)
    pre = torch.full_like(a1, 7.0)
    o.gemm_tn(x, eye, a2, bias=zero, gelu=True, pre=pre)
    assert_within(a2, val, bf16_tol(val, e_val), "gemm_tn gelu (train)")
    assert_within(pre, grad, bf16_tol(grad, e_grad), "gemm_tn gelu' (train)")
    torch.manual_seed(4)
    dy = torch.randn(256, 256, device="cuda").bfloat16()
    du = torch.full_like(a1, 7.0)
    cs0 = torch.randn(256, device="cuda")
    cs = cs0.clone()
    o.gemm_nn(dy, eye, du, gelu_u=pre, colsum=cs)
    assert torch.equal(du, (dy.float() * pre.float()).bfloat16())
    d = du.double()
    # fc1's bias gradient: a warp sums its 32 rows of a tile (32 additions), adds that into its running sum once per
    # 128-row tile it owns (<= M / 128 = 2), and each of the 4 TMEM-quadrant warps flushes one atomic per column per
    # CTA: at most M / 32 = 8 atomics into one column, which also hold the old value
    depth = 32 + 256 // 128 + 256 // 32
    assert_within(cs, cs0.double() + d.sum(0), depth * U32 * (d.abs().sum(0) + cs0.double().abs()), "colsum")


@gpu
def test_mul_bf16_bit_exact():
    """mul_bf16 on 16 M random bit patterns (every class: subnormals, inf, NaN, zeros of both signs) plus specials:
    bit exact to torch's fp32 product rounded once; NaN where torch gives NaN."""
    o = ops()
    torch.manual_seed(5)
    n = 1 << 24
    a = torch.randint(-32768, 32768, (n,), device="cuda", dtype=torch.int32).to(torch.int16).view(BF16)
    b = torch.randint(-32768, 32768, (n,), device="cuda", dtype=torch.int32).to(torch.int16).view(BF16)
    sp = torch.tensor([math.inf, 0.0, -0.0, 3e38, 1e-38, -1e-40, math.nan, 1.0], device="cuda").bfloat16()
    sq = torch.tensor([0.0, math.inf, 5.0, 3e38, 1e-38, 1e-2, 2.0, -math.inf], device="cuda").bfloat16()
    a, b = torch.cat([a, sp]), torch.cat([b, sq])
    out = o.mul_bf16(a, b)
    ref = (a.float() * b.float()).bfloat16()
    nan = torch.isnan(ref)
    assert torch.equal(torch.isnan(out), nan)
    assert torch.equal(out.view(torch.int16)[~nan], ref.view(torch.int16)[~nan])


# =====================================================================================================================
# F. column sums (colsum_bf16 / cast_colsum_bf16)
# =====================================================================================================================
@gpu
@pytest.mark.parametrize("M", [1, 255, 257, 16384, 32768])
@pytest.mark.parametrize("N,ld", [(3, 8), (80, 80), (771, 776), (768, 768), (3072, 3072)])
def test_colsum_bf16_f64(N, ld, M):
    """Column sums of a bf16 [M, N] view with row stride ld (pad columns hold NaN: none may leak in), columns at four
    magnitudes, accumulate on and off, per column against the float64 sum."""
    o = ops()
    torch.manual_seed(M + N)
    buf = torch.full((M, ld), math.nan, device="cuda").bfloat16()
    scale = 10.0 ** -(torch.arange(N, device="cuda") % 4).float()
    buf[:, :N] = (torch.randn(M, N, device="cuda") * scale).bfloat16()
    a = buf[:, :N]
    a64 = a.double()
    depth = colsum_depth_bf16(M)
    for acc in (False, True):
        out0 = torch.randn(N, device="cuda")
        out = out0.clone()
        o.colsum_bf16(a, out, accumulate=acc)
        base = out0.double() if acc else torch.zeros_like(a64[0])
        assert_within(out, base + a64.sum(0), depth * U32 * (a64.abs().sum(0) + base.abs()), "colsum acc=%d" % acc)


@gpu
@pytest.mark.parametrize("M", [1, 31, 33, 16384, 32775])
@pytest.mark.parametrize("N", [8, 88, 768, 776, 2048])
def test_cast_colsum_f64(N, M):
    """dst = bf16(src) bit exact; colsum += the column sums of the ROUNDED values, per column against float64."""
    o = ops()
    torch.manual_seed(M * 7 + N)
    src = torch.randn(M, N, device="cuda") * 10.0 ** -(torch.arange(N, device="cuda") % 4).float()
    cs0 = torch.randn(N, device="cuda")
    cs = cs0.clone()
    dst = o.cast_colsum_bf16(src, cs)
    assert torch.equal(dst.view(torch.int16), src.bfloat16().view(torch.int16))
    d = dst.double()
    depth = colsum_depth_cast(M, N)
    assert_within(cs, cs0.double() + d.sum(0), depth * U32 * (d.abs().sum(0) + cs0.double().abs()), "colsum")


@gpu
def test_cast_colsum_refuses_wide_rows():
    o = ops()
    err = import_module("htr-vt_b200._lib").HtrvtError
    with pytest.raises(err):
        o.cast_colsum_bf16(torch.randn(4, 2056, device="cuda"), torch.zeros(2056, device="cuda"))


# =====================================================================================================================
# G. v1 attention (attention_fwd / attention_bwd / attention_f32)
# =====================================================================================================================
ATTN_T = [1, 2, 7, 17, 31, 33, 64, 100, 125, 127, 128]
H, HD = 6, 128


def _attn_inputs(B, T, kind, gen):
    """qkv fp32 [B, T, 3, H, hd]: 'random'; 'saturated' (key T // 2 beats every other by ~22 in scaled score);
    'flat' (all keys equal: every score of a row the same); 'last' (the maximum on key T - 1, margin ~5.7)."""
    qkv = torch.randn(B, T, 3, H, HD, device="cuda", generator=gen) * 0.7
    if kind in ("saturated", "last"):
        j = T // 2 if kind == "saturated" else T - 1
        qkv[:, :, 0] = 1.0 + 0.1 * qkv[:, :, 0]
        qkv[:, :, 1] *= 0.15
        qkv[:, j, 1] = 2.0 if kind == "saturated" else 0.5
    elif kind == "flat":
        qkv[:, :, 1] = qkv[:, :1, 1]
    return qkv


def _heads(t, i):
    return t[:, :, i].permute(0, 2, 1, 3).double()                      # [B, H, T, hd]


@gpu
@pytest.mark.parametrize("B,T", [(b, t) for t in ATTN_T for b in (1, 3)] + [(128, 128)])
def test_attention_v1_f64(B, T):
    """attn_fwd / attn_bwd per element against float64 softmax(Q K^T scale) V and its gradients on the bf16 q, k, v:
    lse per row, out, dq / dk / dv.  Outputs go into views of larger buffers whose trailing rows hold a sentinel:
    nothing may be written past row T of the last sample.  Four input kinds per shape (_attn_inputs)."""
    o = ops()
    scale = _scale()
    gen = torch.Generator(device="cuda").manual_seed(B * 1000 + T)
    kinds = ["random", "saturated", "flat", "last"] if B < 128 else ["random", "saturated"]
    for kind in kinds:
        qkv = _attn_inputs(B, T, kind, gen).bfloat16()
        q, k, v = _heads(qkv, 0), _heads(qkv, 1), _heads(qkv, 2)
        f = attn_fwd_bounds(q, k, v, scale)
        sent = 12345.0
        obuf = torch.full((B * T + 5, H * HD), sent, device="cuda").bfloat16()
        lbuf = torch.full((B * H * T + 5,), sent, device="cuda")
        out = obuf[:B * T].view(B, T, H * HD)
        lse = lbuf[:B * H * T].view(B, H, T)
        o.attention_fwd(qkv, out, lse, scale)
        assert torch.all(obuf[B * T:].float() == float(torch.tensor(sent).bfloat16())), kind
        assert torch.all(lbuf[B * H * T:] == sent), kind
        assert_within(lse, f["lse"], f["e_lse"], "lse " + kind)
        o_k = out.view(B, T, H, HD).permute(0, 2, 1, 3)
        assert_within(o_k, f["out"], out_tol(f["out"], BF16, f["e_out"]), "out " + kind)
        dout = torch.randn(B, T, H * HD, device="cuda", generator=gen).bfloat16()
        do = dout.view(B, T, H, HD).permute(0, 2, 1, 3).double()
        r = attn_bwd_bounds(q, k, v, do, o_k.double(), lse.double(), f, scale)
        gbuf = torch.full((B * T + 3, 3, H, HD), sent, device="cuda").bfloat16()
        dqkv = gbuf[:B * T].view(B, T, 3, H, HD)
        o.attention_bwd(qkv, out, dout, lse, dqkv, scale)
        assert torch.all(gbuf[B * T:].float() == float(torch.tensor(sent).bfloat16())), kind
        for i, (name, ekey) in enumerate((("dQ", "e_dq"), ("dK", "e_dk"), ("dV", "e_dv"))):
            got = _heads(dqkv, i)
            assert_within(got, r[name], out_tol(r[name], BF16, r[ekey]), "%s %s" % (name, kind))


@gpu
@pytest.mark.parametrize("T", ATTN_T)
def test_attention_f32_f64(T):
    """attention_f32 (exact.cu) at the ragged T: within 2e-6 of sum_j P |v| per element (the tolerance its existing
    check applies to the largest output), against float64."""
    o = ops()
    B = 3
    gen = torch.Generator(device="cuda").manual_seed(T)
    scale = 128 ** -0.5
    for kind in ("random", "saturated", "flat", "last"):
        qkv = _attn_inputs(B, T, kind, gen)
        out = o.attention_f32(qkv, B, H, T, HD, scale).view(B, T, H, HD).permute(0, 2, 1, 3)
        q, k, v = _heads(qkv, 0), _heads(qkv, 1), _heads(qkv, 2)
        s32 = float(torch.tensor(scale, dtype=torch.float32))
        P = torch.softmax((q @ k.transpose(-2, -1)) * s32, -1)
        assert_within(out, P @ v, 2e-6 * (P @ v.abs()), "attention_f32 " + kind)
