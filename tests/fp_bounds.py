"""Constants and comparisons shared by the float64-reference tests (test_gpu_stem_bn.py, test_gpu_transformer_f64.py).

A kernel output is compared element by element (or per row / column for statistics) with a float64 reference computed
from the exact operands the kernel read, against a bound built from the formats:

    |out - ref| <= u_out * |ref| + eta_out + (1 + u_out) * err

where `err` bounds the kernel's arithmetic before the final rounding into the output format.
"""
import math

import torch

F16, BF16 = torch.float16, torch.bfloat16

# unit roundoff of round-to-nearest into the 16-bit output format (half an ulp, relative): 11 / 8 significand bits
U_OUT = {F16: 2.0 ** -11, BF16: 2.0 ** -8}
# absolute floor of that rounding: half the smallest subnormal (fp16 2^-24, bf16 2^-133)
ETA_OUT = {F16: 2.0 ** -25, BF16: 2.0 ** -134}
# fp32 unit roundoff: one IEEE round-to-nearest fp32 operation (the build uses no fast-math)
U32 = 2.0 ** -24


def u_mma(K):
    """Accumulation bound of the tcgen05 tap-GEMM over K products, relative to sum |x||w|: the products of 16-bit
    operands are exact in fp32; each kind::f16 MMA step sums k = 16 of them (alignment may truncate: one fp32 ulp,
    2^-23, per addition, <= 16 additions) and adds the block into the fp32 accumulator once (K / 16 steps)."""
    return (K // 16 + 16) * 2.0 ** -23


def out_tol(ref, fmt, err):
    """Per-element bound of a 16-bit store of a value that is within `err` of `ref` before rounding."""
    return U_OUT[fmt] * ref.abs() + ETA_OUT[fmt] + (1 + U_OUT[fmt]) * err


def half_ulp_bf16(x):
    """Half the spacing of bf16 at |x| (float64): 2^(e - 8) for |x| in [2^e, 2^(e + 1)), 2^-134 in the subnormal range.
    Round-to-nearest into bf16 moves x by at most this much; out_tol's 2^-8 |x| is up to twice as wide."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - 8)


def bf16_tol(ref, err):
    """Tight per-element bound of a bf16 store of a value within `err` of `ref`: the rounded value is within half an
    ulp of the unrounded one, whose magnitude is at most |ref| + err."""
    return half_ulp_bf16(ref.abs() + err) + err


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
