"""GPU checks of the windowed variant's train-mode regularisers against the oracle's restatement of their masks
(htrvt_oracle.dropout_keep_scale / attention_keep): the dropout kernel bit for bit, the attention kernels' forward
and backward dropout masks pair by pair, and the argument refusals of both entries."""
import ctypes
from importlib import import_module

import numpy as np
import pytest
import torch

import htrvt_oracle as O

pytestmark = pytest.mark.gpu
ERR_SHAPE = -1


def ops():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200.ops")


def _lib():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200._lib").lib()


def _status(fn, *args):
    return int(fn(*args, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))


# ------------------------------------------------------------------------------------------------
# 1. dropout / DropPath kernel (htrvt_dropout_bf16)
# ------------------------------------------------------------------------------------------------
SEEDS = [0x0000_0000_1234_5678, 0x2F00_1D3C_0000_0000 + 0x9ABC]     # high word zero / non-zero
N_BIG = 5 * 1_000_008            # > 148 * 16 CTAs x 256 threads x 8 elements: the grid-stride loop runs twice


@pytest.mark.parametrize("p", [0.05, 0.1, 0.5])
@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("dp_kind", ["none", "with_zero", "scales"])
def test_dropout_is_bit_exact_against_the_host_mask(p, seed, dp_kind):
    o = ops()
    B = 5
    per = N_BIG // B
    g = torch.Generator(device="cuda").manual_seed(int(seed) & 0xFFFF)
    x = torch.randn(N_BIG, device="cuda", generator=g).bfloat16()
    dp = {"none": None, "with_zero": np.array([1.25, 0.0, 1.25, 0.0, 1.25], np.float32),
          "scales": np.array([1.0, 2.0, 1.0 / 0.9, 1.5, 0.75], np.float32)}[dp_kind]
    for site in (1, 8 * 2 + 2, 8 * 11 + 3):
        y = x.clone()
        o.dropout_(y, per, p, seed, site, None if dp is None else torch.from_numpy(dp).cuda())
        sc = torch.from_numpy(O.dropout_keep_scale(N_BIG, per, p, seed, site, dp)).cuda()
        want = (x.float() * sc).bfloat16()
        assert torch.equal(y, want), (site, int((y != want).sum()))
        if dp is not None:                                          # a zero DropPath scale clears the whole sample
            for b in np.flatnonzero(dp == 0):
                assert not y[b * per:(b + 1) * per].any()


def _ones_dropped(o, n, p, seed, site):
    x = torch.ones(n, device="cuda", dtype=torch.bfloat16)
    o.dropout_(x, n, p, seed, site)
    return x


def _within_4_sigma(frac, q, n):
    return abs(frac - q) <= 4.0 * (q * (1 - q) / n) ** 0.5


@pytest.mark.parametrize("p", [0.05, 0.1, 0.5])
def test_dropout_keep_rate_scale_and_independence(p):
    o = ops()
    n = 1 << 24
    seed = SEEDS[1]
    a = _ones_dropped(o, n, p, seed, 3)
    ka = a != 0
    assert _within_4_sigma(float(ka.float().mean()), 1 - p, n)
    inv = torch.tensor(np.float32(1.0) / (np.float32(1.0) - np.float32(p))).bfloat16()      # the kernel's 1 / (1 - p)
    assert torch.equal(a[ka], inv.cuda().expand(int(ka.sum())))
    q = (1 - p) ** 2
    for other in (_ones_dropped(o, n, p, seed, 4),                   # another site
                  _ones_dropped(o, n, p, seed + 1, 3),               # another low seed word
                  _ones_dropped(o, n, p, seed + (1 << 32), 3)):      # another high seed word only
        both = float((ka & (other != 0)).float().mean())
        assert _within_4_sigma(both, q, n), (both, q)


def test_dropout_refusals_leave_the_buffer_untouched():
    L, o = _lib(), ops()
    x = torch.randn(4096, device="cuda").bfloat16()
    ref = x.clone()
    dp = torch.ones(2, device="cuda")
    for p in (float("nan"), -0.1, -1e-7, 1.0, 1.5, float("inf")):
        assert _status(L.htrvt_dropout_bf16, o._p(x), 4096, 2048, p, 7, 1, o._p(dp)) == ERR_SHAPE, p
        with pytest.raises(o.HtrvtError):
            o.dropout_(x, 2048, p, 7, 1, dp)
    torch.cuda.synchronize()
    assert torch.equal(x, ref)
    assert _status(L.htrvt_dropout_bf16, o._p(x), 4096, 2048, 0.0, 7, 1, o._p(dp)) == 0


# ------------------------------------------------------------------------------------------------
# 2. attention dropout masks (htrvt_attention2_fwd / _bwd), exact, pair by pair
# ------------------------------------------------------------------------------------------------
# the shape list of test_gpu_attention.py::test_attention2_fwd_bwd
SHAPES = [
    (2, 6, 256, 256, 0, 0, True), (2, 6, 256, 256, 16, 0, True), (2, 6, 256, 256, 16, 8, True),
    (3, 2, 128, 128, 16, 8, True), (2, 3, 128, 128, 0, 0, True), (2, 2, 208, 256, 0, 0, True),
    (2, 2, 48, 64, 16, 0, True), (2, 2, 256, 0, 0, 0, False), (2, 6, 250, 250, 16, 0, True),
    (2, 6, 250, 250, 16, 8, True), (2, 2, 150, 150, 16, 8, True), (2, 2, 202, 256, 16, 8, True),
    (3, 2, 90, 128, 16, 8, True), (2, 2, 90, 128, 16, 0, True), (2, 2, 200, 200, 16, 8, True),
    (1, 2, 7, 16, 16, 8, True), (2, 2, 250, 250, 0, 0, True),
]


def _pairs(T, window, shift):
    """[T, T] bool: (query token i, key token j) attend to each other (same rolled window, or global)."""
    if window == 0:
        return torch.ones(T, T, dtype=torch.bool)
    Tp = -(-T // window) * window
    w = ((torch.arange(T) - shift) % Tp) // window
    return w[:, None] == w[None, :]


@pytest.mark.parametrize("p", [0.05, 0.5])
@pytest.mark.parametrize("seed", [0x0000_0000_0BAD_F00D, 0x7123_4567_89AB_CDEF])
@pytest.mark.parametrize("B,H,T,prel,window,shift,bias", SHAPES)
def test_attention_dropout_masks_are_exact(B, H, T, prel, window, shift, bias, seed, p):
    o = ops()
    hd = 128
    torch.manual_seed(3)
    qkv = (torch.randn(B, T, 3, H, hd, device="cuda") * 0.3).bfloat16()
    table = (torch.randn(2 * prel - 1, H, device="cuda") * 0.5) if bias else None
    scale = hd ** -0.5
    bh = np.arange(B * H).reshape(B, H, 1, 1)
    t = np.arange(T)
    want = torch.from_numpy(O.attention_keep(seed, bh, t.reshape(1, 1, T, 1), t.reshape(1, 1, 1, T), p))
    pairs = _pairs(T, window, shift)                       # [query, key]
    assert want[:, :, pairs].any() and not want[:, :, pairs].all()
    lse = torch.empty(B, H, T, device="cuda")
    for b0 in range(0, T, 128):
        n = min(128, T - b0)
        c = torch.arange(n, device="cuda")
        # forward: V one-hot over keys [b0, b0 + n): out[b, i, h, c] = P~[i, b0 + c], zero exactly where dropped
        probe = qkv.clone()
        probe[:, :, 2] = 0
        probe[:, b0 + c, 2, :, c] = 1
        out = torch.empty(B, T, H * hd, device="cuda", dtype=torch.bfloat16)
        o.attention2_fwd(probe, out, lse, scale, table, prel, window, shift, p, seed)
        got = (out.view(B, T, H, hd)[..., :n] != 0).permute(0, 2, 1, 3).cpu()      # [B, H, query, c]
        valid = pairs[:, b0:b0 + n]
        assert torch.equal(got[:, :, valid], want[:, :, :, b0:b0 + n][:, :, valid]), ("fwd", b0)
        assert not got[:, :, ~valid].any()
        # backward: dO one-hot over queries [b0, b0 + n): dV[b, j, h, c] = P~[b0 + c, j], zero exactly where dropped
        dout = torch.zeros(B, T, H, hd, device="cuda", dtype=torch.bfloat16)
        dout[:, b0 + c, :, c] = 1
        dqkv = torch.zeros(B, T, 3, H, hd, device="cuda", dtype=torch.bfloat16)
        o.attention2_bwd(probe, out, dout.view(B, T, H * hd), lse, dqkv, scale, table, prel, window, shift, None, p,
                         seed)
        got = (dqkv[:, :, 2, :, :n] != 0).permute(0, 2, 1, 3).cpu()                  # [B, H, key, c]
        valid = pairs[b0:b0 + n, :].t()                                              # [key, c]
        want_b = want[:, :, b0:b0 + n, :].transpose(2, 3)
        assert torch.equal(got[:, :, valid], want_b[:, :, valid]), ("bwd", b0)
        assert not got[:, :, ~valid].any()


@pytest.mark.parametrize("entry", ["fwd", "bwd"])
def test_attention_dropout_refusals_leave_the_buffers_untouched(entry):
    L, o = _lib(), ops()
    B, H, T, hd, prel = 2, 2, 64, 128, 64
    qkv = torch.randn(B, T, 3, H, hd, device="cuda").bfloat16()
    table = torch.randn(2 * prel - 1, H, device="cuda")
    out = torch.randn(B, T, H * hd, device="cuda").bfloat16()
    lse = torch.randn(B, H, T, device="cuda")
    dout = torch.randn(B, T, H * hd, device="cuda").bfloat16()
    dqkv = torch.randn(B, T, 3, H, hd, device="cuda").bfloat16()
    dtable = torch.randn_like(table)
    before = [t.clone() for t in (out, lse, dqkv, dtable)]
    p = o._p
    for window, shift in ((0, 0), (16, 8)):
        for drop in (float("nan"), -0.05, -1e-9, 1.0, 2.0, float("-inf")):
            if entry == "fwd":
                s = _status(L.htrvt_attention2_fwd, p(qkv), B, H, T, hd, 0.1, p(table), prel, window, shift, drop, 5,
                            p(out), p(lse))
            else:
                s = _status(L.htrvt_attention2_bwd, p(qkv), p(out), p(dout), p(lse), B, H, T, hd, 0.1, p(table), prel,
                            window, shift, drop, 5, p(dqkv), p(dtable), p(None), 0)
            assert s == ERR_SHAPE, (window, drop, s)
    torch.cuda.synchronize()
    for a, b in zip((out, lse, dqkv, dtable), before):
        assert torch.equal(a, b)
    # the fp32 entry (no dropout) shares the shape check and is unaffected
    q32 = torch.randn(B, T, 3, H, hd, device="cuda")
    o32 = torch.empty(B, T, H * hd, device="cuda")
    assert _status(L.htrvt_attention2_f32, p(q32), B, H, T, hd, 0.1, p(table), prel, 16, 8, p(o32)) == 0
