"""Host checks of the windowed variant's train-mode regularisers: the oracle's restatement of the kernels' dropout and
attention-dropout masks (htrvt_oracle.dropout_keep_scale / attention_keep), the oracle's `regs` injection, and the
argument checks of model_window's set_stochastic / _train_rng.  No GPU needed."""
from functools import partial
from importlib import import_module

import numpy as np
import pytest
import torch

import htrvt_oracle as O


# ------------------------------------------------------------------------------------------------
# mask restatements: a plain-Python transliteration of the kernels' integer code vs the vectorised numpy version
# ------------------------------------------------------------------------------------------------
M32 = 0xFFFFFFFF


def _mix(x):
    x &= M32
    x ^= x >> 16
    x = (x * 0x85EBCA6B) & M32
    x ^= x >> 13
    x = (x * 0xC2B2AE35) & M32
    return x ^ (x >> 16)


def _scalar_dropout_factor(e, per_sample, p, seed, site, dp):
    """dropout_bf16_kernel (csrc/norm.cu) for one element, line by line, in Python integers."""
    p32 = np.float32(p)
    thr = int(p32 * np.float32(16777216.0))
    inv_keep = np.float32(1.0) / (np.float32(1.0) - p32)
    key = _mix((seed & M32) ^ ((site * 0x9E3779B9) & M32)) ^ ((seed >> 32) & M32)
    i, k = e // 8, (e // 2) % 4
    r = _mix(key + ((i & M32) * 4 & M32) + k) ^ ((i >> 30) & M32)
    half = (r & 0xFFFF) if e % 2 == 0 else (r >> 16)
    sc = inv_keep * (np.float32(dp[e // per_sample]) if dp is not None else np.float32(1.0))
    return np.float32(0.0) if (half << 8) < thr else np.float32(sc)


def _scalar_attention_keep(seed, bh, ti, tj, p):
    """attn_keep (csrc/attention2.cu) for one pair, in Python integers."""
    a = _mix((seed & M32) ^ ((bh * 0x9E3779B9) & M32))
    v = _mix(a ^ _mix(((seed >> 32) + ti * 65537 + tj) & M32))
    return not (np.float32(v >> 8) * np.float32(1.0 / 16777216.0) < np.float32(p))


@pytest.mark.parametrize("seed", [0x1234, 0x5EED_0001_9ABC_DEF0, 2 ** 62 - 1])
@pytest.mark.parametrize("offset", [0, 3 << 33])                  # 3 << 33: the (i >> 30) term is non-zero
def test_dropout_keep_scale_matches_the_kernel_arithmetic(seed, offset):
    rs = np.random.RandomState(seed & 0xFFFF)
    n, per_sample = 4096, 1024
    dp = np.array([0.0, 1.25, 2.0, 1.0], dtype=np.float32)
    for p, site in ((0.1, 9), (0.05, 2), (0.5, 27)):
        use_dp = dp if offset == 0 else None
        got = O.dropout_keep_scale(n, per_sample, p, seed, site, use_dp, offset=offset)
        assert got.dtype == np.float32 and got.shape == (n,)
        for e in rs.randint(0, n, size=300):
            want = _scalar_dropout_factor(offset + int(e), per_sample, p, seed, site, use_dp)
            assert got[e] == want, (p, site, int(e))


def test_attention_keep_matches_the_kernel_arithmetic():
    rs = np.random.RandomState(5)
    for seed in (0, 77, 0x0123_4567_89AB_CDEF):
        bh, ti, tj = rs.randint(0, 64, 500), rs.randint(0, 256, 500), rs.randint(0, 256, 500)
        for p in (0.05, 0.5):
            got = O.attention_keep(seed, bh, ti, tj, p)
            want = [_scalar_attention_keep(seed, int(a), int(b), int(c), p) for a, b, c in zip(bh, ti, tj)]
            assert got.tolist() == want


def _within_4_sigma(frac, q, n):
    return abs(frac - q) <= 4.0 * (q * (1 - q) / n) ** 0.5


@pytest.mark.parametrize("p", [0.05, 0.1, 0.5])
def test_dropout_keep_rate_and_scale(p):
    n = 1 << 24
    sc = O.dropout_keep_scale(n, n, p, 0xABCDEF_0000_1234, 8 * 3 + 2)
    kept = sc != 0
    assert _within_4_sigma(float(kept.mean()), 1 - p, n), float(kept.mean())
    assert np.all(sc[kept] == np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


@pytest.mark.parametrize("p", [0.05, 0.5])
def test_attention_keep_rate(p):
    B, H, T = 2, 4, 256
    bh = np.arange(B * H).reshape(-1, 1, 1)
    t = np.arange(T)
    keep = O.attention_keep(12345, bh, t.reshape(1, -1, 1), t.reshape(1, 1, -1), p)
    n = keep.size
    assert _within_4_sigma(float(keep.mean()), 1 - p, n), float(keep.mean())


# ------------------------------------------------------------------------------------------------
# the oracle's regs injection
# ------------------------------------------------------------------------------------------------
CFG = dict(nb_cls=12, W=200, D=64, depth=4, heads=2, B=3, seed=4)       # T = 50: padded windows in blocks 0 / 1


def _setup():
    sd = O.init_state_dict(CFG["nb_cls"], [64, CFG["W"]], seed=CFG["seed"], embed_dim=CFG["D"], depth=CFG["depth"],
                           num_heads=CFG["heads"], variant="window")
    x = torch.from_numpy(np.random.RandomState(5).rand(CFG["B"], 1, 64, CFG["W"]).astype(np.float32))
    return sd, x


def _fwd(sd, x, regs=None):
    with torch.no_grad():
        return O.forward({k: v.clone() for k, v in sd.items()}, x, training=False, num_heads=CFG["heads"],
                         variant="window", regs=regs)


def _ones_regs(B, T, D, H, depth):
    regs = []
    for win, _ in O.window_blocks(depth):
        Tp = -(-T // win) * win if win else T
        regs.append({"attn": torch.ones(B, H, Tp, Tp), "proj": torch.ones(B, T, D), "fc1": torch.ones(B, T, 4 * D),
                     "fc2": torch.ones(B, T, D), "dp1": torch.ones(B), "dp2": torch.ones(B)})
    return regs


def test_all_ones_regs_are_bit_identical_to_none():
    sd, x = _setup()
    B, T, D, H = CFG["B"], CFG["W"] // 4, CFG["D"], CFG["heads"]
    base = _fwd(sd, x)
    assert torch.equal(_fwd(sd, x, _ones_regs(B, T, D, H, CFG["depth"])), base)
    # and train_step's loss / gradients
    tg = torch.from_numpy(np.random.RandomState(6).randint(1, CFG["nb_cls"], size=12).astype(np.int32))
    tl = torch.tensor([4, 5, 3], dtype=torch.int32)
    mask = torch.ones(T)
    l0, g0, _ = O.train_step({k: v.clone() for k, v in sd.items()}, x, tg, tl, mask, variant="window", num_heads=H)
    l1, g1, _ = O.train_step({k: v.clone() for k, v in sd.items()}, x, tg, tl, mask, variant="window", num_heads=H,
                             regs=_ones_regs(B, T, D, H, CFG["depth"]))
    assert l0 == l1 and all(torch.equal(g0[k], g1[k]) for k in g0)


@pytest.mark.parametrize("block,which", [(0, "dp1"), (1, "dp2"), (3, "dp1")])
def test_zero_drop_path_removes_exactly_that_samples_branch(block, which):
    sd, x = _setup()
    B, T, D = CFG["B"], CFG["W"] // 4, CFG["D"]
    regs = [{} for _ in range(CFG["depth"])]
    regs[block][which] = torch.tensor([1.0, 0.0, 1.0])
    got = _fwd(sd, x, regs)
    base = _fwd(sd, x)
    # the other samples are untouched, bit for bit; sample 1 changes
    assert torch.equal(got[0], base[0]) and torch.equal(got[2], base[2])
    assert not torch.allclose(got[1], base[1])
    # sample 1 equals the forward whose branch output is zeroed for that sample by its dropout factor instead
    zero = torch.ones(B, T, D)
    zero[1] = 0
    alt = [{} for _ in range(CFG["depth"])]
    alt[block]["proj" if which == "dp1" else "fc2"] = zero
    assert torch.equal(got, _fwd(sd, x, alt))


def test_window_attention_scale_gathers_tokens_of_the_rolled_windows():
    B, H, T, window, shift = 1, 1, 40, 16, 8
    Tp = 48
    s = torch.arange(Tp * Tp, dtype=torch.float32).reshape(1, 1, Tp, Tp)
    w = O.window_attention_scale(s, window, shift)
    assert w.shape == (Tp // window, 1, window, window)
    for r_i in range(Tp):
        for c in range(window):
            r_j = (r_i // window) * window + c
            ti, tj = (r_i + shift) % Tp, (r_j + shift) % Tp
            assert w[r_i // window, 0, r_i % window, c] == s[0, 0, ti, tj]


# ------------------------------------------------------------------------------------------------
# model_window argument checks (host only)
# ------------------------------------------------------------------------------------------------
def _window_model(depth=4):
    import htrvt_b200  # noqa: F401
    Wm = import_module("htr-vt_b200.model_window.HTR_VT")
    return Wm.MaskedAutoencoderViT(12, img_size=[64, 128], patch_size=(4, 64), embed_dim=256, depth=depth,
                                   num_heads=2, mlp_ratio=4, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))


@pytest.mark.parametrize("kw", [dict(drop=1.0), dict(drop=-0.1), dict(drop=float("nan")), dict(attn_drop=1.0),
                                dict(attn_drop=-1e-3), dict(attn_drop=float("nan")), dict(drop_path_rate=1.01),
                                dict(drop_path_rate=-0.5), dict(drop_path_rate=float("nan"))])
def test_set_stochastic_refuses_rates_outside_their_range(kw):
    m = _window_model()
    before = (m.drop, m.attn_drop, list(m.drop_path))
    with pytest.raises(ValueError):
        m.set_stochastic(**kw)
    assert (m.drop, m.attn_drop, list(m.drop_path)) == before


def test_drop_path_rate_one_gives_zero_scales_not_nan():
    m = _window_model()
    m.set_stochastic(0.0, 0.0, 1.0)
    torch.manual_seed(3)
    rng = m._train_rng(5, torch.device("cpu"))
    dp1, dp2 = rng["drop_path"][-1]
    assert torch.equal(dp1, torch.zeros(5)) and torch.equal(dp2, torch.zeros(5))
    for pair in rng["drop_path"][1:-1]:
        for dp in pair:
            assert torch.isfinite(dp).all()
