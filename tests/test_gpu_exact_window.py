"""fp32-parity mode of the windowed variant (model_window): `set_precision("fp32")` runs the relative-position-bias,
shifted-window attention in fp32 (csrc/exact.cu attention2_f32_kernel) between split-bf16 contractions.
  * the kernel against a float64 restatement of the reference attention, and its argument rules against the 16-bit one;
  * logits against the unmodified reference (committed goldens) within the north_star fp32 bound of 1e-4;
  * greedy decode and the LM-rescored K-best beam (model_window/test_with_kenlm.py:25-59) end to end against the
    oracle, whose window forward reproduces those goldens bit for bit;
  * uint8 lines with widths, and the refusals the mode carries over."""
import ctypes
import os
from importlib import import_module

import numpy as np
import pytest
import torch

import htrvt_oracle as O

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
NB_CLS, W_LINE = 90, 1024
ALPHABET = "".join(chr(33 + i) for i in range(NB_CLS - 1))


def ops():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200.ops")


def _rel(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def _images(seed, B, W):
    return torch.from_numpy(np.random.RandomState(seed).rand(B, 1, 64, W).astype(np.float32))


def _window_model(nb_cls, W, seed):
    """create_model with the reference's img_size = [W, H] convention for this variant, seeded oracle weights."""
    import htrvt_b200  # noqa: F401
    Wm = import_module("htr-vt_b200.model_window.HTR_VT")
    m = Wm.create_model(nb_cls, [W, 64])
    sd = O.init_state_dict(nb_cls, [64, W], seed=seed, variant="window")
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval(), sd


# ------------------------------------------------------------------------------------------------
# 1. kernel
# ------------------------------------------------------------------------------------------------
def _ref_attention2_f64(qkv_tm, table, prel, window, shift, scale):
    """float64 restatement of model_window Attention.forward + Block._attend (model_window/model/HTR_VT.py:33-62,
    114-154) on given q, k, v (token-major [B,T,3,H,hd]): pad to a multiple of the window with zero tokens whose keys
    are masked (mask rolled with the tokens, finfo.min fill), roll by -shift, attend per window with the window-local
    bias, roll back, strip the padded rows."""
    B, T, _, H, hd = qkv_tm.shape
    qkv = qkv_tm.double()
    Tp = T
    valid = torch.ones(B, T, dtype=torch.bool, device=qkv.device)
    if window > 0:
        pad = (window - T % window) % window
        Tp = T + pad
        if pad:
            qkv = torch.cat([qkv, qkv.new_zeros(B, pad, 3, H, hd)], dim=1)
            valid = torch.cat([valid, valid.new_zeros(B, pad)], dim=1)
        if shift > 0:
            qkv = torch.roll(qkv, shifts=(-shift,), dims=1)
            valid = torch.roll(valid, shifts=(-shift,), dims=1)
    N = window if window > 0 else T
    z = qkv.reshape(B * (Tp // N), N, 3, H, hd).permute(2, 0, 3, 1, 4)
    q, k, v = z[0], z[1], z[2]
    attn = (q @ k.transpose(-2, -1)) * scale
    if table is not None:
        coords = torch.arange(prel, device=qkv.device)
        idx = (coords[None, :] - coords[:, None]) + prel - 1
        attn = attn + table.double()[idx[:N, :N]].permute(2, 0, 1).unsqueeze(0)
    if window > 0:
        attn = attn.masked_fill(~valid.reshape(B * (Tp // N), 1, 1, N), torch.finfo(attn.dtype).min)
    out = (attn.softmax(-1) @ v).transpose(1, 2).reshape(B, Tp, H * hd)
    if window > 0 and shift > 0:
        out = torch.roll(out, shifts=(shift,), dims=1)
    return out[:, :T]


# the shape list of test_gpu_attention.py::test_attention2_fwd_bwd
@pytest.mark.parametrize("B,H,T,prel,window,shift,bias", [
    (2, 6, 256, 256, 0, 0, True),
    (2, 6, 256, 256, 16, 0, True),
    (2, 6, 256, 256, 16, 8, True),
    (3, 2, 128, 128, 16, 8, True),
    (2, 3, 128, 128, 0, 0, True),
    (2, 2, 208, 256, 0, 0, True),
    (2, 2, 48, 64, 16, 0, True),
    (2, 2, 256, 0, 0, 0, False),
    (2, 6, 250, 250, 16, 0, True),
    (2, 6, 250, 250, 16, 8, True),
    (2, 2, 150, 150, 16, 8, True),
    (2, 2, 202, 256, 16, 8, True),
    (3, 2, 90, 128, 16, 8, True),
    (2, 2, 90, 128, 16, 0, True),
    (2, 2, 200, 200, 16, 8, True),
    (1, 2, 7, 16, 16, 8, True),
    (2, 2, 250, 250, 0, 0, True),
])
def test_attention2_f32_matches_float64(B, H, T, prel, window, shift, bias):
    o = ops()
    hd = 128
    torch.manual_seed(1)
    qkv = torch.randn(B, T, 3, H, hd, device="cuda") * 0.7
    table = (torch.randn(2 * prel - 1, H, device="cuda") * 0.5) if bias else None
    scale = hd ** -0.5
    out = torch.full((B * T, H * hd), 7.0, device="cuda")
    got = o.attention2_f32(qkv, B, H, T, hd, scale, table, prel, window, shift, out=out)
    assert got.data_ptr() == out.data_ptr()
    assert not bool((out == 7.0).all(-1).any()), "rows left unwritten"
    ref = _ref_attention2_f64(qkv, table, prel, window, shift, scale)
    err = _rel(out.view(B, T, H * hd), ref)
    assert err < 2e-6, err


def _status(fn, *args):
    return int(fn(*args, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))


@pytest.mark.parametrize("B,H,T,hd,window,shift,prel,with_table", [
    (1, 2, 257, 128, 0, 0, 0, False),       # T > 256
    (1, 2, 64, 128, 8, 0, 0, False),        # window other than 0 / 16
    (1, 2, 64, 128, 16, 4, 0, False),       # shift not a multiple of 8
    (1, 2, 64, 128, 16, 16, 0, False),      # shift >= window
    (1, 2, 64, 128, 0, 8, 0, False),        # shift with global attention
    (1, 2, 64, 128, 0, 0, 32, True),        # Prel < T with a table
    (1, 2, 64, 128, 16, 8, 32, True),
    (1, 2, 64, 128, 0, 0, 257, True),       # table of more than 511 rows
    (1, 2, 64, 64, 0, 0, 64, True),         # head_dim 64
    (1, 2, 0, 128, 0, 0, 0, False),         # empty sequence
    (1, 2, 20, 128, 16, 8, 32, True),       # valid: both run
])
def test_attention2_f32_accepts_what_attention2_fwd_accepts(B, H, T, hd, window, shift, prel, with_table):
    o = ops()
    L = import_module("htr-vt_b200._lib").lib()
    n = max(B * max(T, 1) * 3 * H * 128, 1)
    q32 = torch.randn(n, device="cuda")
    q16 = q32.bfloat16()
    o32 = torch.empty(n, device="cuda")
    o16 = torch.empty(n, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(max(B * H * T, 1), device="cuda")
    tbl = torch.randn(max(2 * prel - 1, 1), H, device="cuda") if with_table else None
    p = o._p
    s32 = _status(L.htrvt_attention2_f32, p(q32), B, H, T, hd, 0.1, p(tbl), prel, window, shift, p(o32))
    s16 = _status(L.htrvt_attention2_fwd, p(q16), B, H, T, hd, 0.1, p(tbl), prel, window, shift, 0.0, 0, p(o16), p(lse))
    torch.cuda.synchronize()
    assert s32 == s16, (s32, s16)
    assert s32 == (0 if (T, hd, window, shift, prel) == (20, 128, 16, 8, 32) else -1)


# ------------------------------------------------------------------------------------------------
# 3. logits against the unmodified reference
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["win_full", "win_w1000", "win_w600"])
def test_fp32_mode_window_logits_within_1e4_of_reference(tag):
    g = np.load(os.path.join(G, tag + ".npz"), allow_pickle=True)
    meta = [int(v) for v in g["meta"]]
    nb_cls, W, B, seed = meta[:4]
    if tag == "win_full":                         # built as test_gpu_model.py builds this fixture
        from functools import partial
        import htrvt_b200  # noqa: F401
        Wm = import_module("htr-vt_b200.model_window.HTR_VT")
        D, depth, heads = meta[4:7]
        m = Wm.MaskedAutoencoderViT(nb_cls, img_size=[64, W], patch_size=(4, 64), embed_dim=D, depth=depth,
                                    num_heads=heads, mlp_ratio=4, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))
        sd = O.init_state_dict(nb_cls, [64, W], seed=seed, embed_dim=D, depth=depth, num_heads=heads, variant="window")
        m.load_state_dict(sd, strict=True)
        m = m.cuda().eval()
    else:
        m, _ = _window_model(nb_cls, W, seed)
    x = _images(seed + 1, B, W).cuda()
    want = torch.from_numpy(g["logits_eval"])
    m.set_precision("fp32")
    with torch.no_grad():
        got = m(x)
    assert got.dtype == torch.float32 and got.shape == want.shape == (B, W // 4, nb_cls)
    err = _rel(got.cpu(), want)
    print("%s: fp32-mode logits relative error vs the reference %.3g" % (tag, err))
    assert err < 1e-4, err
    m.set_precision("bf16")
    with torch.no_grad():
        err16 = _rel(m(x).float().cpu(), want)
    assert err16 < 2e-2, err16


# ------------------------------------------------------------------------------------------------
# 4. greedy decode and the LM-rescored beam, end to end, against the oracle
# ------------------------------------------------------------------------------------------------
class StubLM(object):
    """Deterministic stand-in for KenLMTextScorer (oracle/make_golden.py): any object with .score(text)."""

    def score(self, text):
        return sum(((ord(ch) * 31 + i * 17) % 97) / 97.0 for i, ch in enumerate(text)) - 0.6 * len(text)


# Seed of the weights and the 16 lines.  The K-best path beam orders its candidates by float64 sums of log-probs; with
# seeded random weights neighbouring candidates are often near-ties (two paths that each leave the top-1 class at one
# different frame whose top-1 / top-2 margins almost coincide): over seeds 1-44 the smallest gap between consecutive
# candidate scores of the 16 lines ranged from 1.7e-6 to 3.5e-4.  Seed 33 has the widest (3.5e-4; smallest top-1 /
# top-2 logit margin 1.59); the test asserts that margin against the measured deviation.
DECODE_SEED = 33


def test_fp32_mode_decode_and_lm_beam_match_the_oracle():
    import htrvt_b200 as h
    beam = import_module("htr-vt_b200.beam")
    B, K = 16, 5
    m, sd = _window_model(NB_CLS, W_LINE, DECODE_SEED)
    x = _images(DECODE_SEED + 1, B, W_LINE)
    with torch.no_grad():
        ref = O.forward(sd, x, training=False, num_heads=6, variant="window")          # CPU fp32: the oracle
    m.set_precision("fp32")
    conv = h.CTCLabelConverter(ALPHABET)
    T = W_LINE // 4
    with torch.no_grad():
        preds = m(x.cuda())
        # the reference's call sequence (valid.py:32-42) on the drop-in objects, and the fused device decode
        lp = preds.permute(1, 0, 2).log_softmax(2)
        _, idx = lp.max(2)
        idx = idx.transpose(1, 0).contiguous().view(-1)
        strings = conv.decode(idx.data, torch.IntTensor([T] * B))
        fused = conv.decode_logits(preds)
        kb = beam.kbest_candidates(lp, conv, beam_size=K, search="paths")
        picked = beam.beam_search_with_lm_batch(lp, conv, StubLM(), beam_size=K)
    dlogit = float((preds.cpu().double() - ref.double()).abs().max())
    assert _rel(preds.cpu(), ref) < 1e-4
    # greedy: the oracle's strings through the same sequence; no frame's top-2 is within reach of the deviation
    ref_lp = ref.permute(1, 0, 2).log_softmax(2)
    ref_idx = ref_lp.max(2)[1].transpose(1, 0).contiguous().view(-1).numpy()
    want = O.decode_strings(ref_idx, [T] * B, ALPHABET)
    top2 = ref.double().topk(2, -1)[0]
    assert float((top2[..., 0] - top2[..., 1]).min()) > 10 * dlogit
    assert strings == want
    assert fused == want
    # K-best paths: strings and order equal the oracle's; scores within the bound the logit deviation implies
    ref_lp_b = ref.log_softmax(2).numpy()                                 # [B, T, C] fp32, as the device beam reads
    min_gap, gap_dev, score_dev = np.inf, 0.0, 0.0
    for b in range(B):
        paths = O.kbest_paths(ref_lp_b[b], K)
        sc = [s for _, s in paths]
        min_gap = min(min_gap, min(sc[i] - sc[i + 1] for i in range(K - 1)))
        oc = []
        for text, s in paths:
            st = O.decode_strings(np.array(text, dtype=np.int64), [len(text)], ALPHABET)[0]
            if st:
                oc.append((st, s))
        assert [c[0] for c in kb[b]] == [c[0] for c in oc], b
        got_s, want_s = np.array([c[1] for c in kb[b]]), np.array([c[1] for c in oc])
        score_dev = max(score_dev, float(np.abs(got_s - want_s).max()))
        if len(got_s) > 1:
            gap_dev = max(gap_dev, float(np.abs(np.diff(got_s) - np.diff(want_s)).max()))
        assert picked[b] == O.beam_search_with_lm(ref_lp_b[b], ALPHABET, StubLM().score, K), b
    print("logit deviation %.3g, score deviation %.3g, deviation of score differences %.3g, smallest gap %.3g"
          % (dlogit, score_dev, gap_dev, min_gap))
    # a log-prob moves by at most twice the largest logit deviation (the log-sum-exp moves by at most that much once):
    # a path score summed over T frames by at most 2 T dlogit
    assert score_dev <= 2 * T * dlogit + 1e-9, (score_dev, dlogit)
    # not a vacuous pass: two neighbouring candidates share all but a few frames, so what can reorder them is the
    # deviation of their score DIFFERENCE (the common frames cancel); the oracle's smallest gap is well above it
    assert min_gap > 10 * gap_dev, (min_gap, gap_dev)


# ------------------------------------------------------------------------------------------------
# 5. ragged uint8 lines with widths
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,widths", [
    (1000, [1000, 812, 433, 97]),     # T = 250: the last window holds 10 tokens and 6 padded positions
    (964, [964, 640, 301, 12]),       # T = 241: the last window holds 1 token and 15 padded positions
])
def test_fp32_mode_uint8_widths_match_the_oracle(W, widths):
    m, sd = _window_model(NB_CLS, W_LINE, 31)
    B = len(widths)
    u8 = torch.from_numpy(np.random.RandomState(W).randint(0, 256, size=(B, 1, 64, W)).astype(np.uint8))
    wd = torch.tensor(widths, dtype=torch.int32)
    x = u8.float() / 255.
    for b, w in enumerate(widths):
        x[b, :, :, w:] = 1.0
    with torch.no_grad():
        ref = O.forward(sd, x, training=False, num_heads=6, variant="window")
    m.set_precision("fp32")
    with torch.no_grad():
        got = m(u8.cuda(), widths=wd)
    assert got.shape == ref.shape == (B, W // 4, NB_CLS)
    err = _rel(got.cpu(), ref)
    print("W=%d: fp32-mode uint8 + widths vs the oracle %.3g" % (W, err))
    assert err < 1e-4, err


# ------------------------------------------------------------------------------------------------
# 6. refusals carried over
# ------------------------------------------------------------------------------------------------
def test_fp32_mode_window_refusals():
    import htrvt_b200 as h
    m, _ = _window_model(NB_CLS, 512, 5)
    m.set_precision("fp32")
    x = _images(6, 2, 512).cuda()
    m.train()
    with pytest.raises(h._lib.HtrvtError):
        m(x)
    m.eval()
    with pytest.raises(ValueError, match="exceeds configured num_patches"):
        with torch.no_grad():
            m(_images(7, 1, 1024).cuda())
    with torch.no_grad():
        assert m(x).shape == (2, 128, NB_CLS)
