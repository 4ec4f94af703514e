"""GPU parity: tcgen05 attention fwd/bwd vs an fp32 torch reference of Attention.forward
(model_v1/model/HTR_VT.py:32-36) on the same bf16 q, k, v."""
from importlib import import_module

import numpy as np
import pytest
import torch

import htrvt_oracle as O

pytestmark = pytest.mark.gpu


def ops():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200.ops")


def _rel(a, b):
    return float((a.float() - b.float()).abs().max() / (b.float().abs().max() + 1e-12))


@pytest.mark.parametrize("B,H,T", [(2, 6, 128), (128, 6, 128), (3, 2, 32), (2, 6, 96)])
def test_attention_fwd_bwd(B, H, T):
    o = ops()
    hd = 128
    torch.manual_seed(0)
    qkv_tm = (torch.randn(B, T, 3, H, hd, device="cuda") * 0.7).bfloat16()     # token-major, as the QKV GEMM writes it
    qkv = qkv_tm.permute(2, 0, 3, 1, 4)
    scale = hd ** -0.5
    out = torch.empty(B, T, H * hd, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, T, device="cuda")
    o.attention_fwd(qkv_tm, out, lse, scale)
    q, k, v = [t.float().requires_grad_(True) for t in qkv]
    s = (q @ k.transpose(-2, -1)) * scale
    p = s.softmax(-1)
    ref = (p @ v).transpose(1, 2).reshape(B, T, H * hd)
    assert _rel(out, ref) < 1.5e-2
    assert _rel(lse, torch.logsumexp(s, -1)) < 1e-4
    dout = torch.randn(B, T, H * hd, device="cuda").bfloat16()
    ref.backward(dout.float())
    dqkv = torch.empty(B, T, 3, H, hd, device="cuda", dtype=torch.bfloat16)
    o.attention_bwd(qkv_tm, out, dout, lse, dqkv, scale)
    for i, t in enumerate((q, k, v)):
        want = t.grad.permute(0, 2, 1, 3)          # [B,T,H,hd]
        assert _rel(dqkv[:, :, i], want) < 2e-2, i


def _ref_attention2(qkv_tm, table, prel, window, shift, scale, keep=None):
    """fp32 torch restatement of model_window Attention.forward + Block._attend (model_window/model/HTR_VT.py:33-62,
    114-154) on given q, k, v (token-major [B,T,3,H,hd]), INCLUDING the branch for T not a multiple of the window:
    pad to Tp with tokens whose keys are masked (key_padding_mask rolled with the tokens, finfo.min fill, :49-56,
    :121-131) and whose query rows are stripped.  keep: optional attention-dropout keep-scale [B,H,Tp,Tp] over token
    indices, applied to the probabilities after the softmax (timm attn_drop)."""
    B, T, _, H, hd = qkv_tm.shape
    qkv = qkv_tm.float()
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
        attn = attn + table[idx[:N, :N]].permute(2, 0, 1).unsqueeze(0)
    if window > 0:
        attn = attn.masked_fill(~valid.reshape(B * (Tp // N), 1, 1, N), torch.finfo(attn.dtype).min)
    lse = torch.logsumexp(attn, -1)                                    # [Bw, H, N]
    prob = attn.softmax(-1)
    if keep is not None:
        prob = prob * (O.window_attention_scale(keep, window, shift) if window > 0 else keep)
    out = (prob @ v).transpose(1, 2).reshape(B, Tp, H * hd)
    lse = lse.reshape(B, Tp // N, H, N).permute(0, 2, 1, 3).reshape(B, H, Tp)
    if window > 0 and shift > 0:
        out = torch.roll(out, shifts=(shift,), dims=1)
        lse = torch.roll(lse, shifts=(shift,), dims=2)
    return out[:, :T], lse[:, :, :T]


ATTN2_SHAPES = [
    (2, 6, 256, 256, 0, 0, True),      # global block of the wide-line model (T = 256)
    (2, 6, 256, 256, 16, 0, True),     # windowed block 0
    (2, 6, 256, 256, 16, 8, True),     # shifted windows: the wrap-around window mixes head and tail tokens
    (3, 2, 128, 128, 16, 8, True),
    (2, 3, 128, 128, 0, 0, True),
    (2, 2, 208, 256, 0, 0, True),      # ragged: T not a multiple of 128
    (2, 2, 48, 64, 16, 0, True),
    (2, 2, 256, 0, 0, 0, False),       # no bias table
    # token counts that are not a multiple of the 16-token window (W = 1000 / 600 / 808 / 360 lines): zero padding,
    # rolled key-padding mask, padded queries stripped (model_window/model/HTR_VT.py:121-131, 49-56)
    (2, 6, 250, 250, 16, 0, True),
    (2, 6, 250, 250, 16, 8, True),
    (2, 2, 150, 150, 16, 8, True),
    (2, 2, 202, 256, 16, 8, True),
    (3, 2, 90, 128, 16, 8, True),
    (2, 2, 90, 128, 16, 0, True),
    (2, 2, 200, 200, 16, 8, True),     # Tp = 208: multiple of 16 but not of 128
    (1, 2, 7, 16, 16, 8, True),        # shorter than one window
    (2, 2, 250, 250, 0, 0, True),      # global attention at the same ragged length
]


# drop_p 0 keeps the ids the shapes had before the dropout variants were added
@pytest.mark.parametrize("B,H,T,prel,window,shift,bias,drop_p", [
    pytest.param(*shape, d, id="-".join(str(v) for v in shape) + ("" if d == 0 else "-drop%g" % d))
    for shape in ATTN2_SHAPES for d in (0.0, 0.05)])
def test_attention2_fwd_bwd(B, H, T, prel, window, shift, bias, drop_p):
    o = ops()
    hd = 128
    torch.manual_seed(1)
    qkv_tm = (torch.randn(B, T, 3, H, hd, device="cuda") * 0.7).bfloat16().requires_grad_(False)
    table = (torch.randn(2 * prel - 1, H, device="cuda") * 0.5) if bias else None
    scale = hd ** -0.5
    seed = 0x5EED_0000_0000_0000 + 1234 * T + 16 * shift
    keep = None
    if drop_p > 0:              # the kernels' own mask (attn_keep), restated on the host: 0 or 1 / (1 - p)
        Tp = -(-T // window) * window if window else T
        t = np.arange(Tp)
        k = O.attention_keep(seed, np.arange(B * H).reshape(B, H, 1, 1), t.reshape(1, 1, Tp, 1),
                             t.reshape(1, 1, 1, Tp), drop_p)
        keep = torch.from_numpy(np.where(k, 1.0 / (1.0 - drop_p), 0.0).astype(np.float32)).cuda()
    out = torch.empty(B, T, H * hd, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, T, device="cuda")
    o.attention2_fwd(qkv_tm, out, lse, scale, table, prel, window, shift, drop_p, seed)
    x = qkv_tm.float().requires_grad_(True)
    tb = table.clone().requires_grad_(True) if bias else None
    ref, ref_lse = _ref_attention2(x, tb, prel, window, shift, scale, keep)
    assert _rel(out, ref) < 1.5e-2
    assert _rel(lse, ref_lse) < 1e-3
    dout = torch.randn(B, T, H * hd, device="cuda").bfloat16()
    ref.backward(dout.float())
    dqkv = torch.full((B, T, 3, H, hd), 7.0, device="cuda", dtype=torch.bfloat16)
    dtable = torch.zeros_like(table) if bias else None
    o.attention2_bwd(qkv_tm, out, dout, lse, dqkv, scale, table, prel, window, shift, dtable, drop_p, seed)
    for i in range(3):
        assert _rel(dqkv[:, :, i], x.grad[:, :, i]) < 2.5e-2, i
    if bias:
        assert _rel(dtable, tb.grad) < 2e-2


def test_attention2_dropout_statistics():
    """Attention dropout statistics of the forward: the same seed gives the same output, the keep rate recovered with
    a one-hot V probe matches 1 - p, and kept probabilities are scaled by 1 / (1 - p).  (The masks themselves, forward
    and backward, are compared pair by pair with the host restatement in test_gpu_window_regularisers.py.)"""
    o = ops()
    B, H, T, hd, p = 2, 2, 256, 128, 0.25
    torch.manual_seed(2)
    qkv_tm = (torch.randn(B, T, 3, H, hd, device="cuda") * 0.3).bfloat16()
    scale = hd ** -0.5
    out0 = torch.empty(B, T, H * hd, device="cuda", dtype=torch.bfloat16)
    out1 = torch.empty_like(out0)
    out2 = torch.empty_like(out0)
    lse = torch.empty(B, H, T, device="cuda")
    o.attention2_fwd(qkv_tm, out0, lse, scale, None, 0, 0, 0, 0.0, 0)
    o.attention2_fwd(qkv_tm, out1, lse, scale, None, 0, 0, 0, p, 1234)
    o.attention2_fwd(qkv_tm, out2, lse, scale, None, 0, 0, 0, p, 1234)
    assert torch.equal(out1, out2)                                   # same seed, same mask
    assert not torch.equal(out0, out1)
    # v = identity-like probe: recover the per-(i, j) keep mask by making V one-hot over the first 128 keys
    probe = qkv_tm.clone()
    probe[:, :, 2] = 0
    eye = torch.eye(hd, device="cuda").bfloat16()
    probe[:, :hd, 2] = eye[None, :, None, :].expand(B, hd, H, hd)
    po = torch.empty_like(out0)
    pd = torch.empty_like(out0)
    o.attention2_fwd(probe, po, lse, scale, None, 0, 0, 0, 0.0, 0)
    o.attention2_fwd(probe, pd, lse, scale, None, 0, 0, 0, p, 99)
    kept = (pd.float().abs() > 0).float().mean() / (po.float().abs() > 0).float().mean()
    assert abs(float(kept) - (1 - p)) < 0.02
    ratio = pd.float()[po.float().abs() > 1e-4] / po.float()[po.float().abs() > 1e-4]
    nz = ratio[ratio.abs() > 0]
    assert abs(float(nz.median()) - 1 / (1 - p)) < 0.05
