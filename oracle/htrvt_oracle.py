"""CPU oracle for the HTR-VT hot path.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference` legs may
import this file; the product (htr-vt_b200/) never does.

It restates, on the CPU and in functional form over a plain `state_dict`, what the reference
computes on the hot path.  Each function cites the reference lines it follows (paths relative
to /root/reference).  Pinning: tests/golden/*.npz were produced by oracle/make_golden.py from
the UNMODIFIED reference modules imported in the dev container; tests/test_oracle.py checks this
restatement against them (the reference itself ships no golden vectors: its tests/ are 0-byte
files, so those generated fixtures are the pin).

Third-party arithmetic the reference delegates to (absent from /root/reference):
  * torch.nn.CTCLoss  (torch==1.13.0+cu116, environment.yaml:87)  -> ctc_loss_grad() below
    restates the published Graves alpha/beta recursion in float64;
  * timm.Mlp / DropPath (timm==1.0.9, environment.yaml:86)          -> _mlp() below.
"""
from __future__ import annotations

import math
from collections import OrderedDict

import re

import numpy as np
import torch
import torch.nn.functional as F

# ----------------------------------------------------------------------------------------------
# Architecture constants fixed by the reference factory (model_v1/model/HTR_VT.py:244-254)
# ----------------------------------------------------------------------------------------------
V1 = dict(embed_dim=768, depth=4, num_heads=6, mlp_ratio=4, patch=(4, 64), ln_eps=1e-6)


def sincos_pos_embed(embed_dim: int, grid_size) -> np.ndarray:
    """2-D sin/cos table laid over the token axis (model_v1/model/HTR_VT.py:86-131).

    The reference meshgrids (grid_w, grid_h) and encodes grid[0] in the first half of the
    channels and grid[1] in the second half; omega is float64.
    """
    gh, gw = int(grid_size[0]), int(grid_size[1])
    col = np.tile(np.arange(gw, dtype=np.float32), gh)          # n % gw
    row = np.repeat(np.arange(gh, dtype=np.float32), gw)        # n // gw
    half = embed_dim // 2
    omega = 1.0 / 10000 ** (np.arange(half // 2, dtype=np.float64) / (half / 2.0))

    def enc(pos):
        ang = np.einsum("m,d->md", pos, omega)
        return np.concatenate([np.sin(ang), np.cos(ang)], axis=1)

    return np.concatenate([enc(col), enc(row)], axis=1)         # [gh*gw, embed_dim]


def stem_plan(embed_dim: int):
    """Layer list of the truncated ResNet-18 stem (model_v1/model/resnet18.py:42-84)."""
    c1, c2, c3 = embed_dim // 4, embed_dim // 2, embed_dim
    return [("layer1", c1, c1, (2, 1)), ("layer2", c1, c2, (2, 2)), ("layer3", c2, c3, (2, 2))]


def init_state_dict(nb_cls: int, img_size, seed: int = 123, embed_dim: int = 768, depth: int = 4,
                    num_heads: int = 6, mlp_ratio: int = 4, variant: str = "v1",
                    bn_noise: bool = True) -> "OrderedDict[str, torch.Tensor]":
    """Deterministic (numpy RandomState) weights with the reference's state_dict schema.

    Not the reference's initialiser (which draws from torch's global RNG); it produces tensors of
    the same shapes and comparable scales so that both implementations can be loaded with the same
    values through `load_state_dict` (SURVEY.md 8b).  `bn_noise` perturbs BN affine/running stats
    so that eval-mode BN is not an identity.
    """
    rs = np.random.RandomState(seed)
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()

    def t(a):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))

    def conv(name, cout, cin, k):
        bound = 1.0 / math.sqrt(cin * k * k)
        sd[name] = t(rs.uniform(-bound, bound, size=(cout, cin, k, k)))

    def bn(name, c):
        if bn_noise:
            sd[name + ".weight"] = t(rs.uniform(0.8, 1.2, size=c))
            sd[name + ".bias"] = t(rs.uniform(-0.1, 0.1, size=c))
            sd[name + ".running_mean"] = t(rs.uniform(-0.05, 0.05, size=c))
            sd[name + ".running_var"] = t(rs.uniform(0.8, 1.2, size=c))
        else:
            sd[name + ".weight"] = torch.ones(c)
            sd[name + ".bias"] = torch.zeros(c)
            sd[name + ".running_mean"] = torch.zeros(c)
            sd[name + ".running_var"] = torch.ones(c)
        sd[name + ".num_batches_tracked"] = torch.zeros((), dtype=torch.int64)

    def linear(name, cout, cin, bias_scale=0.02):
        bound = math.sqrt(6.0 / (cin + cout))
        sd[name + ".weight"] = t(rs.uniform(-bound, bound, size=(cout, cin)))
        sd[name + ".bias"] = t(rs.uniform(-bias_scale, bias_scale, size=cout))

    def ln(name, c):
        sd[name + ".weight"] = t(rs.uniform(0.9, 1.1, size=c))
        sd[name + ".bias"] = t(rs.uniform(-0.05, 0.05, size=c))

    H, W = int(img_size[0]), int(img_size[1])
    sd["mask_token"] = t(rs.normal(0, 0.02, size=(1, 1, embed_dim)))
    T = W // 4
    if variant == "v1":
        grid = [img_size[0] // 4, img_size[1] // 64]
        sd["pos_embed"] = t(sincos_pos_embed(embed_dim, grid))[None]
    conv("patch_embed.conv1.weight", embed_dim // 4, 1, 3)
    bn("patch_embed.bn1", embed_dim // 4)
    for lname, cin, cout, _stride in stem_plan(embed_dim):
        for b in range(2):
            ci = cin if b == 0 else cout
            conv(f"patch_embed.{lname}.{b}.conv1.weight", cout, ci, 3)
            bn(f"patch_embed.{lname}.{b}.bn1", cout)
            conv(f"patch_embed.{lname}.{b}.conv2.weight", cout, cout, 3)
            bn(f"patch_embed.{lname}.{b}.bn2", cout)
            if b == 0:
                conv(f"patch_embed.{lname}.0.downsample.0.weight", cout, ci, 1)
                bn(f"patch_embed.{lname}.0.downsample.1", cout)
    for i in range(depth):
        ln(f"blocks.{i}.norm1", embed_dim)
        linear(f"blocks.{i}.attn.qkv", 3 * embed_dim, embed_dim)
        linear(f"blocks.{i}.attn.proj", embed_dim, embed_dim)
        if variant == "window":
            sd[f"blocks.{i}.attn.relative_position_bias_table"] = t(
                rs.normal(0, 0.2, size=(2 * T - 1, num_heads)))
            coords = torch.arange(T)
            sd[f"blocks.{i}.attn.relative_position_index"] = (coords[None, :] - coords[:, None]) + T - 1
        ln(f"blocks.{i}.norm2", embed_dim)
        linear(f"blocks.{i}.mlp.fc1", mlp_ratio * embed_dim, embed_dim)
        linear(f"blocks.{i}.mlp.fc2", embed_dim, mlp_ratio * embed_dim)
    ln("norm", embed_dim)
    linear("head", nb_cls, embed_dim)
    return sd


def reorder_like(sd, ref_keys):
    """Return `sd` reordered to the reference's state_dict key order (strict load ignores order,
    but tests compare key lists)."""
    return OrderedDict((k, sd[k]) for k in ref_keys)


# ----------------------------------------------------------------------------------------------
# Forward pass
# ----------------------------------------------------------------------------------------------
def draw_span_mask(L: int, mask_ratio: float, max_span_length: int) -> torch.Tensor:
    """`generate_span_mask` (model_v1/model/HTR_VT.py:202-210): int(L*ratio)//span draws of
    torch.randint(L-span,(1,)) from the CPU default generator; one mask for the whole batch.
    Returns float mask [L] (1 = keep, 0 = replaced by mask_token)."""
    mask = torch.ones(L)
    num_spans = int(L * mask_ratio) // max_span_length
    for _ in range(num_spans):
        idx = int(torch.randint(L - max_span_length, (1,)))
        mask[idx:idx + max_span_length] = 0
    return mask


def _bn(sd, name, x, training, momentum=0.1):
    """nn.BatchNorm2d(eps=1e-5) (model_v1/model/resnet18.py:15,18,49,61): batch statistics and
    running-stat update in train mode, running statistics in eval mode."""
    rm, rv = sd[name + ".running_mean"], sd[name + ".running_var"]
    if training:
        sd[name + ".num_batches_tracked"] += 1
    return F.batch_norm(x, rm, rv, sd[name + ".weight"], sd[name + ".bias"], training, momentum, 1e-5)


def _basic_block(sd, p, x, stride, training):
    """BasicBlock.forward (model_v1/model/resnet18.py:23-39)."""
    out = F.conv2d(x, sd[p + ".conv1.weight"], None, stride, 1)
    out = F.relu(_bn(sd, p + ".bn1", out, training))
    out = F.conv2d(out, sd[p + ".conv2.weight"], None, 1, 1)
    out = _bn(sd, p + ".bn2", out, training)
    if (p + ".downsample.0.weight") in sd:
        res = F.conv2d(x, sd[p + ".downsample.0.weight"], None, stride, 0)
        res = _bn(sd, p + ".downsample.1", res, training)
    else:
        res = x
    return F.relu(out + res)


def stem_forward(sd, x, training):
    """ResNet18.forward (model_v1/model/resnet18.py:73-84)."""
    embed_dim = sd["patch_embed.layer3.1.conv2.weight"].shape[0]
    x = F.conv2d(x, sd["patch_embed.conv1.weight"], None, (2, 1), 1)
    x = F.relu(_bn(sd, "patch_embed.bn1", x, training))
    x = F.max_pool2d(x, 3, (2, 1), 1)
    for lname, _cin, _cout, stride in stem_plan(embed_dim):
        x = _basic_block(sd, f"patch_embed.{lname}.0", x, stride, training)
        x = _basic_block(sd, f"patch_embed.{lname}.1", x, 1, training)
    return F.max_pool2d(x, 3, (2, 1), 1)


def _attention(sd, p, x, num_heads, window=0, shift=0, regs=None):
    """Attention.forward (model_v1/model/HTR_VT.py:27-39); with the window variant's relative
    bias and 1-D window partition (model_window/model/HTR_VT.py:33-62, 114-154).
    regs: optional dict of one block's train-mode regularisers (see train_regs): "attn" multiplies the attention
    probabilities after the softmax (timm attn_drop), "proj" the projection's output (timm proj_drop)."""
    has_bias = (p + ".relative_position_bias_table") in sd
    ascale = regs.get("attn") if regs is not None else None
    pscale = regs.get("proj") if regs is not None else None

    def attend(z, key_mask=None, drop=None):
        Bz, N, C = z.shape
        hd = C // num_heads
        qkv = F.linear(z, sd[p + ".qkv.weight"], sd[p + ".qkv.bias"])
        qkv = qkv.reshape(Bz, N, 3, num_heads, hd).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0], qkv[1], qkv[2]
        attn = (q @ k.transpose(-2, -1)) * (hd ** -0.5)
        if has_bias:
            idx = sd[p + ".relative_position_index"][:N, :N]
            attn = attn + sd[p + ".relative_position_bias_table"][idx].permute(2, 0, 1).unsqueeze(0)
        if key_mask is not None:                       # True = valid key (model_window/model/HTR_VT.py:49-56)
            attn = attn.masked_fill(~key_mask.reshape(Bz, 1, 1, N), torch.finfo(attn.dtype).min)
        attn = attn.softmax(dim=-1)
        if key_mask is not None:
            attn = torch.nan_to_num(attn, nan=0.0)
        if drop is not None:                           # attention dropout: after the softmax, before @ v
            attn = attn * drop.to(attn.dtype)
        z = (attn @ v).transpose(1, 2).reshape(Bz, N, C)
        return F.linear(z, sd[p + ".proj.weight"], sd[p + ".proj.bias"])

    if window <= 0:
        x = attend(x, drop=ascale)
        return x if pscale is None else x * pscale.to(x.dtype)
    # Block._attend (model_window/model/HTR_VT.py:114-154): zero-pad to a multiple of the window, roll tokens and
    # the validity mask by -shift, attend inside consecutive windows with the padded keys masked, undo, strip
    B, N0, C = x.shape
    pad = (window - N0 % window) % window
    if pad:
        x = torch.cat([x, x.new_zeros(B, pad, C)], dim=1)
    N = N0 + pad
    valid = torch.ones(B, N, dtype=torch.bool, device=x.device)
    if pad:
        valid[:, -pad:] = False
    if shift > 0:
        x = torch.roll(x, shifts=(-shift,), dims=1)
        valid = torch.roll(valid, shifts=(-shift,), dims=1)
    drop = window_attention_scale(ascale, window, shift) if ascale is not None else None
    x = attend(x.reshape(B * (N // window), window, C), valid.reshape(B * (N // window), window),
               drop).reshape(B, N, C)
    if shift > 0:
        x = torch.roll(x, shifts=(shift,), dims=1)
    x = x[:, :N0]
    return x if pscale is None else x * pscale.to(x.dtype)


def window_attention_scale(scale, window, shift):
    """[B, H, Tp, Tp] attention keep-scale over ORIGINAL token indices (Tp = T padded to a multiple of the window) ->
    [B * Tp / window, H, window, window] in the layout of Block._attend's windows: rolled position r holds token
    (r + shift) mod Tp, and only the pairs inside one window are kept."""
    B, H, Tp, _ = scale.shape
    nw = Tp // window
    tok = (torch.arange(Tp, device=scale.device) + shift) % Tp
    s = scale[:, :, tok][:, :, :, tok].reshape(B, H, nw, window, nw, window)
    s = torch.diagonal(s, dim1=2, dim2=4)                      # [B, H, window, window, nw]
    return s.permute(0, 4, 1, 2, 3).reshape(B * nw, H, window, window)


def _mlp(sd, p, x, regs=None):
    """timm 1.0.9 Mlp with nn.GELU (erf form): fc1 -> GELU -> drop1 -> fc2 -> drop2; dropouts are p=0 in model_v1,
    regs["fc1"] / regs["fc2"] (train_regs) are the keep-scales of drop1 / drop2."""
    h = F.gelu(F.linear(x, sd[p + ".fc1.weight"], sd[p + ".fc1.bias"]))
    if regs is not None and regs.get("fc1") is not None:
        h = h * regs["fc1"].to(h.dtype)
    y = F.linear(h, sd[p + ".fc2.weight"], sd[p + ".fc2.bias"])
    if regs is not None and regs.get("fc2") is not None:
        y = y * regs["fc2"].to(y.dtype)
    return y


def _drop_path(y, dp):
    """timm DropPath with a given per-sample scale dp [B] (0 or 1 / keep)."""
    return y if dp is None else y * dp.to(y.dtype).reshape(-1, 1, 1)


def forward(sd, x, mask=None, training=False, num_heads=6, ln_eps=1e-6, variant="v1", regs=None):
    """MaskedAutoencoderViT.forward (model_v1/model/HTR_VT.py:222-241;
    model_window/model/HTR_VT.py:320-337 in eval mode / dropout disabled).

    `mask`: optional float [T] (1 keep / 0 masked) as produced by draw_span_mask.
    `regs`: optional list of per-block train-mode regulariser dicts (train_regs) injected in timm 1.0.9's places
    (SURVEY.md 13): softmax -> attention dropout -> @ v; proj -> dropout -> DropPath; fc1 -> GELU -> dropout -> fc2 ->
    dropout -> DropPath.  None: no dropout and no DropPath (the arithmetic is then unchanged).
    In train mode BN running statistics in `sd` are updated in place, as the reference does."""
    D = sd["norm.weight"].shape[0]
    x = F.layer_norm(x, x.shape[1:], None, None, 1e-5)                      # :224
    x = stem_forward(sd, x, training)                                       # :225
    b, c = x.shape[0], x.shape[1]
    x = x.reshape(b, c, -1).permute(0, 2, 1)                                # :226-227
    if mask is not None:                                                    # :212-220
        m = mask.to(x.dtype).reshape(1, -1, 1)
        x = x * m + (1 - m) * sd["mask_token"]
    if variant == "v1":
        x = x + sd["pos_embed"]                                             # :231
    depth = 1 + max(int(k.split(".")[1]) for k in sd if k.startswith("blocks."))
    for i in range(depth):                                                  # Block.forward :80-83
        p = f"blocks.{i}"
        win, shift = (0, 0)
        if variant == "window":
            win, shift = ((16, 0), (16, 8), (0, 0), (0, 0))[i] if i < 4 else (0, 0)
        blk = regs[i] if regs is not None else None
        h = F.layer_norm(x, (D,), sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], ln_eps)
        y = _attention(sd, p + ".attn", h, num_heads, win, shift, blk)
        x = x + (y if blk is None else _drop_path(y, blk.get("dp1")))
        h = F.layer_norm(x, (D,), sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], ln_eps)
        y = _mlp(sd, p + ".mlp", h, blk)
        x = x + (y if blk is None else _drop_path(y, blk.get("dp2")))
    x = F.layer_norm(x, (D,), sd["norm.weight"], sd["norm.bias"], ln_eps)   # :236
    x = F.linear(x, sd["head.weight"], sd["head.bias"])                     # :238
    if variant == "v1":
        x = F.layer_norm(x, x.shape[1:], None, None, 1e-5)                  # :239
    return x


# ----------------------------------------------------------------------------------------------
# CTC loss + gradient (float64 restatement of the algorithm behind torch.nn.CTCLoss)
# ----------------------------------------------------------------------------------------------
def _lse(*vals):
    m = max(vals)
    if m == -math.inf:
        return -math.inf
    return m + math.log(sum(math.exp(v - m) for v in vals))


def ctc_loss_grad(logits: np.ndarray, targets: np.ndarray, input_lengths: np.ndarray,
                  target_lengths: np.ndarray, zero_infinity: bool = True):
    """Per-sample negative log likelihood and d(sum_b nll_b)/d(logits) for blank = 0.

    Call-site semantics (model_v1/train.py:21-30, :95): lp = log_softmax(logits); criterion =
    CTCLoss(reduction='none', zero_infinity=True)(lp[T,B,C], targets 1-D concatenated, in_len,
    tgt_len).  Recursion (SURVEY.md 8a): alpha_t(s) = lse(alpha_{t-1}(s), alpha_{t-1}(s-1),
    [alpha_{t-1}(s-2) if l'_s != blank and l'_s != l'_{s-2}]) + lp_t(l'_s); beta symmetric;
    grad_{t,c} = softmax_{t,c} - sum_{s: l'_s=c} exp(alpha_t(s)+beta_t(s)-lp_t(c)+nll) for
    t < input_length, 0 elsewhere.  logits: [B,T,C] float; returns (nll[B], grad[B,T,C]) float64.
    Pure-Python loops: small cases only.
    """
    logits = np.asarray(logits, dtype=np.float64)
    B, T, C = logits.shape
    mx = logits.max(axis=2, keepdims=True)
    lp = logits - (mx + np.log(np.exp(logits - mx).sum(axis=2, keepdims=True)))
    nll = np.zeros(B)
    grad = np.zeros_like(lp)
    off = 0
    NEG = -math.inf
    for b in range(B):
        L = int(target_lengths[b])
        Tb = int(input_lengths[b])
        lab = [int(v) for v in targets[off:off + L]]
        off += L
        S = 2 * L + 1
        ext = [0] * S
        for i, v in enumerate(lab):
            ext[2 * i + 1] = v
        alpha = [[NEG] * S for _ in range(Tb)]
        beta = [[NEG] * S for _ in range(Tb)]
        if Tb > 0:
            alpha[0][0] = lp[b, 0, 0]
            if S > 1:
                alpha[0][1] = lp[b, 0, ext[1]]
        for t in range(1, Tb):
            for s in range(S):
                a = alpha[t - 1][s]
                a1 = alpha[t - 1][s - 1] if s >= 1 else NEG
                a2 = alpha[t - 1][s - 2] if (s >= 2 and ext[s] != 0 and ext[s] != ext[s - 2]) else NEG
                alpha[t][s] = _lse(a, a1, a2) + lp[b, t, ext[s]]
        if Tb > 0:
            ll = _lse(alpha[Tb - 1][S - 1], alpha[Tb - 1][S - 2] if S > 1 else NEG)
        else:
            ll = 0.0 if L == 0 else NEG
        if ll == NEG:
            nll[b] = 0.0 if zero_infinity else math.inf
            continue                                   # zero_infinity: loss 0, grad 0
        nll[b] = -ll
        beta[Tb - 1][S - 1] = lp[b, Tb - 1, ext[S - 1]]
        if S > 1:
            beta[Tb - 1][S - 2] = lp[b, Tb - 1, ext[S - 2]]
        for t in range(Tb - 2, -1, -1):
            for s in range(S):
                v = beta[t + 1][s]
                v1 = beta[t + 1][s + 1] if s + 1 < S else NEG
                v2 = beta[t + 1][s + 2] if (s + 2 < S and ext[s + 2] != 0 and ext[s + 2] != ext[s]) else NEG
                beta[t][s] = _lse(v, v1, v2) + lp[b, t, ext[s]]
        for t in range(Tb):
            post = np.zeros(C)
            for s in range(S):
                ab = alpha[t][s] + beta[t][s]
                if ab > NEG:
                    post[ext[s]] += math.exp(ab - lp[b, t, ext[s]] - ll)
            grad[b, t] = np.exp(lp[b, t]) - post
    return nll, grad


def ctc_loss_torch(logits: torch.Tensor, targets, input_lengths, target_lengths):
    """The call the reference makes (model_v1/train.py:23-29) on CPU tensors: returns per-sample
    nll [B] (float32) with autograd attached to `logits` [B,T,C]."""
    lp = logits.float().permute(1, 0, 2).log_softmax(2)
    return F.ctc_loss(lp, targets, input_lengths, target_lengths, blank=0, reduction="none",
                      zero_infinity=True)


# ----------------------------------------------------------------------------------------------
# Greedy decode
# ----------------------------------------------------------------------------------------------
def greedy_ids(index_flat, lengths, n_character: int):
    """`CTCLabelConverter.decode` (model_v1/utils/utils.py:72-86) up to the id->char lookup:
    keep t[i] iff t[i] != 0, t[i] != t[i-1] (raw previous frame) and t[i] < len(character)."""
    out, pos = [], 0
    idx = [int(v) for v in index_flat]
    for l in [int(v) for v in lengths]:
        t = idx[pos:pos + l]
        out.append([t[i] for i in range(l)
                    if t[i] != 0 and not (i > 0 and t[i - 1] == t[i]) and t[i] < n_character])
        pos += l
    return out


def decode_strings(index_flat, lengths, alphabet: str):
    """Full decode contract: character table is ['[blank]'] + list(alphabet) (utils.py:63)."""
    character = ["[blank]"] + list(alphabet)
    return ["".join(character[i] for i in ids) for ids in greedy_ids(index_flat, lengths, len(character))]


def argmax_first(logits: np.ndarray) -> np.ndarray:
    """torch.max(dim) index semantics used at model_v1/valid.py:40: lowest index among ties,
    a NaN beats every number (first NaN wins) [SURVEY.md 9.17]."""
    a = np.asarray(logits)
    nan = np.isnan(a)
    idx = np.where(nan.any(axis=-1), nan.argmax(axis=-1), np.where(nan, -np.inf, a).argmax(axis=-1))
    return idx.astype(np.int64)


# ----------------------------------------------------------------------------------------------
# Input pipeline (device half) and error rates: SURVEY.md 8(f) rows 2 and 3
# ----------------------------------------------------------------------------------------------
def line_prep_u8(img_u8: np.ndarray, widths=None, eps: float = 1e-5) -> np.ndarray:
    """What reaches the first convolution for a uint8 line batch [B,H,W]: `/ 255.` (dataset.py:44), right padding
    with 1.0 from column widths[b] on (dataset.py:129-130), then the whole-sample LayerNorm of
    model_v1/model/HTR_VT.py:134-136,224 (biased variance, eps 1e-5, no affine)."""
    x = torch.from_numpy(np.ascontiguousarray(img_u8)).float() / 255.
    if widths is not None:
        for b, w in enumerate(widths):
            x[b, :, int(w):] = 1.0
    return F.layer_norm(x, x.shape[1:], eps=eps).numpy()


def levenshtein(a, b) -> int:
    """Unit-cost edit distance of two sequences = `editdistance.eval` (model_v1/valid.py:50,63); the recurrence is
    the one the reference restates at model_v1/test.py:114-133."""
    a, b = list(a), list(b)
    if a == b:
        return 0
    if not a:
        return len(b)
    if not b:
        return len(a)
    prev = list(range(len(b) + 1))
    for i in range(1, len(a) + 1):
        cur = [i]
        for j in range(1, len(b) + 1):
            cur.append(min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (0 if a[i - 1] == b[j - 1] else 1)))
        prev = cur
    return prev[-1]


# (in the reference's non-raw literal `\\(` is an escaped parenthesis: the backslash itself is NOT in the class)
_WER_PUNCT = re.compile(r"""([\[\]{}/()"'&+*=<>?.;:,!\-\u2014_\u20ac#%\u00b0])""")


def format_string_for_wer(s: str) -> str:
    """model_v1/utils/utils.py:176-179: isolate punctuation with spaces, collapse runs of blanks / newlines, strip."""
    s = _WER_PUNCT.sub(r" \1 ", s)
    return re.sub(r"([ \n])+", " ", s).strip()


def error_rates(preds_str, labels):
    """The accumulation of model_v1/valid.py:49-75 for one list of (prediction, label) strings."""
    r = dict(norm_ED=0.0, tot_ED=0, length_of_gt=0, norm_ED_wer=0.0, tot_ED_wer=0, length_of_gt_wer=0)
    for pred, gt in zip(preds_str, labels):
        d = levenshtein(pred, gt)
        r["norm_ED"] += 1 if len(gt) == 0 else d / float(len(gt))
        r["tot_ED"] += d
        r["length_of_gt"] += len(gt)
        pw = format_string_for_wer(pred).split(" ")
        gw = format_string_for_wer(gt).split(" ")
        d = levenshtein(pw, gw)
        r["norm_ED_wer"] += 1 if len(gw) == 0 else d / float(len(gw))
        r["tot_ED_wer"] += d
        r["length_of_gt_wer"] += len(gw)
    r["CER"] = r["tot_ED"] / float(r["length_of_gt"]) if r["length_of_gt"] else 0.0
    r["WER"] = r["tot_ED_wer"] / float(r["length_of_gt_wer"]) if r["length_of_gt_wer"] else 0.0
    return r


# ----------------------------------------------------------------------------------------------
# K-best alignment paths + LM rescoring (model_window/test_with_kenlm.py:25-59)
# ----------------------------------------------------------------------------------------------
def kbest_paths(log_probs: np.ndarray, beam_size: int, acc_dtype=np.float64):
    """`simple_ctc_beam_search_with_lm` up to its collapse step (test_with_kenlm.py:30-51): returns
    [(collapsed id list, path score)] for the surviving beams in the reference's order.
    Per frame the beam_size most probable classes (np.argsort(probs)[-k:][::-1]; a stable sort here, so equal
    values rank by DEscending index) extend every beam; sorted(..., reverse=True) is stable, so among equal scores
    the earlier (beam, class) pair survives.  acc_dtype: the reference's `score + probs[c]` starts from the Python
    float 0.0, which numpy 1.24 (environment.yaml:58) promotes to float64."""
    T = log_probs.shape[0]
    beams = [([], acc_dtype(0.0))]
    for t in range(T):
        probs = log_probs[t]
        top_c = np.argsort(probs, kind="stable")[-beam_size:][::-1]
        new_beams = []
        for seq, score in beams:
            for c in top_c:
                new_beams.append((seq + [int(c)], acc_dtype(score + acc_dtype(probs[c]))))
        beams = sorted(new_beams, key=lambda x: x[1], reverse=True)[:beam_size]
    out = []
    for seq, score in beams:
        text, prev = [], None
        for idx in seq:                                          # :46-51
            if idx != 0 and idx != prev:
                text.append(idx)
            prev = idx
        out.append((text, float(score)))
    return out


def beam_search_with_lm(log_probs: np.ndarray, alphabet: str, lm_score, beam_size: int = 5) -> str:
    """The whole reference function: candidates -> converter.decode (which filters blanks / repeats / ids beyond the
    alphabet AGAIN, utils.py:72-86) -> empty strings dropped -> arg-max of the LM score (:52-59)."""
    cands = []
    for text, score in kbest_paths(log_probs, beam_size):
        s = decode_strings(np.array(text, dtype=np.int64), np.array([len(text)]), alphabet)
        if s and s[0]:
            cands.append((s[0], score))
    if not cands:
        return ""
    lm = [lm_score(c[0]) for c in cands]
    return cands[int(np.argmax(lm))][0]


# ----------------------------------------------------------------------------------------------
# CTC prefix beam search (SURVEY.md 8(f) row 4: the search that replaces the toy per-frame beam of
# model_window/test_with_kenlm.py:25-59).  The reference holds no such function (its beam ranks alignment paths, see
# kbest_paths above), so this restates the published algorithm - Hannun et al., "First-Pass Large Vocabulary Continuous
# Speech Recognition using Bi-Directional Recurrent DNNs", 2014, algorithm 1 without the language-model term - and is
# pinned by `labelling_logprobs_bruteforce` (an enumeration of all C^T alignments): with a beam that holds every prefix
# the search returns the exact posterior of every labelling.  Parity of the CUDA kernel = this function.
# ----------------------------------------------------------------------------------------------
def _lae(a: float, b: float) -> float:
    if a == -math.inf:
        return b
    if b == -math.inf:
        return a
    return max(a, b) + math.log1p(math.exp(-abs(a - b)))


def ctc_prefix_beam_search(log_probs: np.ndarray, beam_size: int):
    """log_probs [T, C] (blank = 0) -> [(label list, log P(labelling | frames))], best first, at most beam_size.
    Beam entry = collapsed prefix with (pb, pnb): log-mass of its alignments ending in blank / in its last label.
    Per frame every entry stays (pb' = tot + lp[0], pnb' = pnb + lp[last]) and is extended by every label c >= 1
    (pnb' = (pb if c == last else tot) + lp[c]); an extension that spells a prefix of the beam adds to that entry.
    Survivors: the beam_size largest lae(pb', pnb'); ties by candidate number - stay entries (rank in the beam) before
    extensions (parent rank, then label)."""
    T, C = log_probs.shape
    K = int(beam_size)
    beam = [((), 0.0, -math.inf)]
    for t in range(T):
        lp = [float(v) for v in log_probs[t]]
        cand = {}                                             # prefix -> [pb', pnb', candidate number]
        for i, (p, pb, pnb) in enumerate(beam):
            tot = _lae(pb, pnb)
            cand[p] = [tot + lp[0], (pnb + lp[p[-1]]) if p else -math.inf, i]
        for i, (p, pb, pnb) in enumerate(beam):
            tot = _lae(pb, pnb)
            for c in range(1, C):
                s = (pb if (p and p[-1] == c) else tot) + lp[c]
                q = p + (c,)
                if q in cand:                                 # q is an entry of the beam (extensions never collide)
                    cand[q][1] = _lae(cand[q][1], s)
                else:
                    cand[q] = [-math.inf, s, K + i * C + c]
        ranked = sorted(((-_lae(v[0], v[1]), v[2], q, v[0], v[1]) for q, v in cand.items()))
        beam = [(q, pb, pnb) for _, _, q, pb, pnb in ranked[:K]]
    return [(list(q), _lae(pb, pnb)) for q, pb, pnb in beam]


def labelling_logprobs_bruteforce(log_probs: np.ndarray):
    """{labelling tuple: log sum of exp(path score) over ALL C^T alignment paths that collapse to it} (small T, C)."""
    import itertools
    T, C = log_probs.shape
    acc = {}
    for path in itertools.product(range(C), repeat=T):
        s = float(sum(float(log_probs[t, c]) for t, c in enumerate(path)))
        lab, prev = [], None
        for c in path:
            if c != 0 and c != prev:
                lab.append(c)
            prev = c
        k = tuple(lab)
        acc[k] = _lae(acc.get(k, -math.inf), s)
    return acc


def prefix_beam_search_with_lm(log_probs: np.ndarray, alphabet: str, lm_score, beam_size: int = 5) -> str:
    """beam_search_with_lm with the prefix search as the candidate generator: labellings -> strings (no second
    repeat filter: a doubled label IS a doubled letter; ids beyond the alphabet dropped), empty strings dropped,
    arg-max of the LM score."""
    table = ["[blank]"] + list(alphabet)
    cands = []
    for lab, _ in ctc_prefix_beam_search(log_probs, beam_size):
        s = "".join(table[i] for i in lab if i < len(table))
        if s:
            cands.append(s)
    if not cands:
        return ""
    lm = [lm_score(c) for c in cands]
    return cands[int(np.argmax(lm))]


# ----------------------------------------------------------------------------------------------
# One training step (loss + parameter gradients), the unit bench.py's reference arm times
# ----------------------------------------------------------------------------------------------
def grad_sample_index(name, numel, n=8192):
    """Reproducible element sample of a gradient tensor for the committed goldens (full gradients are 214 MB; 8192
    elements per tensor estimate a cosine to ~1e-3): sorted indices from a RandomState seeded by the tensor NAME."""
    if numel <= n:
        return np.arange(numel)
    rs = np.random.RandomState(sum((i + 1) * ord(ch) for i, ch in enumerate(name)) % (2 ** 31))
    return np.sort(rs.choice(numel, size=n, replace=False))


def train_step(sd, image, targets, target_lengths, mask, variant="v1", num_heads=6, regs=None):
    """compute_loss + backward (model_v1/train.py:21-30,122-123) with an explicit span mask and optional
    train-mode regularisers (`regs`, see forward / train_regs).
    Returns (loss, {name: grad}) for every floating-point parameter except pos_embed."""
    names = [k for k, v in sd.items() if v.is_floating_point() and "running_" not in k and k != "pos_embed"]
    work = OrderedDict(sd)
    leaves = {}
    for k in names:
        leaves[k] = sd[k].detach().clone().requires_grad_(True)
        work[k] = leaves[k]
    logits = forward(work, image, mask=mask, training=True, num_heads=num_heads, variant=variant, regs=regs)
    B, T = logits.shape[0], logits.shape[1]
    in_len = torch.full((B,), T, dtype=torch.int32)
    loss = ctc_loss_torch(logits, targets, in_len, target_lengths).mean()
    loss.backward()
    for k in sd:                                  # propagate in-place BN buffer updates
        if "running_" in k or k.endswith("num_batches_tracked"):
            sd[k] = work[k]
    return float(loss.detach()), {k: v.grad for k, v in leaves.items()}, logits.detach()


# ----------------------------------------------------------------------------------------------
# Train-mode regularisers of the windowed variant with the CUDA kernels' own masks.  The kernels draw dropout and
# attention dropout from counter-based hashes (htr-vt_b200/csrc/norm.cu dropout_bf16_kernel, csrc/attention2.cu
# attn_keep); the functions below restate that uint32 arithmetic exactly, so a reference can apply the very masks the
# kernels applied and compare values instead of statistics.
# ----------------------------------------------------------------------------------------------
def _mix32(x):
    """murmur3 finaliser on uint32 arrays (wrap-around arithmetic)."""
    x = np.asarray(x, dtype=np.uint32)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint32(16))
        x = x * np.uint32(0x85EBCA6B)
        x = x ^ (x >> np.uint32(13))
        x = x * np.uint32(0xC2B2AE35)
    return x ^ (x >> np.uint32(16))


def _u32(v):
    return np.uint32(int(v) & 0xFFFFFFFF)


def dropout_keep_scale(n, per_sample, p, seed, site, dp=None, offset=0):
    """Per-element factor of htrvt_dropout_bf16(x, n, per_sample, p, seed, site, dp) for the flat elements
    [offset, offset + n): 0 (dropped) or inv_keep * dp[element // per_sample] in float32, inv_keep = 1 / (1 - p).
    Element e sits in 16-byte group i = e // 8, 32-bit word k = (e // 2) % 4 of it; the word's hash
    r = mix32(key + uint32(i) * 4 + k) ^ (i >> 30), key = mix32(uint32(seed) ^ site * 0x9e3779b9) ^ (seed >> 32),
    decides the even element with its low 16 bits and the odd one with its high 16 bits: dropped iff
    (half << 8) < uint32(float32(p) * 2^24)."""
    p32 = np.float32(p)
    thr = np.uint32(int(p32 * np.float32(16777216.0)))
    inv_keep = np.float32(1.0) / (np.float32(1.0) - p32)
    key = _mix32(_u32(seed) ^ _u32(int(site) * 0x9E3779B9)) ^ _u32(int(seed) >> 32)
    e = np.arange(offset, offset + n, dtype=np.int64)
    w = e >> 1                                                   # 32-bit word index = 4 * i + k
    with np.errstate(over="ignore"):
        r = _mix32(key + (w & 0xFFFFFFFF).astype(np.uint32)) ^ ((w >> 2) >> 30).astype(np.uint32)
    half = np.where((e & 1) == 0, r & np.uint32(0xFFFF), r >> np.uint32(16)).astype(np.uint32)
    dropped = (half << np.uint32(8)) < thr
    sc = np.full(n, inv_keep, dtype=np.float32)
    if dp is not None:
        dp = np.asarray(dp, dtype=np.float32)
        sc = inv_keep * dp[e // int(per_sample)]
    return np.where(dropped, np.float32(0.0), sc).astype(np.float32)


def attention_keep(seed, bh, ti, tj, p):
    """attn_keep of csrc/attention2.cu as a bool (True = kept) for broadcastable integer arrays bh (= b * H + h),
    ti (query token), tj (key token): a = mix32(uint32(seed) ^ bh * 0x9e3779b9),
    v = mix32(a ^ mix32((seed >> 32) + ti * 65537 + tj)), dropped iff float32(v >> 8) * 2^-24 < float32(p)."""
    bh, ti, tj = (np.asarray(v, dtype=np.int64) for v in (bh, ti, tj))
    with np.errstate(over="ignore"):
        a = _mix32(_u32(seed) ^ ((bh & 0xFFFFFFFF).astype(np.uint32) * np.uint32(0x9E3779B9)))
        c = _u32(int(seed) >> 32) + (ti & 0xFFFFFFFF).astype(np.uint32) * np.uint32(65537) + \
            (tj & 0xFFFFFFFF).astype(np.uint32)
    v = _mix32(a ^ _mix32(c))
    u = (v >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return ~(u < np.float32(p))


def window_blocks(depth):
    """(window, shift) per block of the windowed variant: 16-token windows in block 0, shifted by 8 in block 1,
    global attention in the rest (as forward above and the model's engine use them)."""
    return [((16, 0) if i == 0 else ((16, 8) if i == 1 else (0, 0))) for i in range(depth)]


def train_regs(seed, drop, attn_drop, drop_path, B, T, D, hidden, num_heads):
    """The per-block `regs` of forward / train_step for one train-mode step of the windowed variant's engine
    (htr-vt_b200/engine.py), from the draw the model made for it (model_window HTR_VT._train_rng: seed, rates, and
    drop_path = [(dp1, dp2) per block], tensors [B] or None).  Block i uses attention seed seed + 16 i and dropout
    sites 8 i + 1 (proj, DropPath dp1), 8 i + 2 (fc1 activation), 8 i + 3 (fc2, DropPath dp2) over the token-major
    [B, T, features] tensors.  Entries: "attn" [B, H, Tp, Tp] keep-scale over token indices (Tp = T padded to the
    window in windowed blocks), "proj" / "fc2" [B, T, D], "fc1" [B, T, hidden] (DropPath folded out: the dropout
    factors alone), "dp1" / "dp2" [B] - each None where that regulariser is off."""
    regs = []
    for i, (window, shift) in enumerate(window_blocks(len(drop_path))):
        blk = {"attn": None, "proj": None, "fc1": None, "fc2": None}
        if attn_drop > 0:
            Tp = -(-T // window) * window if window else T
            bh = np.arange(B * num_heads).reshape(B, num_heads, 1, 1)
            t = np.arange(Tp)
            keep = attention_keep(seed + 16 * i, bh, t.reshape(1, 1, Tp, 1), t.reshape(1, 1, 1, Tp), attn_drop)
            inv = np.float32(1.0) / (np.float32(1.0) - np.float32(attn_drop))
            blk["attn"] = torch.from_numpy(np.where(keep, inv, np.float32(0.0)).astype(np.float32))
        if drop > 0:
            for name, site, width in (("proj", 8 * i + 1, D), ("fc1", 8 * i + 2, hidden), ("fc2", 8 * i + 3, D)):
                blk[name] = torch.from_numpy(
                    dropout_keep_scale(B * T * width, T * width, drop, seed, site).reshape(B, T, width))
        dp1, dp2 = drop_path[i]
        blk["dp1"] = None if dp1 is None else torch.as_tensor(dp1).detach().float().cpu()
        blk["dp2"] = None if dp2 is None else torch.as_tensor(dp2).detach().float().cpu()
        regs.append(blk)
    return regs
