"""GPU parity of the whole drop-in path (create_model -> forward -> CTC loss -> backward -> decode) against
the CPU oracle and the committed goldens generated from the unmodified reference."""
import os
from importlib import import_module

import numpy as np
import pytest
import torch

import htrvt_oracle as O

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def _images(seed, B, W):
    return torch.from_numpy(np.random.RandomState(seed).rand(B, 1, 64, W).astype(np.float32))


def _labels(seed, B, C, lo, hi):
    rs = np.random.RandomState(seed)
    lens = rs.randint(lo, hi + 1, size=B).astype(np.int32)
    tg = rs.randint(1, C, size=int(lens.sum())).astype(np.int32)
    return torch.from_numpy(tg), torch.from_numpy(lens)


def _mod():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200.model.HTR_VT")


def _relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-12))


def _build(nb_cls, W, D, depth, heads, seed):
    H = _mod()
    from functools import partial
    m = H.MaskedAutoencoderViT(nb_cls, img_size=[64, W], patch_size=(4, 64), embed_dim=D, depth=depth,
                               num_heads=heads, mlp_ratio=4, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))
    sd = O.init_state_dict(nb_cls, [64, W], seed=seed, embed_dim=D, depth=depth, num_heads=heads)
    m.load_state_dict(sd, strict=True)
    return m.cuda(), sd


@pytest.mark.parametrize("cfg", [dict(nb_cls=24, W=128, D=256, depth=2, heads=2, B=3, seed=5),
                                 dict(nb_cls=80, W=512, D=768, depth=4, heads=6, B=2, seed=123)])
def test_eval_logits_match_oracle(cfg):
    m, sd = _build(cfg["nb_cls"], cfg["W"], cfg["D"], cfg["depth"], cfg["heads"], cfg["seed"])
    m.eval()
    x = _images(cfg["seed"] + 1, cfg["B"], cfg["W"])
    with torch.no_grad():
        got = m(x.cuda()).float().cpu().numpy()
        want = O.forward(sd, x, training=False, num_heads=cfg["heads"]).numpy()
    if cfg["D"] == 768:
        g = np.load(os.path.join(G, "v1_full.npz"))
        np.testing.assert_allclose(want, g["logits_eval"], atol=2e-4)      # oracle == reference (pinned)
        want = g["logits_eval"]
    # north_star tolerance for the bf16 path: 2e-2 relative
    assert _relerr(got, want) < 2e-2, _relerr(got, want)
    # greedy decode of both logits agrees except where the reference's own top-2 margin is below the tolerance
    am_got, am_want = got.argmax(-1), want.argmax(-1)
    top2 = np.sort(want, axis=-1)[..., -2:]
    margin = top2[..., 1] - top2[..., 0]
    assert ((am_got == am_want) | (margin < 4e-2 * np.abs(want).max())).all()


def test_backward_through_eval_forward_refuses_before_writing_gradients():
    """The BatchNorm backward kernels differentiate through batch statistics: a backward after model.eval() must fail
    loudly and must not leave partial gradients behind (INTEGRATION.md, limits)."""
    ops = import_module("htr-vt_b200.ops")
    m, _ = _build(24, 128, 256, 2, 2, 5)
    m.eval()
    out = m(_images(6, 3, 128).cuda()).float()
    with pytest.raises(ops.HtrvtError, match="train-mode forward"):
        out.sum().backward()
    assert all(p.grad is None or float(p.grad.abs().max()) == 0.0 for p in m.parameters())


@pytest.mark.parametrize("cfg", [dict(nb_cls=24, W=128, D=256, depth=2, heads=2, B=3, seed=5),
                                 dict(nb_cls=80, W=512, D=768, depth=4, heads=6, B=2, seed=123)])
def test_train_step_matches_oracle(cfg):
    import htrvt_b200 as h
    m, sd = _build(cfg["nb_cls"], cfg["W"], cfg["D"], cfg["depth"], cfg["heads"], cfg["seed"])
    m.train()
    B, W = cfg["B"], cfg["W"]
    x = _images(cfg["seed"] + 1, B, W)
    tg, tl = _labels(cfg["seed"] + 2, B, cfg["nb_cls"], 4, 12)
    torch.manual_seed(7)
    preds = m(x.cuda(), 0.4, 8, use_masking=True)
    preds_f = preds.float()
    lp = preds_f.permute(1, 0, 2).log_softmax(2)
    crit = h.CTCLoss(reduction="none", zero_infinity=True).to("cuda")
    loss = crit(lp, tg.cuda(), torch.IntTensor([preds.size(1)] * B).cuda(), tl.cuda()).mean()
    loss.backward()
    torch.manual_seed(7)
    mask = O.draw_span_mask(W // 4, 0.4, 8)
    sd_ref = {k: v.clone() for k, v in sd.items()}
    ref_loss, ref_grads, ref_logits = O.train_step(sd_ref, x, tg, tl, mask, num_heads=cfg["heads"])
    if cfg["D"] == 768:
        g = np.load(os.path.join(G, "v1_full.npz"))
        np.testing.assert_allclose(ref_logits.numpy(), g["logits_train"], atol=3e-4)
        assert abs(ref_loss - float(g["loss"])) < 1e-4 * abs(float(g["loss"]))
    # north_star bound for 16-bit operands, no calibration against a library path (the forward stem is fp16: a
    # bf16-only stem sits at 3-4e-2 here, DESIGN.md 4)
    err = _relerr(preds.detach().cpu().numpy(), ref_logits.numpy())
    assert err < 2e-2, err
    assert abs(loss.item() - ref_loss) < 2e-2 * abs(ref_loss)
    # BN running statistics and counters updated in place, as nn.BatchNorm2d does
    msd = m.state_dict()
    assert int(msd["patch_embed.bn1.num_batches_tracked"]) == 1
    assert _relerr(msd["patch_embed.bn1.running_mean"].cpu().numpy(), sd_ref["patch_embed.bn1.running_mean"].numpy()) < 2e-2
    assert _relerr(msd["patch_embed.layer3.1.bn2.running_var"].cpu().numpy(),
                   sd_ref["patch_embed.layer3.1.bn2.running_var"].numpy()) < 2e-2
    # every trainable parameter gets a gradient close to the fp32 reference's (bf16 operands: cosine + norm)
    bad = []
    for name, p in m.named_parameters():
        if name == "pos_embed":
            assert p.grad is None
            continue
        assert p.grad is not None, name
        a = p.grad.detach().float().cpu().double().reshape(-1)
        b = ref_grads[name].double().reshape(-1)
        cos = float((a @ b) / (a.norm() * b.norm() + 1e-30))
        ratio = float(a.norm() / (b.norm() + 1e-30))
        # tiny batches (B = 2 / 3): batch statistics amplify bf16 noise in the stem, so the stem bound is looser here;
        # test_train_batch32_vs_reference_golden holds the tight per-family bounds at a well-conditioned batch
        lo_cos, tol = (0.99, 0.05) if _family(name) == "transformer" else (0.93, 0.10)
        if not (cos > lo_cos and abs(ratio - 1.0) < tol):
            bad.append((name, round(cos, 4), round(ratio, 4)))
    assert not bad, bad


def test_side_stream_weight_gradients_equal_single_stream():
    """engine.WGRAD_STREAM: weight-gradient GEMMs (and the steady-state weight re-pack) on a second stream.  Same
    kernels, same inputs: every gradient must equal the single-stream schedule's up to the split-K reduce-add order
    (fp32 atomics), over several steps so that the in-place re-pack path and buffer reuse are exercised."""
    import htrvt_b200 as h
    eng = import_module("htr-vt_b200.engine")
    cfg = dict(nb_cls=80, W=512, D=768, depth=4, heads=6, B=4, seed=31)
    x = _images(cfg["seed"] + 1, cfg["B"], cfg["W"]).cuda()
    tg, tl = _labels(cfg["seed"] + 2, cfg["B"], cfg["nb_cls"], 4, 12)
    crit = h.CTCLoss(reduction="none", zero_infinity=True).to("cuda")
    out = []
    old = eng.WGRAD_STREAM
    try:
        for flag in (False, False, True):
            eng.WGRAD_STREAM = flag
            m, _ = _build(cfg["nb_cls"], cfg["W"], cfg["D"], cfg["depth"], cfg["heads"], cfg["seed"])
            m.train()
            for it in range(3):
                for p in m.parameters():
                    p.grad = None
                torch.manual_seed(7 + it)
                preds = m(x, 0.4, 8, use_masking=True).float()
                lp = preds.permute(1, 0, 2).log_softmax(2)
                loss = crit(lp, tg.cuda(), torch.IntTensor([preds.size(1)] * cfg["B"]).cuda(), tl.cuda()).mean()
                loss.backward()
            torch.cuda.synchronize()
            out.append((preds.detach().clone(), {n: p.grad.detach().double() for n, p in m.named_parameters()
                                                 if p.grad is not None}))
    finally:
        eng.WGRAD_STREAM = old
    (l0, g0), (l0b, g0b), (l1, g1) = out
    assert torch.equal(l0, l1) and torch.equal(l0, l0b)                  # the forward (incl. the re-pack) is identical
    assert g0.keys() == g1.keys() and len(g0) > 50
    # noise floor: two IDENTICAL single-stream runs differ (free summation order of split-K slices and BatchNorm sums)
    den = sum(float((g0[n] ** 2).sum()) for n in g0)
    noise = (sum(float(((g0[n] - g0b[n]) ** 2).sum()) for n in g0) / den) ** 0.5
    diff = (sum(float(((g0[n] - g1[n]) ** 2).sum()) for n in g0) / den) ** 0.5
    # (a missing dependency between the streams reads stale or half-written tensors: O(1) errors; the floor covers a box
    # on which two single-stream runs happen to sum in the same order)
    assert diff <= 4.0 * noise + 2e-3, (diff, noise)
    for n in g0:
        a, b = g0[n].reshape(-1), g1[n].reshape(-1)
        cos = float(a @ b / (a.norm() * b.norm() + 1e-30))
        assert cos > 0.999, (n, cos)


def _family(name):
    """Tensor classes of the gradient check: stem convolution / BatchNorm tensors vs transformer tensors."""
    return "stem" if name.startswith("patch_embed.") else "transformer"


def test_train_batch32_vs_reference_golden():
    """VERDICT r1 items 1a / 1b: train mode at a batch where BatchNorm batch statistics are well conditioned (B = 32,
    full architecture) against the committed output of the UNMODIFIED reference (oracle/make_golden.py
    train_batch_case, model_v1/train.py:21-30): logits within the north-star bf16 bound of 2e-2 with no calibration
    escape hatch, loss within 1 %, and per-tensor-class gradient bounds on all 101 trainable tensors."""
    import htrvt_b200 as h
    g = np.load(os.path.join(G, "v1_train_b32.npz"))
    nb_cls, W, B, seed, train_seed = [int(v) for v in g["meta"]]
    m, sd = _build(nb_cls, W, 768, 4, 6, seed)
    m.train()
    x = _images(seed + 1, B, W)
    tg, tl = _labels(seed + 2, B, nb_cls, 16, 64)
    torch.manual_seed(train_seed)
    preds = m(x.cuda(), 0.4, 8, use_masking=True)
    lp = preds.float().permute(1, 0, 2).log_softmax(2)
    crit = h.CTCLoss(reduction="none", zero_infinity=True).to("cuda")
    nll = crit(lp, tg.cuda(), torch.IntTensor([preds.size(1)] * B).cuda(), tl.cuda())
    loss = nll.mean()
    loss.backward()
    err = _relerr(preds.detach().float().cpu().numpy(), g["logits_train"])
    assert err < 2e-2, err
    assert abs(loss.item() - float(g["loss"])) < 1e-2 * abs(float(g["loss"]))
    np.testing.assert_allclose(nll.detach().cpu().numpy(), g["nll"], rtol=3e-2)
    offs = np.concatenate([[0], np.cumsum(g["grad_sample_counts"])])
    where = {n: i for i, n in enumerate(g["grad_names"].tolist())}

    def ref_of(name, a):
        i = where[name]
        return torch.from_numpy(g["grad_samples"][offs[i]:offs[i + 1]]).double(), float(g["grad_norms"][i])

    named = []
    for name, p in m.named_parameters():
        if name == "pos_embed":
            assert p.grad is None
            continue
        assert p.grad is not None, name
        named.append((name, p.grad.detach().float().cpu()))
    assert len(named) == 101

    # sampled cosine (8192 reproducible elements per tensor) + exact norm ratio against the reference's full norm
    bad = []
    for name, a in named:
        i = where[name]
        idx = torch.from_numpy(O.grad_sample_index(name, a.numel()))
        a_s = a.reshape(-1)[idx].double()
        b_s, bnorm = ref_of(name, a)
        cos = float((a_s @ b_s) / (a_s.norm() * b_s.norm() + 1e-30))
        ratio = float(a.double().norm() / (bnorm + 1e-30))
        lo_cos, tol = (0.995, 0.03) if _family(name) == "transformer" else (0.98, 0.05)
        if not (cos >= lo_cos and abs(ratio - 1.0) <= tol):
            bad.append((name, round(cos, 4), round(ratio, 4)))
    assert not bad, bad
    msd = m.state_dict()
    got_bn = np.concatenate([msd[k].float().cpu().numpy().reshape(-1) for k in msd if "running_" in k])
    assert _relerr(got_bn, g["bn_running"]) < 1e-2


def test_stem_gradients_match_finite_differences_of_the_oracle():
    """Finite differences of the ORACLE's float64 loss (float64 forward + the float64 CTC restatement: no autograd
    anywhere) along OUR gradient's direction, for directions confined to (a) the fused stem head's tensors (conv1 /
    bn1: stem_head_bwd), (b) every other BatchNorm's affine parameters (bn_bwd) and (c) the stem convolutions.
    With d = g_ours / |g_ours| the derivative of the true loss along d is |g_true| cos(g_ours, g_true), so
    FD / |g_ours| = cos x (norm ratio): a dropped or mis-scaled term in a backward kernel shows up here."""
    import htrvt_b200 as h
    cfg = dict(nb_cls=24, W=128, D=256, depth=1, heads=2, B=8, seed=15)
    m, sd = _build(cfg["nb_cls"], cfg["W"], cfg["D"], cfg["depth"], cfg["heads"], cfg["seed"])
    m.train()
    B, W = cfg["B"], cfg["W"]
    x = _images(cfg["seed"] + 1, B, W)
    tg, tl = _labels(cfg["seed"] + 2, B, cfg["nb_cls"], 4, 12)
    preds = m(x.cuda())                                        # no span mask: a deterministic function of the weights
    loss = h.ctc_loss_from_logits(preds.float(), tg.cuda(), tl).mean()
    loss.backward()
    grads = {n: p.grad.detach().double().cpu() for n, p in m.named_parameters() if p.grad is not None}

    def oracle_loss(sd64):
        with torch.no_grad():
            lg = O.forward({k: v.clone() for k, v in sd64.items()}, x.double(), training=True, num_heads=cfg["heads"])
        nll, _ = O.ctc_loss_grad(lg.numpy(), tg.numpy(), np.full(B, lg.shape[1]), tl.numpy())
        return float(np.mean(nll))

    sd64 = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in sd.items()}
    assert abs(oracle_loss(sd64) - loss.item()) < 2e-2 * abs(loss.item())
    groups = {
        "stem_head": [k for k in grads if k in ("patch_embed.conv1.weight", "patch_embed.bn1.weight", "patch_embed.bn1.bias")],
        "bn_affine": [k for k in grads if k.startswith("patch_embed.layer") and (".bn" in k or ".downsample.1." in k)],
        "stem_convs": [k for k in grads if k.startswith("patch_embed.layer") and k.endswith(".weight") and ".conv" in k],
    }
    for gname, names in groups.items():
        assert names, gname
        gnorm = sum(float((grads[k] ** 2).sum()) for k in names) ** 0.5
        wnorm = sum(float((sd64[k] ** 2).sum()) for k in names) ** 0.5
        step = 1e-5 * wnorm                                   # a 1e-5 relative move of the group's weights
        plus, minus = dict(sd64), dict(sd64)
        for k in names:
            plus[k] = sd64[k] + step * grads[k] / gnorm
            minus[k] = sd64[k] - step * grads[k] / gnorm
        fd = (oracle_loss(plus) - oracle_loss(minus)) / (2 * step)
        assert 0.95 <= fd / gnorm <= 1.03, (gname, fd, gnorm)


def test_end_to_end_decode_strings():
    import htrvt_b200 as h
    m, sd = _build(80, 512, 768, 4, 6, 123)
    m.eval()
    x = _images(124, 2, 512)
    alphabet = "".join(chr(33 + i) for i in range(79))
    conv = h.CTCLabelConverter(alphabet)
    with torch.no_grad():
        preds = m(x.cuda()).float()
        lp = preds.permute(1, 0, 2).log_softmax(2)
        _, idx = lp.max(2)
        idx = idx.transpose(1, 0).contiguous().view(-1)
        got = conv.decode(idx.data, torch.IntTensor([preds.size(1)] * 2))
        fused = conv.decode_logits(preds)
    assert got == fused
    # bit-exact against the oracle decode of the SAME logits (kernel-level exactness)
    want = O.decode_strings(O.argmax_first(preds.cpu().numpy()).reshape(-1), [preds.size(1)] * 2, alphabet)
    assert got == want


# ------------------------------------------------------------------------------------------------
# windowed variant (model_window): relative-position bias, 16-token shifted windows, T up to 256
# ------------------------------------------------------------------------------------------------
def _build_window(nb_cls, W, D, depth, heads, seed, table_size_from_w=False):
    """table_size_from_w: size the bias table for exactly W / 4 tokens (img_size = [W, 64], the convention of
    create_model), which a line whose token count is not a multiple of 16 needs to load init_state_dict's weights."""
    import htrvt_b200  # noqa: F401
    from functools import partial
    Wm = import_module("htr-vt_b200.model_window.HTR_VT")
    m = Wm.MaskedAutoencoderViT(nb_cls, img_size=[W, 64] if table_size_from_w else [64, W], patch_size=(4, 64),
                                embed_dim=D, depth=depth, num_heads=heads, mlp_ratio=4,
                                norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))
    sd = O.init_state_dict(nb_cls, [64, W], seed=seed, embed_dim=D, depth=depth, num_heads=heads, variant="window")
    m.load_state_dict(sd, strict=True)
    return m.cuda(), sd


def test_window_eval_logits_match_reference_golden():
    g = np.load(os.path.join(G, "win_full.npz"), allow_pickle=True)
    nb_cls, W, B, seed, D, depth, heads, _ = [int(v) for v in g["meta"]]
    m, sd = _build_window(nb_cls, W, D, depth, heads, seed)
    assert [str(k) for k in g["keys"]] == list(m.state_dict().keys())          # reference key order
    m.eval()
    x = _images(seed + 1, B, W)
    with torch.no_grad():
        got = m(x.cuda()).float().cpu().numpy()
        want = O.forward(sd, x, training=False, num_heads=heads, variant="window").numpy()
    np.testing.assert_allclose(want, g["logits_eval"], atol=3e-4)              # oracle == reference (pinned)
    assert got.shape == g["logits_eval"].shape == (B, W // 4, nb_cls)
    assert _relerr(got, g["logits_eval"]) < 2e-2, _relerr(got, g["logits_eval"])


@pytest.mark.parametrize("tag", ["win_w1000", "win_w600"])
def test_window_ragged_widths_match_reference_golden(tag):
    """Line widths whose token count is not a multiple of the 16-token window (T = 250 / 150): the reference pads, rolls
    the key-padding mask and strips the pad (model_window/model/HTR_VT.py:121-131, 49-56); goldens from the unmodified
    reference (oracle/make_golden.py window_ragged_case).  Eval logits + a train step's gradients vs the oracle."""
    import htrvt_b200 as h
    g = np.load(os.path.join(G, tag + ".npz"))
    nb_cls, W, B, seed = [int(v) for v in g["meta"]]
    Wm = import_module("htr-vt_b200.model_window.HTR_VT")
    m = Wm.create_model(nb_cls, [W, 64])                 # the reference's convention for this variant: img_size = [W, H]
    sd = O.init_state_dict(nb_cls, [64, W], seed=seed, variant="window")
    m.load_state_dict(sd, strict=True)
    m = m.cuda()
    assert [str(k) for k in g["keys"]] == list(m.state_dict().keys())
    m.eval()
    x = _images(seed + 1, B, W)
    with torch.no_grad():
        got = m(x.cuda()).float().cpu().numpy()
    assert got.shape == g["logits_eval"].shape == (B, W // 4, nb_cls) and (W // 4) % 16 != 0
    assert _relerr(got, g["logits_eval"]) < 2e-2, _relerr(got, g["logits_eval"])
    # backward through the padded / masked windows
    m.train().set_stochastic(0.0, 0.0, 0.0)
    tg, tl = _labels(seed + 2, B, nb_cls, 4, 40)
    torch.manual_seed(7)
    preds = m(x.cuda(), 0.4, 8, use_masking=True)
    h.ctc_loss_from_logits(preds.float(), tg.cuda(), tl).mean().backward()
    torch.manual_seed(7)
    mask = O.draw_span_mask(W // 4, 0.4, 8)
    ref_loss, ref_grads, ref_logits = O.train_step({k: v.clone() for k, v in sd.items()}, x, tg, tl, mask,
                                                   variant="window", num_heads=6)
    assert _relerr(preds.detach().float().cpu().numpy(), ref_logits.numpy()) < 2e-2
    bad = []
    for name, p in m.named_parameters():
        a = p.grad.detach().float().cpu().double().reshape(-1)
        b = ref_grads[name].double().reshape(-1)
        cos = float((a @ b) / (a.norm() * b.norm() + 1e-30))
        if not cos > (0.99 if _family(name) == "transformer" else 0.93):
            bad.append((name, round(cos, 4)))
    assert not bad, bad


def _capture_draws(m):
    """Record every train-mode draw (seed, rates, DropPath scales) the model makes, by wrapping its _train_rng."""
    draws = []
    orig = m._train_rng

    def capture(batch, device):
        rng = orig(batch, device)
        draws.append(rng)
        return rng

    m._train_rng = capture
    return draws


def _regs_of(draw, B, T, D, heads):
    """Oracle regs (htrvt_oracle.train_regs) for the masks the engine applied in the step that made `draw`."""
    if draw is None:
        return None
    return O.train_regs(draw["seed"], draw["drop"], draw["attn_drop"], draw["drop_path"], B, T, D, 4 * D, heads)


@pytest.mark.parametrize("cfg", [
    dict(nb_cls=20, W=512, D=256, depth=4, heads=2, B=3, seed=9),
    dict(nb_cls=90, W=1024, D=768, depth=4, heads=6, B=2, seed=321),
    # train-mode regularisers on (rates = drop, attn_drop, drop_path_rate), compared with the oracle applying the masks
    # the kernels applied; depth 4 covers blocks 0 (window 16, shift 0), 1 (16, 8) and 2-3 (global)
    pytest.param(dict(nb_cls=90, W=1024, D=768, depth=4, heads=6, B=2, seed=321, rates=(0.1, 0.05, 0.1)),
                 id="defaults"),
    pytest.param(dict(nb_cls=20, W=512, D=256, depth=4, heads=2, B=3, seed=9, rates=(0.1, 0.0, 0.0)),
                 id="drop_only"),
    pytest.param(dict(nb_cls=20, W=512, D=256, depth=4, heads=2, B=3, seed=9, rates=(0.0, 0.05, 0.0)),
                 id="attn_drop_only"),
    pytest.param(dict(nb_cls=20, W=512, D=256, depth=4, heads=2, B=4, seed=9, rates=(0.0, 0.0, 0.5)),
                 id="drop_path_only"),
    pytest.param(dict(nb_cls=40, W=1000, D=256, depth=4, heads=2, B=3, seed=19, rates=(0.1, 0.05, 0.1)),
                 id="ragged_w1000_defaults"),
])
def test_window_train_step_matches_oracle(cfg):
    """Train-mode forward/backward against the oracle.  With the regularisers off (the first two configs) the step is
    deterministic.  With them on, the reference draws its masks from the device generator, so only the distribution
    could match it (SURVEY.md 9.13); here the oracle applies the kernels' own masks (train_regs: the same seed, sites
    and DropPath draw), which makes the comparison value by value again."""
    import htrvt_b200 as h
    rates = cfg.get("rates", (0.0, 0.0, 0.0))
    B, W, D, heads = cfg["B"], cfg["W"], cfg["D"], cfg["heads"]
    T = W // 4
    m, sd = _build_window(cfg["nb_cls"], W, D, cfg["depth"], heads, cfg["seed"], table_size_from_w=T % 16 != 0)
    m.train().set_stochastic(*rates)
    draws = _capture_draws(m)
    x = _images(cfg["seed"] + 1, B, W)
    tg, tl = _labels(cfg["seed"] + 2, B, cfg["nb_cls"], 4, 40)
    torch.manual_seed(7)
    preds = m(x.cuda(), 0.4, 8, use_masking=True)
    loss = h.ctc_loss_from_logits(preds.float(), tg.cuda(), tl).mean()
    loss.backward()
    assert len(draws) == 1
    regs = _regs_of(draws[0], B, T, D, heads)
    drop, attn_drop, dpr = rates
    if regs is None:
        assert rates == (0.0, 0.0, 0.0)
    else:
        # the draw exercises what the config targets
        assert draws[0]["drop"] == drop and draws[0]["attn_drop"] == attn_drop
        for blk in regs:
            for name in ("proj", "fc1", "fc2"):
                assert (blk[name] is not None) == (drop > 0)
                if drop > 0:
                    assert (blk[name] == 0).any() and (blk[name] > 1).any()
            assert (blk["attn"] is not None) == (attn_drop > 0)
            if attn_drop > 0:
                assert (blk["attn"] == 0).any()
        if dpr > 0:
            dps = [d for blk in regs for d in (blk["dp1"], blk["dp2"]) if d is not None]
            assert len(dps) == 2 * (cfg["depth"] - 1)
            assert any((d == 0).any() for d in dps)                         # some sample loses a branch
        if dpr >= 0.5:
            assert any(not torch.equal(blk["dp1"], blk["dp2"]) for blk in regs if blk["dp1"] is not None)
    torch.manual_seed(7)
    mask = O.draw_span_mask(T, 0.4, 8)
    sd_ref = {k: v.clone() for k, v in sd.items()}
    ref_loss, ref_grads, ref_logits = O.train_step(sd_ref, x, tg, tl, mask, variant="window", num_heads=heads,
                                                   regs=regs)
    err = _relerr(preds.detach().cpu().numpy(), ref_logits.numpy())
    assert err < 2e-2, err
    assert abs(loss.item() - ref_loss) < 2e-2 * abs(ref_loss)
    bad = []
    for name, p in m.named_parameters():
        assert p.grad is not None, name
        a = p.grad.detach().float().cpu().double().reshape(-1)
        b = ref_grads[name].double().reshape(-1)
        if float(b.norm()) == 0.0:           # a branch DropPath removed for every sample: no gradient at all
            if float(a.abs().max()) != 0.0:
                bad.append((name, "want 0", float(a.abs().max())))
            continue
        cos = float((a @ b) / (a.norm() * b.norm() + 1e-30))
        ratio = float(a.norm() / (b.norm() + 1e-30))
        # tiny batches (B = 2 / 3): batch statistics amplify bf16 noise in the stem, so the stem bound is looser here;
        # test_train_batch32_vs_reference_golden holds the tight per-family bounds at a well-conditioned batch
        lo_cos, tol = (0.99, 0.05) if _family(name) == "transformer" else (0.93, 0.10)
        if not (cos > lo_cos and abs(ratio - 1.0) < tol):
            bad.append((name, round(cos, 4), round(ratio, 4)))
    assert not bad, bad


def test_window_drop_path_rate_one_removes_the_last_block():
    """set_stochastic(drop_path_rate=1.0): the last block's DropPath keeps no sample.  Its scales are 0 (as timm's
    DropPath, which skips the division by keep = 0), so the logits stay finite, the block's parameters get exactly
    zero gradient, and the step matches the oracle with the captured DropPath draw."""
    import htrvt_b200 as h
    nb_cls, W, D, heads, B = 20, 512, 256, 2, 3
    m, sd = _build_window(nb_cls, W, D, 4, heads, 9)
    m.train().set_stochastic(0.0, 0.0, 1.0)
    draws = _capture_draws(m)
    x = _images(10, B, W)
    tg, tl = _labels(11, B, nb_cls, 4, 40)
    torch.manual_seed(7)
    preds = m(x.cuda(), 0.4, 8, use_masking=True)
    assert torch.isfinite(preds).all()
    h.ctc_loss_from_logits(preds.float(), tg.cuda(), tl).mean().backward()
    dp1, dp2 = draws[0]["drop_path"][-1]
    assert not dp1.any() and not dp2.any()
    for name, p in m.named_parameters():
        if name.startswith("blocks.3."):
            assert not p.grad.any(), name
    assert m.head.weight.grad.abs().max() > 0 and m.blocks[0].mlp.fc1.weight.grad.abs().max() > 0
    torch.manual_seed(7)
    mask = O.draw_span_mask(W // 4, 0.4, 8)
    regs = _regs_of(draws[0], B, W // 4, D, heads)
    _, _, ref_logits = O.train_step({k: v.clone() for k, v in sd.items()}, x, tg, tl, mask, variant="window",
                                    num_heads=heads, regs=regs)
    assert _relerr(preds.detach().cpu().numpy(), ref_logits.numpy()) < 2e-2


def test_window_train_mode_is_stochastic_and_seeded():
    import htrvt_b200 as h
    m, sd = _build_window(90, 512, 768, 4, 6, 11)
    m.train()
    x = _images(12, 4, 512).cuda()
    tg, tl = _labels(13, 4, 90, 4, 30)

    def run(seed):
        torch.manual_seed(seed)
        for p in m.parameters():
            p.grad = None
        preds = m(x, 0.4, 8, use_masking=True)
        loss = h.ctc_loss_from_logits(preds.float(), tg.cuda(), tl).mean()
        loss.backward()
        return preds.detach().clone(), m.head.weight.grad.detach().clone()

    a, ga = run(3)
    b, gb = run(3)
    c, _ = run(4)
    assert torch.equal(a, b)                                    # same seed: same masks in the forward ...
    # ... and in the backward (split-K slices reduce-add in a free order: equal up to fp32 summation order)
    assert float((ga - gb).abs().max()) <= 1e-5 * float(ga.abs().max())
    assert not torch.equal(a, c)
    assert torch.isfinite(a).all() and torch.isfinite(ga).all()
    m.eval()
    with torch.no_grad():
        e1, e2 = m(x), m(x)
    assert torch.equal(e1, e2)
    # inverted dropout keeps the expectation: with the regularisers off the SAME train-mode graph (same span mask,
    # batch statistics) gives logits the dropout run scatters around
    m.train().set_stochastic(0.0, 0.0, 0.0)
    d, _ = run(3)
    assert float((a.float() - d.float()).abs().mean()) < 0.6 * float(d.float().abs().mean())
    assert float((a.float() - d.float()).abs().mean()) > 1e-3
