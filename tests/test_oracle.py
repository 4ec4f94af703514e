"""Pin the CPU oracle (oracle/htrvt_oracle.py) to fixtures generated from the unmodified reference
(oracle/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest
import torch

import htrvt_oracle as O

G = os.path.join(os.path.dirname(__file__), "golden")


def _images(seed, B, W):
    return torch.from_numpy(np.random.RandomState(seed).rand(B, 1, 64, W).astype(np.float32))


def _labels(seed, B, C, lo, hi):
    rs = np.random.RandomState(seed)
    lens = rs.randint(lo, hi + 1, size=B).astype(np.int32)
    tg = rs.randint(1, C, size=int(lens.sum())).astype(np.int32)
    return torch.from_numpy(tg), torch.from_numpy(lens)


@pytest.mark.parametrize("tag,variant", [("v1_small", "v1"), ("v1_full", "v1"),
                                         ("win_small", "window"), ("win_full", "window")])
def test_forward_eval_matches_reference(tag, variant):
    g = np.load(os.path.join(G, tag + ".npz"))
    nb_cls, W, B, seed, D, depth, heads, _ = [int(v) for v in g["meta"]]
    sd = O.init_state_dict(nb_cls, [64, W], seed=seed, embed_dim=D, depth=depth, num_heads=heads, variant=variant)
    assert sorted(sd.keys()) == sorted(g["keys"].tolist())
    with torch.no_grad():
        y = O.forward(sd, _images(seed + 1, B, W), training=False, num_heads=heads, variant=variant)
    np.testing.assert_allclose(y.numpy(), g["logits_eval"], rtol=0, atol=2e-4)


@pytest.mark.parametrize("tag", ["v1_small", "v1_full"])
def test_train_step_matches_reference(tag):
    g = np.load(os.path.join(G, tag + ".npz"))
    nb_cls, W, B, seed, D, depth, heads, train_seed = [int(v) for v in g["meta"]]
    sd = O.init_state_dict(nb_cls, [64, W], seed=seed, embed_dim=D, depth=depth, num_heads=heads)
    torch.manual_seed(train_seed)
    mask = O.draw_span_mask(W // 4, 0.4, 8)
    np.testing.assert_array_equal(mask.numpy(), g["mask"])
    tg, tl = _labels(seed + 2, B, nb_cls, 4, 12)
    loss, grads, logits = O.train_step(sd, _images(seed + 1, B, W), tg, tl, mask, num_heads=heads)
    np.testing.assert_allclose(logits.numpy(), g["logits_train"], rtol=0, atol=3e-4)
    assert abs(loss - float(g["loss"])) <= 1e-4 * abs(float(g["loss"]))
    names = sorted(grads)
    assert names == g["grad_names"].tolist()
    norms = np.array([float(grads[k].double().norm()) for k in names])
    np.testing.assert_allclose(norms, g["grad_norms"], rtol=2e-3, atol=1e-6)
    np.testing.assert_allclose(sd["patch_embed.bn1.running_mean"].numpy(), g["bn1_running_mean"], atol=1e-6)
    np.testing.assert_allclose(sd["patch_embed.layer3.1.bn2.running_var"].numpy(), g["l3_running_var"], rtol=1e-4)
    assert int(sd["patch_embed.bn1.num_batches_tracked"]) == int(g["nbt"]) == 1


@pytest.mark.parametrize("tag", ["win_w1000", "win_w600"])
def test_window_pad_and_key_mask_path_matches_reference(tag):
    """Token counts that are not a multiple of the 16-token window (T = 250 / 150): zero padding + rolled key
    padding mask (model_window/model/HTR_VT.py:121-131,49-56)."""
    g = np.load(os.path.join(G, tag + ".npz"))
    nb_cls, W, B, seed = [int(v) for v in g["meta"]]
    sd = O.init_state_dict(nb_cls, [64, W], seed=seed, variant="window")
    with torch.no_grad():
        y = O.forward(sd, _images(seed + 1, B, W), training=False, variant="window")
    assert y.shape[1] % 16 != 0
    np.testing.assert_allclose(y.numpy(), g["logits_eval"], rtol=0, atol=3e-4)


def test_train_batch32_matches_reference():
    """Full architecture, B = 32 (well-conditioned batch statistics): logits, loss, per-sample nll, sampled gradients of
    all 101 trainable tensors and the decoded strings of valid.py:40-42."""
    g = np.load(os.path.join(G, "v1_train_b32.npz"))
    nb_cls, W, B, seed, train_seed = [int(v) for v in g["meta"]]
    sd = O.init_state_dict(nb_cls, [64, W], seed=seed)
    x = _images(seed + 1, B, W)
    with torch.no_grad():
        ye = O.forward(sd, x, training=False).numpy()
    np.testing.assert_allclose(ye, g["logits_eval"], rtol=0, atol=3e-4)
    alphabet = "".join(chr(33 + i) for i in range(nb_cls - 1))
    idx = O.argmax_first(g["logits_eval"]).reshape(-1)
    np.testing.assert_array_equal(idx, g["index_eval"].astype(np.int64))
    assert O.decode_strings(idx, [W // 4] * B, alphabet) == g["strings_eval"].tolist()
    torch.manual_seed(train_seed)
    mask = O.draw_span_mask(W // 4, 0.4, 8)
    np.testing.assert_array_equal(mask.numpy(), g["mask"])
    tg, tl = _labels(seed + 2, B, nb_cls, 16, 64)
    loss, grads, logits = O.train_step(sd, x, tg, tl, mask)
    np.testing.assert_allclose(logits.numpy(), g["logits_train"], rtol=0, atol=3e-4)
    assert abs(loss - float(g["loss"])) <= 1e-4 * abs(float(g["loss"]))
    off = 0
    for name, cnt, norm in zip(g["grad_names"].tolist(), g["grad_sample_counts"].tolist(), g["grad_norms"].tolist()):
        want = g["grad_samples"][off:off + cnt]
        off += cnt
        got = grads[name].reshape(-1)[torch.from_numpy(O.grad_sample_index(name, grads[name].numel()))].numpy()
        cos = float(got.astype(np.float64) @ want.astype(np.float64) /
                    (np.linalg.norm(got.astype(np.float64)) * np.linalg.norm(want.astype(np.float64)) + 1e-30))
        assert cos > 0.9999, (name, cos)
        assert abs(float(grads[name].double().norm()) - norm) <= 5e-3 * norm + 1e-7, name
    got_bn = np.concatenate([sd[k].numpy().reshape(-1) for k in sd if "running_" in k])
    np.testing.assert_allclose(got_bn, g["bn_running"], rtol=1e-4, atol=1e-6)


def test_ctc_f64_restatement_matches_torch_ctcloss():
    g = np.load(os.path.join(G, "ctc_cases.npz"))
    for name in g["names"].tolist():
        if name in ("iam_shape", "long_labels"):       # pure-python loops: keep the CPU suite fast
            sl = slice(0, 1)
        else:
            sl = slice(None)
        logits, tg = g[name + ".logits"], g[name + ".targets"]
        il, tl = g[name + ".in_len"], g[name + ".tgt_len"]
        B = logits[sl].shape[0]
        nll, grad = O.ctc_loss_grad(logits[:B], tg[: int(tl[:B].sum())], il[:B], tl[:B])
        np.testing.assert_allclose(nll, g[name + ".nll"][:B], rtol=1e-5, atol=1e-5, err_msg=name)
        np.testing.assert_allclose(grad, g[name + ".grad"][:B], rtol=1e-3, atol=1e-4, err_msg=name)  # torch CPU golden is fp32 (nll~1e3 => ~3e-4 rel)


def test_decode_restatement_matches_reference_converter():
    g = np.load(os.path.join(G, "decode_cases.npz"))
    alphabet = str(g["alphabet"])
    assert O.decode_strings(g["index"], g["lens"], alphabet) == g["strings"].tolist()
    assert O.decode_strings(g["index"], g["lens2"], alphabet) == g["strings2"].tolist()


def test_argmax_semantics_match_torch_max():
    g = np.load(os.path.join(G, "argmax_cases.npz"))
    np.testing.assert_array_equal(O.argmax_first(g["logits"]), g["index"])


def test_metrics_oracle_matches_reference_formatting_and_known_answers():
    """format_string_for_wer against strings produced by the reference's own function; Levenshtein against
    classic known answers, a brute-force check and metric axioms; the valid.py:49-75 accumulation."""
    import json
    with open(os.path.join(G, "metrics_cases.json")) as fh:
        g = json.load(fh)
    assert [O.format_string_for_wer(t) for t in g["texts"]] == g["formatted"]
    for a, b, d in g["kat"]:
        assert O.levenshtein(a, b) == d and O.levenshtein(b, a) == d
    rs = np.random.RandomState(0)
    seqs = [rs.randint(0, 4, size=rs.randint(0, 9)).tolist() for _ in range(24)]
    for a in seqs[:8]:
        for b in seqs[8:16]:
            d = O.levenshtein(a, b)
            assert abs(len(a) - len(b)) <= d <= max(len(a), len(b))
            for c in seqs[16:]:
                assert d <= O.levenshtein(a, c) + O.levenshtein(c, b)
    r = O.error_rates(g["preds"], g["labels"])
    for k, v in g["rates"].items():
        assert r[k] == pytest.approx(v)
    # "" formats to "" and "".split(" ") == ['']: the reference counts one (empty) word there (valid.py:56-66)
    assert O.error_rates([""], [""])["length_of_gt_wer"] == 1


def test_line_prep_oracle_matches_reference_ops():
    g = np.load(os.path.join(G, "line_prep_cases.npz"))
    y = O.line_prep_u8(g["img"], g["widths"])
    np.testing.assert_allclose(y, g["y"], rtol=0, atol=1e-6)
    # no widths: the u8 image is taken as is (padding already 255 in the loader's output)
    y2 = O.line_prep_u8(g["img"])
    x = torch.from_numpy(g["img"]).float() / 255.
    np.testing.assert_allclose(y2, torch.nn.functional.layer_norm(x, x.shape[1:], eps=1e-5).numpy(), atol=1e-6)


def test_beam_restatement_matches_reference_function():
    """kbest_paths / beam_search_with_lm vs the strings the reference's own `simple_ctc_beam_search_with_lm`
    (model_window/test_with_kenlm.py:25-59, exec'd from its source by oracle/make_golden.py) returned."""
    g = np.load(os.path.join(G, "beam_cases.npz"))

    def lm(text):
        return sum(((ord(ch) * 31 + i * 17) % 97) / 97.0 for i, ch in enumerate(text)) - 0.6 * len(text)

    for i in range(len(g["best"])):
        got = O.beam_search_with_lm(g["log_probs"][i], str(g["alphabet"]), lm, int(g["beam"][i]))
        assert got == str(g["best"][i])
    # K = 1 is the greedy path; float32 and float64 accumulation agree on these fixtures (they were selected so)
    lp = g["log_probs"][0]
    am = O.argmax_first(lp[None])[0]
    greedy = [int(v) for i, v in enumerate(am) if v != 0 and not (i > 0 and am[i - 1] == v)]
    assert O.kbest_paths(lp, 1)[0][0] == greedy
    assert [c[0] for c in O.kbest_paths(lp, 5, np.float32)] == [c[0] for c in O.kbest_paths(lp, 5)]


def test_prefix_beam_search_is_the_exact_labelling_posterior():
    """ctc_prefix_beam_search pinned by brute force: with a beam that holds every prefix, the score of every
    labelling equals the log-sum over all C^T alignment paths collapsing to it, and the order is the posterior order;
    the best labelling's score is bounded by the CTC likelihood identity (-nll of ctc_loss_grad on that labelling)."""
    rs = np.random.RandomState(5)
    for T, C in [(1, 3), (2, 3), (4, 3), (5, 4), (6, 2), (3, 5)]:
        x = rs.randn(T, C) * 1.5
        lp = (x - np.log(np.exp(x).sum(1, keepdims=True))).astype(np.float32)
        exact = O.labelling_logprobs_bruteforce(lp)
        got = O.ctc_prefix_beam_search(lp, 10 ** 6)
        assert len(got) >= len(exact)                       # prefixes longer than T carry -inf and rank last
        gd = {tuple(l): s for l, s in got}
        for lab, s in exact.items():
            assert abs(gd[lab] - s) < 1e-9, (T, C, lab)
        for lab, s in gd.items():
            if lab not in exact:
                assert s == -np.inf
        want_order = sorted(exact.items(), key=lambda kv: -kv[1])
        assert [tuple(l) for l, _ in got[:3]] == [k for k, _ in want_order[:3]]
        # total mass = 1
        assert abs(np.log(sum(np.exp(s) for s in exact.values()))) < 1e-5
    # the score of a labelling = -CTC nll of that labelling (the float64 alpha recursion of ctc_loss_grad)
    T, C = 7, 4
    x = rs.randn(1, T, C).astype(np.float32)
    lp = x[0] - np.log(np.exp(x[0].astype(np.float64)).sum(1, keepdims=True))
    best = O.ctc_prefix_beam_search(lp.astype(np.float32), 10 ** 6)[:4]
    for lab, s in best:
        if not lab:
            continue
        nll, _ = O.ctc_loss_grad(x, np.array(lab, dtype=np.int32), np.array([T]), np.array([len(lab)], dtype=np.int32))
        assert abs(-float(nll[0]) - s) < 2e-5 * max(1.0, abs(s)), (lab, nll, s)


def test_prefix_beam_narrow_beam_and_lm_pick():
    """A narrow beam returns at most K entries, best first, every score <= the exact posterior of its labelling
    (pruned mass only ever lowers a score); K = 1 on peaked frames is the greedy labelling; the LM pick keeps doubled
    letters."""
    rs = np.random.RandomState(6)
    T, C = 6, 4
    x = rs.randn(T, C) * 2
    lp = (x - np.log(np.exp(x).sum(1, keepdims=True))).astype(np.float32)
    exact = O.labelling_logprobs_bruteforce(lp)
    for K in (1, 2, 5):
        got = O.ctc_prefix_beam_search(lp, K)
        assert len(got) == K
        assert all(got[i][1] >= got[i + 1][1] for i in range(K - 1))
        for lab, s in got:
            assert s <= exact[tuple(lab)] + 1e-9
    peaked = np.full((7, 4), -30.0, dtype=np.float32)
    for t, c in enumerate([1, 1, 0, 1, 2, 2, 0]):
        peaked[t, c] = 0.0
    assert O.ctc_prefix_beam_search(peaked, 1)[0][0] == [1, 1, 2]
    assert O.prefix_beam_search_with_lm(peaked, "abc", lambda s: len(s), 3) in ("aab", "aabb", "aaab", "aabc", "aaba")
    assert O.prefix_beam_search_with_lm(peaked, "abc", lambda s: -abs(len(s) - 3) + (s == "aab"), 3) == "aab"
