"""GPU: the LM-fused CTC prefix beam search (csrc/prefix_beam.cu, LM instantiation; ops.ctc_prefix_beam_lm,
ctc_lm_decode, kbest_candidates(lm=...)) against the float64 oracle `ctc_prefix_beam_search_lm` (itself pinned to a
brute-force enumeration in tests/test_oracle_lm.py), alpha = beta = 0 against the plain kernel bit for bit, and the
refusals.  Kept apart from test_gpu_ctc_decode.py, whose autouse fixture repeats every test once per CTC kernel."""
import math

import numpy as np
import pytest
import torch

import htrvt_lm_oracle as LO
import htrvt_oracle as O
from test_oracle_lm import HAND_ARPA

pytestmark = pytest.mark.gpu

WEIGHTS = [(0.7, 0.0), (1.5, 2.0), (0.3, -1.0)]


def _h():
    import htrvt_b200
    return htrvt_b200


def _ops():
    from importlib import import_module
    _h()
    return import_module("htr-vt_b200.ops")


def _alphabet(C):
    """C - 1 characters: a, b, the space, then letters the LMs below do not list (<unk>)"""
    return ("ab " + "".join(chr(0x100 + i) for i in range(300)))[: C - 1]


def rand_arpa(path, order=8, seed=3, per_order=250, vocab=("a", "b", "<space>", "Ā", "ā", "Ă")):
    """A seeded random ARPA file whose n-gram set is closed under prefixes (every k-gram extends a listed (k-1)-gram,
    n-grams may start with <s> and end with </s>), random probs and bows.  ă stays out: an alphabet character
    the LM does not list."""
    rs = np.random.RandomState(seed)
    words = list(vocab)
    grams = [[(w,) for w in words + ["<s>", "</s>", "<unk>"]]]
    for k in range(2, order + 1):
        prev = [g for g in grams[-1] if g[-1] != "</s>" and (k > 2 or g[-1] != "<unk>")]
        got = set()
        for _ in range(per_order * 3):
            g = prev[rs.randint(len(prev))]
            if k == 2 and g != ("<s>",) and rs.rand() < 0.2:
                g = ("<s>",)
            w = (words + ["</s>"])[rs.randint(len(words) + 1)]
            got.add(g + (w,))
            if len(got) >= per_order:
                break
        grams.append(sorted(got))
    lines = ["\\data\\"] + ["ngram %d=%d" % (k + 1, len(g)) for k, g in enumerate(grams)] + [""]
    for k, gk in enumerate(grams):
        lines.append("\\%d-grams:" % (k + 1))
        for g in gk:
            p = -99.0 if g == ("<s>",) else -rs.uniform(0.05, 3.0)
            if k + 1 < order and g[-1] != "</s>":
                lines.append("%.6f\t%s\t%.6f" % (p, " ".join(g), -rs.uniform(0.0, 1.0)))
            else:
                lines.append("%.6f\t%s" % (p, " ".join(g)))
        lines.append("")
    lines.append("\\end\\")
    with open(path, "w", encoding="utf-8") as fh:
        fh.write("\n".join(lines) + "\n")
    return path


@pytest.fixture(scope="module")
def lm_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("lm")
    hand = d / "hand3.arpa"
    hand.write_text(HAND_ARPA, encoding="utf-8")
    return {"hand3": str(hand), "rand8": rand_arpa(str(d / "rand8.arpa"))}


def _load(path, C):
    h = _h()
    alphabet = _alphabet(C)
    return h.CharNGramLM.from_arpa(path, h.CTCLabelConverter(alphabet)), LO.arpa_load(path, alphabet)


def _lines(T, C, K, B=6):
    """the line mix of test_prefix_beam_matches_oracle: random, quantised ties, blank-heavy, peaked, ragged, every
    frame twice"""
    rs = np.random.RandomState(7 * T + C + K)
    x = rs.randn(B, T, C).astype(np.float32) * 2.0
    x[1] = np.round(x[1] * 2) / 2
    x[2, :, 0] += 5.0
    x[3] *= 4.0
    x[5] = np.repeat(x[5, ::2], 2, axis=0)[:T]
    lp = torch.from_numpy(x).log_softmax(-1).numpy()
    lengths = np.array([T, T, max(1, T // 2), T, max(1, T - 1), T], dtype=np.int32)[:B]
    return lp, lengths


def _close(a, b):
    if not np.isfinite(b):
        return a == b
    return abs(a - b) <= 1e-9 * max(1.0, abs(b))


def _check_line(ids, lens, sc, ctc, b, want):
    assert (lens[b] >= 0).sum() == len(want), b
    for r, (lab, fused, c) in enumerate(want):
        assert ids[b, r, : lens[b, r]].tolist() == lab, (b, r)
        assert _close(sc[b, r], fused), (b, r, sc[b, r], fused)
        assert _close(ctc[b, r], c), (b, r, ctc[b, r], c)
        assert not ids[b, r, lens[b, r]:].any()
    assert (lens[b, len(want):] == -1).all() and not ids[b, len(want):].any()


SHAPES = [(1, 7, 5), (9, 3, 8), (6, 4, 16), (128, 80, 5), (128, 80, 16), (256, 90, 8), (64, 228, 1), (40, 33, 3)]


@pytest.mark.parametrize("lm_name", ["hand3", "rand8"])
@pytest.mark.parametrize("T,C,K", SHAPES)
def test_kernel_matches_oracle(lm_files, lm_name, T, C, K):
    """labellings, their fused order, fused and ctc scores of every surviving entry; each weight pair on every line"""
    ops = _ops()
    lm, ref = _load(lm_files[lm_name], C)
    lp, lengths = _lines(T, C, K)
    x = torch.from_numpy(lp).cuda()
    for alpha, beta in WEIGHTS:
        ids, lens, sc, ctc = ops.ctc_prefix_beam_lm(x, K, lm, alpha, beta, torch.from_numpy(lengths), layout="btc")
        ids, lens, sc, ctc = ids.cpu().numpy(), lens.cpu().numpy(), sc.cpu().numpy(), ctc.cpu().numpy()
        for b in range(lp.shape[0]):
            want = LO.ctc_prefix_beam_search_lm(lp[b, : lengths[b]], K, ref, alpha, beta)
            _check_line(ids, lens, sc, ctc, b, want)


@pytest.mark.parametrize("T,C,K", SHAPES)
def test_zero_weights_are_bit_equal_to_the_plain_kernel(lm_files, T, C, K):
    ops = _ops()
    lp, lengths = _lines(T, C, K)
    x = torch.from_numpy(lp).cuda()
    ln = torch.from_numpy(lengths)
    ids0, lens0, sc0 = ops.ctc_prefix_beam(x, K, ln, layout="btc")
    for name in ("hand3", "rand8"):
        lm, _ = _load(lm_files[name], C)
        ids, lens, sc, ctc = ops.ctc_prefix_beam_lm(x, K, lm, 0.0, 0.0, ln, layout="btc")
        assert torch.equal(ids, ids0) and torch.equal(lens, lens0)
        assert torch.equal(sc.view(torch.int64), sc0.view(torch.int64))        # bit for bit
        assert torch.equal(ctc.view(torch.int64), sc0.view(torch.int64))


def test_exact_posterior(lm_files):
    """K = 16 holds every prefix of these lines: ctc_scores are the brute-force labelling posterior and the fused
    scores add exactly the LM's sentence score"""
    ops = _ops()
    rs = np.random.RandomState(11)
    for T, C in [(2, 3), (3, 3), (5, 2), (2, 4)]:
        lm, ref = _load(lm_files["hand3"], C)
        x = rs.randn(1, T, C).astype(np.float32) * 1.5
        lp = torch.from_numpy(x).log_softmax(-1)
        exact = O.labelling_logprobs_bruteforce(lp[0].numpy())
        for alpha, beta in WEIGHTS:
            ids, lens, sc, ctc = ops.ctc_prefix_beam_lm(lp.cuda(), 16, lm, alpha, beta, layout="btc")
            got = {}
            for r in range(16):
                if lens[0, r] >= 0:
                    got[tuple(ids[0, r, : int(lens[0, r])].cpu().tolist())] = (float(sc[0, r]), float(ctc[0, r]))
            toks = ref["tokens"]
            for lab, s in exact.items():
                words = [toks[c] if c < len(toks) else "<unk>" for c in lab]
                lmterm = alpha * LO.LN10 * LO.arpa_sentence_log10(ref, words) + beta * len(lab)
                assert abs(got[lab][1] - s) < 1e-9, (T, C, lab)
                assert abs(got[lab][0] - (s + lmterm)) < 1e-9, (T, C, lab)
            fs = [float(v) for v in sc[0][lens[0] >= 0].cpu()]
            assert fs == sorted(fs, reverse=True)


def test_the_lm_changes_the_answer(lm_files):
    """Acoustically "ba" beats "ab" (0.3025 vs 0.2025 over two frames); the hand 3-gram prefers "ab" (log10 P -1.45
    vs -2.1), so the fused search returns "ab" where the plain prefix search returns "ba"."""
    h, ops = _h(), _ops()
    lm, ref = _load(lm_files["hand3"], 3)
    conv = h.CTCLabelConverter("ab")
    p = np.array([[1e-13, 0.45, 0.55], [1e-13, 0.55, 0.45]], dtype=np.float64)
    lp = torch.from_numpy(np.log(p / p.sum(1, keepdims=True)).astype(np.float32)).unsqueeze(1)    # [T, 1, C]
    ids, lens, _ = ops.ctc_prefix_beam(lp.cuda(), 8)
    assert ids[0, 0, : int(lens[0, 0])].tolist() == [2, 1]                                        # "ba"
    assert h.ctc_lm_decode(lp.cuda(), conv, lm, alpha=1.0, beta=1.0) == ["ab"]
    assert LO.ctc_prefix_beam_search_lm(lp[:, 0].numpy(), 8, ref, 1.0, 1.0)[0][0] == [1, 2]
    assert h.ctc_lm_decode(lp.cuda(), conv, lm, alpha=0.0, beta=0.0) == ["ba"]


@pytest.mark.parametrize("with_lengths", [False, True])
def test_public_entry_points_match_the_oracle(lm_files, with_lengths):
    h = _h()
    T, B, C, K = 40, 7, 11, 8
    lm, ref = _load(lm_files["rand8"], C)
    alphabet = _alphabet(C)
    conv = h.CTCLabelConverter(alphabet)
    rs = np.random.RandomState(5)
    x = rs.randn(T, B, C).astype(np.float32) * 3
    x[:, 1, 0] += 4.0
    lp = torch.from_numpy(x).log_softmax(-1)
    lengths = rs.randint(1, T + 1, size=B).astype(np.int32) if with_lengths else np.full(B, T, dtype=np.int32)
    ln = torch.from_numpy(lengths) if with_lengths else None
    table = ["[blank]"] + list(alphabet)
    alpha, beta = 0.8, 0.5
    want = [LO.ctc_prefix_beam_search_lm(lp[: lengths[b], b].numpy(), K, ref, alpha, beta) for b in range(B)]
    spell = lambda lab: "".join(table[c] for c in lab if c < len(table))   # noqa: E731
    got = h.ctc_lm_decode(lp.cuda(), conv, lm, alpha, beta, beam_size=K, lengths=ln)
    assert got == [spell(w[0][0]) for w in want]
    for layout, t in (("tbc", lp), ("btc", lp.transpose(0, 1).contiguous())):
        cands = h.kbest_candidates(t.cuda(), conv, K, ln, layout=layout, search="prefix", lm=lm, alpha=alpha, beta=beta)
        for b in range(B):
            exp = [(spell(lab), fused) for lab, fused, _ in want[b] if spell(lab)]
            assert [c[0] for c in cands[b]] == [e[0] for e in exp], (layout, b)
            for c, e in zip(cands[b], exp):
                assert _close(c[1], e[1])


def test_refusals(lm_files):
    h, ops = _h(), _ops()
    lm, _ = _load(lm_files["hand3"], 5)
    x = torch.randn(10, 2, 5).log_softmax(-1)
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lm(x, 4, lm, 0.5)                                        # CPU tensor
    with pytest.raises(h._lib.HtrvtError):
        h.ctc_lm_decode(x, h.CTCLabelConverter("ab c"), lm, 0.5)
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lm(x.cuda().double(), 4, lm, 0.5)                         # not fp32
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lm(x.cuda().half(), 4, lm, 0.5)
    for bad in (math.nan, math.inf, -math.inf):
        with pytest.raises(h._lib.HtrvtError):
            ops.ctc_prefix_beam_lm(x.cuda(), 4, lm, bad)                              # non-finite alpha
        with pytest.raises(h._lib.HtrvtError):
            ops.ctc_prefix_beam_lm(x.cuda(), 4, lm, 0.5, bad)                         # non-finite beta
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lm(x.cuda(), 17, lm, 0.5)                                 # K > 16
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lm(torch.randn(10, 2, 257).log_softmax(-1).cuda(), 4, lm, 0.5)   # C > 256
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lm(torch.randn(5000, 1, 5).log_softmax(-1).cuda(), 16, lm, 0.5)  # T * K >= 65535
    with pytest.raises(ValueError):
        h.kbest_candidates(x.cuda(), h.CTCLabelConverter("ab c"), 4, lm=lm, alpha=0.5)     # search="paths"
    with pytest.raises(ValueError):
        h.kbest_candidates(x.cuda(), h.CTCLabelConverter("ab c"), 4, search="prefix", lm=lm)   # no alpha
    import copy
    other = copy.copy(lm)
    other.table = lm.table.cpu()                                                     # the table on another device
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lm(x.cuda(), 4, other, 0.5)
    if torch.cuda.device_count() > 1:
        other.table = lm.table.to("cuda:1")
        with pytest.raises(h._lib.HtrvtError):
            ops.ctc_prefix_beam_lm(x.cuda(), 4, other, 0.5)


def test_full_size_batch(lm_files):
    """512 lines, T = 256, C = 80, K = 8 (the inference batch): four sampled lines against the oracle"""
    ops = _ops()
    B, T, C, K = 512, 256, 80, 8
    lm, ref = _load(lm_files["rand8"], C)
    rs = np.random.RandomState(17)
    x = rs.randn(T, B, C).astype(np.float32) * 2.0
    x[:, ::2, 0] += 3.0
    lp = torch.from_numpy(x).log_softmax(-1)
    ids, lens, sc, ctc = ops.ctc_prefix_beam_lm(lp.cuda(), K, lm, 0.7, 0.5)
    ids, lens, sc, ctc = ids.cpu().numpy(), lens.cpu().numpy(), sc.cpu().numpy(), ctc.cpu().numpy()
    assert (lens[:, 0] >= 0).all() and np.isfinite(sc[:, 0]).all()
    for b in (0, 131, 302, 511):
        _check_line(ids, lens, sc, ctc, b, LO.ctc_prefix_beam_search_lm(lp[:, b].numpy(), K, ref, 0.7, 0.5))
