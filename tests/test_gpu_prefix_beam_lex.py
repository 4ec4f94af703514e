"""GPU: the lexicon-constrained CTC prefix beam search (csrc/prefix_beam.cu, LEX instantiations;
ops.ctc_prefix_beam_lex, ctc_lexicon_decode, kbest_candidates(lexicon=...)) against the oracle
`ctc_prefix_beam_search_lex` (pinned to a brute-force enumeration in tests/test_oracle_lex.py), with and without the
LM; an empty word-character set against the plain and LM kernels bit for bit; and the refusals."""
import math

import numpy as np
import pytest
import torch

import htrvt_lex_oracle as XO
import htrvt_oracle as O
from test_gpu_prefix_beam_lm import SHAPES, WEIGHTS, _alphabet, _check_line, _lines, _load, lm_files  # noqa: F401

pytestmark = pytest.mark.gpu


def _h():
    import htrvt_b200
    return htrvt_b200


def _ops():
    from importlib import import_module
    _h()
    return import_module("htr-vt_b200.ops")


def _words(C, n=40, seed=5):
    """seeded words of 1-4 characters over the alphabet's first letters except the space (so the space and the
    remaining letters are free)"""
    alphabet = _alphabet(C)
    letters = [ch for ch in alphabet if ch != " "][: max(1, min(6, (C - 1) * 2 // 3))]
    rs = np.random.RandomState(seed + C)
    return sorted({"".join(letters[i] for i in rs.randint(0, len(letters), size=rs.randint(1, 5))) for _ in range(n)})


def _lexicon(C, words=None, word_chars=None):
    h = _h()
    alphabet = _alphabet(C)
    conv = h.CTCLabelConverter(alphabet)
    lx = h.Lexicon.from_words(_words(C) if words is None else words, conv, word_chars)
    cls_of = {ch: c for c, ch in enumerate(conv.character) if c >= 1}
    kept = {tuple(cls_of[ch] for ch in w) for w in (_words(C) if words is None else words)
            if all(ch in cls_of and ch in lx.word_chars for ch in w)}
    is_word = lx.is_word.cpu().numpy().tolist()
    return lx, kept, is_word


def _run_and_check(x, lengths, lp, K, lx, kept, is_word, lm=None, ref=None, alpha=0.0, beta=0.0):
    ops = _ops()
    ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(x, K, lx, lm, alpha, beta, torch.from_numpy(lengths), layout="btc")
    ids, lens, sc, ctc = ids.cpu().numpy(), lens.cpu().numpy(), sc.cpu().numpy(), ctc.cpu().numpy()
    for b in range(lp.shape[0]):
        want = XO.ctc_prefix_beam_search_lex(lp[b, : lengths[b]], K, kept, is_word, ref, alpha, beta)
        _check_line(ids, lens, sc, ctc, b, want)
        for r in range(K):
            if lens[b, r] >= 0:
                assert XO.accepted(ids[b, r, : lens[b, r]].tolist(), kept, is_word), (b, r)


@pytest.mark.parametrize("T,C,K", SHAPES)
def test_lexicon_only_matches_oracle(T, C, K):
    lx, kept, is_word = _lexicon(C)
    lp, lengths = _lines(T, C, K)
    _run_and_check(torch.from_numpy(lp).cuda(), lengths, lp, K, lx, kept, is_word)


@pytest.mark.parametrize("lm_name", ["hand3", "rand8"])
@pytest.mark.parametrize("T,C,K", SHAPES)
def test_lexicon_and_lm_match_oracle(lm_files, lm_name, T, C, K):
    lx, kept, is_word = _lexicon(C)
    lm, ref = _load(lm_files[lm_name], C)
    lp, lengths = _lines(T, C, K)
    x = torch.from_numpy(lp).cuda()
    for alpha, beta in (WEIGHTS if lm_name == "rand8" else WEIGHTS[:1]):
        _run_and_check(x, lengths, lp, K, lx, kept, is_word, lm, ref, alpha, beta)


@pytest.mark.parametrize("T,C,K", SHAPES)
def test_no_word_characters_is_bit_equal_to_both_kernels(lm_files, T, C, K):
    ops = _ops()
    lx, _, _ = _lexicon(C, word_chars="")
    assert lx.n_words == 0 and lx.n_nodes == 1
    lp, lengths = _lines(T, C, K)
    x = torch.from_numpy(lp).cuda()
    ln = torch.from_numpy(lengths)
    ids0, lens0, sc0 = ops.ctc_prefix_beam(x, K, ln, layout="btc")
    ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(x, K, lx, lengths=ln, layout="btc")
    assert torch.equal(ids, ids0) and torch.equal(lens, lens0)
    assert torch.equal(sc.view(torch.int64), sc0.view(torch.int64))
    assert torch.equal(ctc.view(torch.int64), sc0.view(torch.int64))
    lm, _ = _load(lm_files["rand8"], C)
    for alpha, beta in WEIGHTS:
        want = ops.ctc_prefix_beam_lm(x, K, lm, alpha, beta, ln, layout="btc")
        got = ops.ctc_prefix_beam_lex(x, K, lx, lm, alpha, beta, ln, layout="btc")
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
        assert torch.equal(got[2].view(torch.int64), want[2].view(torch.int64))
        assert torch.equal(got[3].view(torch.int64), want[3].view(torch.int64))


def test_exact_posterior():
    """K = 16 holds every prefix of these lines: the accepted labellings with their exact posterior"""
    ops = _ops()
    rs = np.random.RandomState(11)
    for T, C in [(2, 3), (3, 3), (3, 4), (4, 3)]:
        lx, kept, is_word = _lexicon(C, words=["a", "ab", "ba", "bb"])
        x = rs.randn(1, T, C).astype(np.float32) * 1.5
        lp = torch.from_numpy(x).log_softmax(-1)
        exact = {k: v for k, v in O.labelling_logprobs_bruteforce(lp[0].numpy()).items()
                 if XO.accepted(k, kept, is_word)}
        ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(lp.cuda(), 16, lx, layout="btc")
        got = {tuple(ids[0, r, : int(lens[0, r])].cpu().tolist()): float(ctc[0, r])
               for r in range(16) if lens[0, r] >= 0 and ctc[0, r] > -math.inf}
        assert set(got) == set(exact), (T, C)
        for lab, s in exact.items():
            assert abs(got[lab] - s) < 1e-9, (T, C, lab)


def test_the_lexicon_changes_the_answer():
    """acoustically "ba" beats "ab"; with the lexicon {"ab"} the search returns "ab".  With {"aba"} only the empty
    labelling is accepted, and a beam of one that keeps "a" after the first frame finds no accepted labelling"""
    h, ops = _h(), _ops()
    conv = h.CTCLabelConverter("ab")
    p = np.array([[1e-13, 0.45, 0.55], [1e-13, 0.55, 0.45]], dtype=np.float64)
    lp = torch.from_numpy(np.log(p / p.sum(1, keepdims=True)).astype(np.float32)).unsqueeze(1)    # [T, 1, C]
    ids, lens, _ = ops.ctc_prefix_beam(lp.cuda(), 8)
    assert ids[0, 0, : int(lens[0, 0])].tolist() == [2, 1]
    lx = h.Lexicon.from_words(["ab"], conv)
    assert h.ctc_lexicon_decode(lp.cuda(), conv, lx) == ["ab"]
    assert XO.ctc_prefix_beam_search_lex(lp[:, 0].numpy(), 8, {(1, 2)}, [0, 1, 1])[0][0] == [1, 2]
    lx = h.Lexicon.from_words(["aba"], conv)                      # two frames cannot spell "aba": only "" is accepted
    ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(lp.cuda(), 4, lx)
    assert lens.tolist() == [[0, -1, -1, -1]] and not ids.any()
    ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(lp.cuda(), 1, lx)  # K = 1 keeps "a", which cannot end the line
    assert lens.tolist() == [[-1]] and not ids.any() and (sc == -math.inf).all() and (ctc == -math.inf).all()
    assert XO.ctc_prefix_beam_search_lex(lp[:, 0].numpy(), 1, {(1, 2, 1)}, [0, 1, 1]) == []
    assert h.ctc_lexicon_decode(lp.cuda(), conv, lx, beam_size=1) == [""]


@pytest.mark.parametrize("with_lengths", [False, True])
def test_public_entry_points_match_the_oracle(lm_files, with_lengths):
    h = _h()
    T, B, C, K = 40, 7, 11, 8
    lm, ref = _load(lm_files["rand8"], C)
    alphabet = _alphabet(C)
    conv = h.CTCLabelConverter(alphabet)
    lx, kept, is_word = _lexicon(C)
    rs = np.random.RandomState(5)
    x = rs.randn(T, B, C).astype(np.float32) * 3
    x[:, 1, 0] += 4.0
    lp = torch.from_numpy(x).log_softmax(-1)
    lengths = rs.randint(1, T + 1, size=B).astype(np.int32) if with_lengths else np.full(B, T, dtype=np.int32)
    ln = torch.from_numpy(lengths) if with_lengths else None
    table = ["[blank]"] + list(alphabet)
    spell = lambda lab: "".join(table[c] for c in lab if c < len(table))   # noqa: E731
    for use_lm, alpha, beta in ((False, 0.0, 0.0), (True, 0.8, 0.5)):
        lmx, refx = (lm, ref) if use_lm else (None, None)
        want = [XO.ctc_prefix_beam_search_lex(lp[: lengths[b], b].numpy(), K, kept, is_word, refx, alpha, beta)
                for b in range(B)]
        got = h.ctc_lexicon_decode(lp.cuda(), conv, lx, beam_size=K, lengths=ln, lm=lmx, alpha=alpha, beta=beta)
        assert got == [spell(w[0][0]) if w else "" for w in want]
        for layout, t in (("tbc", lp), ("btc", lp.transpose(0, 1).contiguous())):
            kw = dict(lm=lm, alpha=alpha, beta=beta) if use_lm else {}
            cands = h.kbest_candidates(t.cuda(), conv, K, ln, layout=layout, search="prefix", lexicon=lx, **kw)
            for b in range(B):
                exp = [(spell(lab), fused) for lab, fused, _ in want[b] if spell(lab)]
                assert [c[0] for c in cands[b]] == [e[0] for e in exp], (layout, b)
                for c, e in zip(cands[b], exp):
                    assert abs(c[1] - e[1]) <= 1e-9 * max(1.0, abs(e[1]))


def test_refusals(lm_files):
    h, ops = _h(), _ops()
    lm, _ = _load(lm_files["hand3"], 5)
    lx, _, _ = _lexicon(5)
    conv = h.CTCLabelConverter(_alphabet(5))
    x = torch.randn(10, 2, 5).log_softmax(-1)
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x, 4, lx)                                            # CPU tensor
    with pytest.raises(h._lib.HtrvtError):
        h.ctc_lexicon_decode(x, conv, lx)
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda().double(), 4, lx)                             # not fp32
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda().transpose(0, 2).contiguous().transpose(0, 2), 4, lx)   # strided classes
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda(), 4, lx, None, 0.5)                          # weights without an LM
    for bad in (math.nan, math.inf):
        with pytest.raises(h._lib.HtrvtError):
            ops.ctc_prefix_beam_lex(x.cuda(), 4, lx, lm, bad)                         # non-finite alpha
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda(), 17, lx)                                    # K > 16
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(torch.randn(10, 2, 257).log_softmax(-1).cuda(), 4, lx)   # C > 256
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(torch.randn(5000, 1, 5).log_softmax(-1).cuda(), 16, lx)  # T * K >= 65535
    with pytest.raises(ValueError):
        h.kbest_candidates(x.cuda(), conv, 4, lexicon=lx)                             # search="paths"
    with pytest.raises(ValueError):
        h.kbest_candidates(x.cuda(), conv, 4, search="prefix", lexicon=lx, lm=lm)     # no alpha
    import copy
    other = copy.copy(lx)
    other.first = lx.first.cpu()                                                     # the lexicon on another device
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda(), 4, other)
    other_lm = copy.copy(lm)
    other_lm.table = lm.table.cpu()
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda(), 4, lx, other_lm, 0.5)


def synthetic_words(n, alphabet, seed):
    """n distinct seeded words of 2-10 letters over alphabet"""
    rs = np.random.RandomState(seed)
    out = set()
    while len(out) < n:
        k = rs.randint(2, 11, size=n)
        idx = rs.randint(0, len(alphabet), size=int(k.sum()))
        s = "".join(alphabet[i] for i in idx)
        ends = np.cumsum(k)
        out.update(s[e - m:e] for e, m in zip(ends.tolist(), k.tolist()))
    return sorted(out)[:n]


def test_full_size_batch():
    """512 lines, T = 256, C = 80, K = 8 with a 10 000-word lexicon: every returned labelling accepted, four sampled
    lines against the oracle"""
    h, ops = _h(), _ops()
    B, T, C, K = 512, 256, 80, 8
    alphabet = "".join(chr(0x21 + i) for i in range(C - 2)) + " "
    conv = h.CTCLabelConverter(alphabet)
    words = synthetic_words(10000, alphabet[:52], seed=9)
    lx = h.Lexicon.from_words(words, conv)
    assert lx.n_words == 10000
    cls_of = {ch: c for c, ch in enumerate(conv.character) if c >= 1}
    kept = {tuple(cls_of[ch] for ch in w) for w in words}
    is_word = lx.is_word.cpu().numpy().tolist()
    rs = np.random.RandomState(17)
    x = rs.randn(T, B, C).astype(np.float32) * 2.0
    x[:, ::2, 0] += 3.0
    lp = torch.from_numpy(x).log_softmax(-1)
    ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(lp.cuda(), K, lx)
    ids, lens, sc, ctc = ids.cpu().numpy(), lens.cpu().numpy(), sc.cpu().numpy(), ctc.cpu().numpy()
    live = lens[:, 0] >= 0                  # random logits can leave every entry of a line inside a word at its end
    assert live.mean() > 0.5 and np.isfinite(sc[live, 0]).all() and (sc[~live] == -math.inf).all()
    for b in range(B):
        for r in range(K):
            if lens[b, r] >= 0:
                assert XO.accepted(ids[b, r, : lens[b, r]].tolist(), kept, is_word), (b, r)
    for b in (0, 131, 302, 511):
        _check_line(ids, lens, sc, ctc, b, XO.ctc_prefix_beam_search_lex(lp[:, b].numpy(), K, kept, is_word))
