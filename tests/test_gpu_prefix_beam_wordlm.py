"""GPU: the lexicon-constrained CTC prefix beam search with a word n-gram LM (csrc/prefix_beam.cu, word-LM
instantiations; ops.ctc_prefix_beam_lex(lm=WordNGramLM), ctc_lexicon_decode, kbest_candidates) against the oracle
`ctc_prefix_beam_search_wordlm` (pinned to a brute-force enumeration in tests/test_oracle_wordlm.py); zero weights
against the lexicon-only kernel bit for bit; a 10^5-word lexicon whose token ids pass 2^16; and the refusals."""
import math

import numpy as np
import pytest
import torch

import htrvt_lex_oracle as XO
import htrvt_lm_oracle as LO
import htrvt_oracle as O
import htrvt_wordlm_oracle as WO
from test_gpu_prefix_beam_lm import SHAPES, _alphabet, _check_line, _lines
from test_oracle_wordlm import HAND_WORD_ARPA

pytestmark = pytest.mark.gpu

WEIGHTS = [(0.7, 0.0), (1.5, 2.0), (0.3, -1.0)]


def _h():
    import htrvt_b200
    return htrvt_b200


def _ops():
    from importlib import import_module
    _h()
    return import_module("htr-vt_b200.ops")


def _words(C, n=40, seed=5):
    """seeded words of 1-4 characters over the alphabet's first letters except the space (the space and the remaining
    letters are free); "a", "ab", "ba" (the hand 3-gram's words) are among them"""
    alphabet = _alphabet(C)
    letters = [ch for ch in alphabet if ch != " "][: max(1, min(6, (C - 1) * 2 // 3))]
    rs = np.random.RandomState(seed + C)
    ws = {"".join(letters[i] for i in rs.randint(0, len(letters), size=rs.randint(1, 5))) for _ in range(n)}
    return sorted(ws | {w for w in ("a", "ab", "ba") if set(w) <= set(letters)})


def rand_word_arpa(path, vocab, order=6, seed=3, per_order=300):
    """a seeded random ARPA file over the words vocab (plus one word that is no lexicon word), closed under
    prefixes, with random probs and bows"""
    rs = np.random.RandomState(seed)
    words = list(vocab) + ["zzz"]
    grams = [[(w,) for w in words + ["<s>", "</s>", "<unk>"]]]
    for k in range(2, order + 1):
        prev = [g for g in grams[-1] if g[-1] != "</s>"]
        got = set()
        for _ in range(per_order * 3):
            g = ("<s>",) if (k == 2 and rs.rand() < 0.2) else prev[rs.randint(len(prev))]
            got.add(g + ((words + ["</s>"])[rs.randint(len(words) + 1)],))
            if len(got) >= per_order:
                break
        grams.append(sorted(got))
    write_arpa(path, grams, order, rs)
    return path


def write_arpa(path, grams, order, rs):
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


@pytest.fixture(scope="module")
def arpa_dir(tmp_path_factory):
    d = tmp_path_factory.mktemp("wordlm")
    (d / "hand3.arpa").write_text(HAND_WORD_ARPA, encoding="utf-8")
    return d


def _setup(C, arpa_dir, lm_name, words=None):
    """(lexicon, word LM, oracle words, is_word, alphabet, oracle LM) on C classes"""
    h = _h()
    alphabet = _alphabet(C)
    conv = h.CTCLabelConverter(alphabet)
    words = _words(C) if words is None else words
    lx = h.Lexicon.from_words(words, conv)
    if lm_name == "hand3":
        path = str(arpa_dir / "hand3.arpa")
    else:
        path = str(arpa_dir / ("rand6_%d.arpa" % C))
        rand_word_arpa(path, lx.words[::2], seed=C)                  # every other word listed, the rest are <unk>
    lm = h.WordNGramLM.from_arpa(path, lx)
    cls_of = {ch: c for c, ch in enumerate(conv.character) if c >= 1}
    kept = {tuple(cls_of[ch] for ch in w) for w in lx.words}
    return lx, lm, kept, lx.is_word.cpu().numpy().tolist(), alphabet, LO.arpa_load(path, "")


def _run_and_check(x, lengths, lp, K, lx, lm, kept, is_word, alphabet, ref, alpha, beta):
    ops = _ops()
    ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(x, K, lx, lm, alpha, beta, torch.from_numpy(lengths), layout="btc")
    ids, lens, sc, ctc = ids.cpu().numpy(), lens.cpu().numpy(), sc.cpu().numpy(), ctc.cpu().numpy()
    for b in range(lp.shape[0]):
        want = WO.ctc_prefix_beam_search_wordlm(lp[b, : lengths[b]], K, kept, is_word, alphabet, ref, alpha, beta)
        _check_line(ids, lens, sc, ctc, b, want)


@pytest.mark.parametrize("lm_name", ["hand3", "rand6"])
@pytest.mark.parametrize("T,C,K", SHAPES)
def test_kernel_matches_oracle(arpa_dir, lm_name, T, C, K):
    lx, lm, kept, is_word, alphabet, ref = _setup(C, arpa_dir, lm_name)
    lp, lengths = _lines(T, C, K)
    x = torch.from_numpy(lp).cuda()
    for alpha, beta in WEIGHTS:
        _run_and_check(x, lengths, lp, K, lx, lm, kept, is_word, alphabet, ref, alpha, beta)


@pytest.mark.parametrize("T,C,K", SHAPES)
def test_zero_weights_are_bit_equal_to_the_lexicon_kernel(arpa_dir, T, C, K):
    ops = _ops()
    lp, lengths = _lines(T, C, K)
    x = torch.from_numpy(lp).cuda()
    ln = torch.from_numpy(lengths)
    for name in ("hand3", "rand6"):
        lx, lm, _, _, _, _ = _setup(C, arpa_dir, name)
        ids0, lens0, sc0, ctc0 = ops.ctc_prefix_beam_lex(x, K, lx, lengths=ln, layout="btc")
        ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(x, K, lx, lm, 0.0, 0.0, ln, layout="btc")
        assert torch.equal(ids, ids0) and torch.equal(lens, lens0)
        assert torch.equal(ctc.view(torch.int64), ctc0.view(torch.int64))          # bit for bit
        assert torch.equal(sc.view(torch.int64), ctc.view(torch.int64))


def test_exact_posterior(arpa_dir):
    """K = 16 holds every prefix of these lines: every accepted labelling, its exact posterior, and a fused score that
    adds exactly the LM's sentence score over its words"""
    ops = _ops()
    rs = np.random.RandomState(11)
    for T, C in [(2, 3), (3, 3), (3, 4), (4, 3)]:
        lx, lm, kept, is_word, alphabet, ref = _setup(C, arpa_dir, "hand3", words=["a", "ab", "ba", "bb"])
        x = rs.randn(1, T, C).astype(np.float32) * 1.5
        lp = torch.from_numpy(x).log_softmax(-1)
        exact = {k: v for k, v in O.labelling_logprobs_bruteforce(lp[0].numpy()).items()
                 if XO.accepted(k, kept, is_word)}
        for alpha, beta in WEIGHTS:
            ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(lp.cuda(), 16, lx, lm, alpha, beta, layout="btc")
            got = {tuple(ids[0, r, : int(lens[0, r])].cpu().tolist()): (float(sc[0, r]), float(ctc[0, r]))
                   for r in range(16) if lens[0, r] >= 0 and ctc[0, r] > -math.inf}
            assert set(got) == set(exact), (T, C)
            for lab, s in exact.items():
                fin, run = WO.words_of(lab, is_word)
                toks = [WO.word_token(ref, "".join(alphabet[c - 1] for c in w)) for w in fin + ([run] if run else [])]
                lmterm = alpha * LO.LN10 * LO.arpa_sentence_log10(ref, toks) + beta * len(toks)
                assert abs(got[lab][1] - s) < 1e-9, (T, C, lab)
                assert abs(got[lab][0] - (s + lmterm)) < 1e-9, (T, C, lab)
            fs = [float(v) for v in sc[0][lens[0] >= 0].cpu()]
            assert fs == sorted(fs, reverse=True)


def test_the_word_lm_changes_the_answer(arpa_dir):
    """acoustically "ba" beats "ab" (0.3025 vs 0.2025); the hand 3-gram prefers "ab" (log10 P(ab </s>) = -1.3 vs
    log10 P(ba </s>) = -1.8), so with the lexicon {ab, ba} the lexicon-only search returns "ba" and the word LM "ab"."""
    h, ops = _h(), _ops()
    conv = h.CTCLabelConverter("ab")
    p = np.array([[1e-13, 0.45, 0.55], [1e-13, 0.55, 0.45]], dtype=np.float64)
    lp = torch.from_numpy(np.log(p / p.sum(1, keepdims=True)).astype(np.float32)).unsqueeze(1)    # [T, 1, C]
    lx = h.Lexicon.from_words(["ab", "ba"], conv)
    lm = h.WordNGramLM.from_arpa(str(arpa_dir / "hand3.arpa"), lx)
    assert h.ctc_lexicon_decode(lp.cuda(), conv, lx) == ["ba"]
    assert h.ctc_lexicon_decode(lp.cuda(), conv, lx, lm=lm, alpha=1.0, beta=0.0) == ["ab"]
    ref = LO.arpa_load(str(arpa_dir / "hand3.arpa"), "")
    assert WO.ctc_prefix_beam_search_wordlm(lp[:, 0].numpy(), 8, {(1, 2), (2, 1)}, [0, 1, 1], "ab", ref, 1.0,
                                            0.0)[0][0] == [1, 2]


@pytest.mark.parametrize("with_lengths", [False, True])
def test_public_entry_points_match_the_oracle(arpa_dir, with_lengths):
    h = _h()
    T, B, C, K = 40, 7, 11, 8
    lx, lm, kept, is_word, alphabet, ref = _setup(C, arpa_dir, "rand6")
    conv = h.CTCLabelConverter(alphabet)
    rs = np.random.RandomState(5)
    x = rs.randn(T, B, C).astype(np.float32) * 3
    x[:, 1, 0] += 4.0
    lp = torch.from_numpy(x).log_softmax(-1)
    lengths = rs.randint(1, T + 1, size=B).astype(np.int32) if with_lengths else np.full(B, T, dtype=np.int32)
    ln = torch.from_numpy(lengths) if with_lengths else None
    table = ["[blank]"] + list(alphabet)
    spell = lambda lab: "".join(table[c] for c in lab if c < len(table))   # noqa: E731
    alpha, beta = 0.8, 0.5
    want = [WO.ctc_prefix_beam_search_wordlm(lp[: lengths[b], b].numpy(), K, kept, is_word, alphabet, ref, alpha, beta)
            for b in range(B)]
    got = h.ctc_lexicon_decode(lp.cuda(), conv, lx, beam_size=K, lengths=ln, lm=lm, alpha=alpha, beta=beta)
    assert got == [spell(w[0][0]) if w else "" for w in want]
    for layout, t in (("tbc", lp), ("btc", lp.transpose(0, 1).contiguous())):
        cands = h.kbest_candidates(t.cuda(), conv, K, ln, layout=layout, search="prefix", lexicon=lx, lm=lm,
                                   alpha=alpha, beta=beta)
        for b in range(B):
            exp = [(spell(lab), fused) for lab, fused, _ in want[b] if spell(lab)]
            assert [c[0] for c in cands[b]] == [e[0] for e in exp], (layout, b)
            for c, e in zip(cands[b], exp):
                assert abs(c[1] - e[1]) <= 1e-9 * max(1.0, abs(e[1]))


def test_refusals(arpa_dir):
    h, ops = _h(), _ops()
    lx, lm, _, _, _, _ = _setup(5, arpa_dir, "hand3")
    conv = h.CTCLabelConverter(_alphabet(5))
    x = torch.randn(10, 2, 5).log_softmax(-1)
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x, 4, lx, lm, 0.5)                                   # CPU tensor
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda().double(), 4, lx, lm, 0.5)                    # not fp32
    for bad in (math.nan, math.inf):
        with pytest.raises(h._lib.HtrvtError):
            ops.ctc_prefix_beam_lex(x.cuda(), 4, lx, lm, bad)                         # non-finite alpha
        with pytest.raises(h._lib.HtrvtError):
            ops.ctc_prefix_beam_lex(x.cuda(), 4, lx, lm, 0.5, bad)                    # non-finite beta
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda(), 17, lx, lm, 0.5)                           # K > 16
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(torch.randn(10, 2, 257).log_softmax(-1).cuda(), 4, lx, lm, 0.5)   # C > 256
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(torch.randn(5000, 1, 5).log_softmax(-1).cuda(), 16, lx, lm, 0.5)  # T * K >= 65535
    import copy
    for field, value in (("order", 7), ("slots", lm.slots + 1)):
        bad_lm = copy.copy(lm)
        setattr(bad_lm, field, value)
        with pytest.raises(h._lib.HtrvtError):
            ops.ctc_prefix_beam_lex(x.cuda(), 4, lx, bad_lm, 0.5)                     # order 7, slots not 2^k
    with pytest.raises(ValueError):
        ops.ctc_prefix_beam_lex(x.cuda(), 4, h.Lexicon.from_words(lx.words, conv), lm, 0.5)   # another lexicon
    with pytest.raises(ValueError):
        h.ctc_lm_decode(x.cuda(), conv, lm, 0.5)                                     # a word LM without a lexicon
    with pytest.raises(ValueError):
        h.kbest_candidates(x.cuda(), conv, 4, search="prefix", lm=lm, alpha=0.5)
    with pytest.raises(ValueError):
        h.kbest_candidates(x.cuda(), conv, 4, lexicon=lx, lm=lm, alpha=0.5)          # search="paths"
    other = copy.copy(lm)
    other.table = lm.table.cpu()                                                     # the table on another device
    with pytest.raises(h._lib.HtrvtError):
        ops.ctc_prefix_beam_lex(x.cuda(), 4, lx, other, 0.5)


def test_large_vocabulary_batch(tmp_path):
    """512 lines, T = 128, C = 80, K = 8 with 10^5 words, every word listed as a unigram and with a <s> bigram: token
    ids reach 10^5 + 2, so the queried keys hold ids >= 2^16; three sampled lines against the oracle"""
    from test_gpu_prefix_beam_lex import synthetic_words
    h, ops = _h(), _ops()
    B, T, C, K = 512, 128, 80, 8
    alphabet = "".join(chr(0x21 + i) for i in range(C - 2)) + " "
    conv = h.CTCLabelConverter(alphabet)
    words = synthetic_words(100000, alphabet[:52], seed=9)
    lx = h.Lexicon.from_words(words, conv)
    assert lx.n_words == 100000
    rs = np.random.RandomState(21)
    grams = [[(w,) for w in lx.words + ["<s>", "</s>", "<unk>"]], [("<s>", w) for w in lx.words]]
    pairs = rs.randint(0, len(lx.words), size=(20000, 2))
    grams[1] += sorted({(lx.words[i], lx.words[j]) for i, j in pairs.tolist()} |
                       {(w, "</s>") for w in lx.words[::3]})
    path = str(tmp_path / "big2.arpa")
    write_arpa(path, grams, 2, rs)
    lm = h.WordNGramLM.from_arpa(path, lx)
    assert lm.n_unk_words == 0 and int(lm.node_tok.max()) == 100002
    ref = LO.arpa_load(path, "")
    cls_of = {ch: c for c, ch in enumerate(conv.character) if c >= 1}
    kept = {tuple(cls_of[ch] for ch in w) for w in lx.words}
    is_word = lx.is_word.cpu().numpy().tolist()
    x = rs.randn(T, B, C).astype(np.float32) * 2.0
    x[:, ::2, 0] += 3.0
    lp = torch.from_numpy(x).log_softmax(-1)
    ids, lens, sc, ctc = ops.ctc_prefix_beam_lex(lp.cuda(), K, lx, lm, 0.8, 1.0)
    ids, lens, sc, ctc = ids.cpu().numpy(), lens.cpu().numpy(), sc.cpu().numpy(), ctc.cpu().numpy()
    live = lens[:, 0] >= 0
    assert live.mean() > 0.5 and np.isfinite(sc[live, 0]).all()
    word_id = {w: 3 + i for i, w in enumerate(lx.words)}
    high = 0
    for b in range(B):
        for r in range(K):
            if lens[b, r] >= 0:
                lab = ids[b, r, : lens[b, r]].tolist()
                assert XO.accepted(lab, kept, is_word), (b, r)
                fin, _ = WO.words_of(lab + [C - 1], is_word)
                high += sum(word_id["".join(alphabet[c - 1] for c in w)] >= 1 << 16 for w in fin)
    assert high > 0                                                   # the returned words include ids >= 2^16
    for b in (0, 131, 302):
        _check_line(ids, lens, sc, ctc, b,
                    WO.ctc_prefix_beam_search_wordlm(lp[:, b].numpy(), K, kept, is_word, alphabet, ref, 0.8, 1.0))
