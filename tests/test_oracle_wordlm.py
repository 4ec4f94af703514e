"""CPU: the word n-gram LM of the lexicon-constrained CTC prefix beam search - the oracle against a brute-force
enumeration of the accepted labellings ranked by the fused score, hand-derived backoff values, and the host-side
packing (htr-vt_b200/wordlm.py: 21-bit keys, node tokens, smear, counters, refusals)."""
import math
from importlib import import_module

import numpy as np
import pytest
import torch

import htrvt_lex_oracle as XO
import htrvt_lm_oracle as LO
import htrvt_oracle as O
import htrvt_wordlm_oracle as WO

# words "a", "ab", "ba" (listed), "bb" (not listed: <unk>); "zz" is no lexicon word, so its two n-grams are dropped
HAND_WORD_ARPA = """\\data\\
ngram 1=7
ngram 2=5
ngram 3=2

\\1-grams:
-1.0\t<unk>
-99\t<s>\t-0.5
-0.7\t</s>
-0.6\tab\t-0.3
-0.8\tba\t-0.2
-1.2\ta\t-0.4
-2.0\tzz

\\2-grams:
-0.3\t<s> ab\t-0.1
-0.4\tab ba\t-0.25
-0.5\tba </s>
-0.9\tab </s>
-0.2\tzz ab

\\3-grams:
-0.2\t<s> ab ba
-0.15\tab ba </s>

\\end\\
"""
ALPHABET = "ab "                    # a = 1, b = 2 (word characters), the space = 3 (free)
LEX_WORDS = ["a", "ab", "ba", "bb"]
WORDS = {(1,), (1, 2), (2, 1), (2, 2)}
IS_WORD = [0, 1, 1, 0]


def _h():
    import htrvt_b200
    return htrvt_b200


def _wordlm():
    _h()
    return import_module("htr-vt_b200.wordlm")


def _lm(tmp_path, text=HAND_WORD_ARPA, name="w3.arpa"):
    path = tmp_path / name
    path.write_text(text, encoding="utf-8")
    return str(path), LO.arpa_load(str(path), "")


def _lp(T, C, seed, scale=1.5):
    x = np.random.RandomState(seed).randn(T, C).astype(np.float32) * scale
    return torch.from_numpy(x).log_softmax(-1).numpy()


def _spell(run):
    return "".join(ALPHABET[c - 1] for c in run)


def _fused_direct(ctc, labels, lm, alpha, beta):
    """ctc + alpha ln10 log10 P(w_1 .. w_m </s>) + beta m, from the sentence score of the LM oracle"""
    fin, run = WO.words_of(labels, IS_WORD)
    toks = [WO.word_token(lm, _spell(w)) for w in fin + ([run] if run else [])]
    return ctc + alpha * LO.LN10 * LO.arpa_sentence_log10(lm, toks) + beta * len(toks)


@pytest.mark.parametrize("T,C", [(2, 3), (3, 3), (3, 4), (4, 4), (5, 3)])
def test_wide_beam_is_the_bruteforce_ranking(tmp_path, T, C):
    """a beam wider than the number of prefixes: the oracle returns every accepted labelling with fused = ctc + the
    word LM's sentence score, best first - the top K of the brute-force enumeration for every K"""
    _, lm = _lm(tmp_path)
    for seed in range(3):
        lp = _lp(T, C, 10 * T + C + seed)
        for alpha, beta in ((0.7, 0.0), (1.5, 2.0), (0.3, -1.0)):
            exact = {k: _fused_direct(v, k, lm, alpha, beta)
                     for k, v in O.labelling_logprobs_bruteforce(lp).items() if XO.accepted(k, WORDS, IS_WORD)}
            got = [e for e in WO.ctc_prefix_beam_search_wordlm(lp, 300, WORDS, IS_WORD, ALPHABET, lm, alpha, beta)
                   if e[2] > -math.inf]
            assert {tuple(lab) for lab, _, _ in got} == set(exact)
            for lab, fused, _ in got:
                assert abs(fused - exact[tuple(lab)]) < 1e-9
            ranked = sorted(exact.values(), reverse=True)
            assert all(abs(a - b) < 1e-9 for a, b in zip([f for _, f, _ in got], ranked))


def test_hand_backoff(tmp_path):
    """log10 P by hand: "ab ba" = -0.3 - 0.2 - 0.15; "ba ab" = (-0.5 - 0.8) + (-0.2 - 0.6) + (0 - 0.9) (the context
    "ba ab" is not listed); "bb" is <unk>: (-0.5 - 1.0) + (0 + 0 - 0.7); the empty line = -0.5 - 0.7"""
    _, lm = _lm(tmp_path)
    f32 = lambda v: float(np.float32(v))   # noqa: E731
    cases = {("ab", "ba"): f32(-0.3) + f32(-0.2) + f32(-0.15),
             ("ba", "ab"): (f32(-0.5) + f32(-0.8)) + (f32(-0.2) + f32(-0.6)) + f32(-0.9),
             ("<unk>",): (f32(-0.5) + f32(-1.0)) + f32(-0.7),
             (): f32(-0.5) + f32(-0.7)}
    for toks, want in cases.items():
        assert abs(LO.arpa_sentence_log10(lm, list(toks)) - want) < 1e-12, toks
    assert WO.word_token(lm, "bb") == "<unk>" and WO.word_token(lm, "ab") == "ab"
    # a peaked line spelling "ab ba": the oracle's fused score carries exactly that sentence score and two bonuses
    p = np.full((5, 4), 0.1 / 3)
    for t, c in enumerate([1, 2, 3, 2, 1]):
        p[t, c] = 0.9
    lp = np.log(p).astype(np.float32)
    lab, fused, ctc = WO.ctc_prefix_beam_search_wordlm(lp, 8, WORDS, IS_WORD, ALPHABET, lm, 1.0, 0.5)[0]
    assert lab == [1, 2, 3, 2, 1]
    assert abs(fused - (ctc + LO.LN10 * cases[("ab", "ba")] + 1.0)) < 1e-9


def test_zero_weights_are_the_lexicon_search(tmp_path):
    _, lm = _lm(tmp_path)
    for T, C, K in [(6, 4, 3), (9, 4, 5), (7, 4, 1)]:
        lp = _lp(T, C, T * C + K, scale=2.0)
        got = WO.ctc_prefix_beam_search_wordlm(lp, K, WORDS, IS_WORD, ALPHABET, lm, 0.0, 0.0)
        assert [(lab, c) for lab, _, c in got] == [(lab, c) for lab, _, c in XO.ctc_prefix_beam_search_lex(
            lp, K, WORDS, IS_WORD)]
        assert all(f == c for _, f, c in got)


def test_smear_decides_a_narrow_beam(tmp_path):
    """K = 1, lexicon {ab, ba}: after the first frame "b" (0.55) beats "a" (0.45) acoustically and no word is finished
    yet, so only the smear term can keep "a": smear(a) = log10 p(ab) = -0.6 against smear(b) = log10 p(ba) = -0.8, and
    ln10 * 0.2 > ln(0.55 / 0.45).  Without the LM the beam keeps "b" and ends on "ba"; with it, on "ab".  The returned
    score is the sentence score of "ab", without the smear term"""
    _, lm = _lm(tmp_path)
    words = {(1, 2), (2, 1)}
    p = np.array([[1e-6, 0.45, 0.55, 1e-6], [1e-6, 0.5, 0.5, 1e-6]])
    lp = np.log(p / p.sum(1, keepdims=True)).astype(np.float32)
    assert [lab for lab, _, _ in XO.ctc_prefix_beam_search_lex(lp, 1, words, IS_WORD)] == [[2, 1]]
    assert [lab for lab, _, _ in WO.ctc_prefix_beam_search_wordlm(lp, 1, words, IS_WORD, ALPHABET, lm, 0.0, 0.0)] == \
        [[2, 1]]
    (lab, fused, ctc), = WO.ctc_prefix_beam_search_wordlm(lp, 1, words, IS_WORD, ALPHABET, lm, 1.0, 0.5)
    assert lab == [1, 2]
    assert abs(fused - _fused_direct(ctc, (1, 2), lm, 1.0, 0.5)) < 1e-12
    assert abs(ctc - O.labelling_logprobs_bruteforce(lp)[(1, 2)]) < 1e-9


# ---- host packing -------------------------------------------------------------------------------------------------
def test_21_bit_keys_round_trip():
    _h()
    L = import_module("htr-vt_b200.lm")
    rs = np.random.RandomState(4)
    keys = {tuple(rs.randint(0, (1 << 21) - 1, size=k).tolist()) for k in range(1, 7) for _ in range(300)}
    keys |= {(0,), ((1 << 21) - 2,) * 6, (65535, 65536, 3)}
    keys = sorted(keys, key=lambda t: (len(t), t))
    lo = np.concatenate([L.pack_keys(np.array([k]), bits=21)[0] for k in keys])
    hi = np.concatenate([L.pack_keys(np.array([k]), bits=21)[1] for k in keys])
    assert len(set(zip(lo.tolist(), hi.tolist()))) == len(keys)
    ps = np.arange(len(keys), dtype=np.float64) * -0.001
    table = L.pack_table(lo, hi, ps, ps / 2)
    idx = L.table_find(table, lo, hi)
    assert (idx >= 0).all()
    p, b = L.table_values(table, idx)
    assert np.array_equal(p, ps.astype(np.float32)) and np.array_equal(b, (ps / 2).astype(np.float32))
    # the field layout: last token first, three 21-bit fields per word
    lo1, hi1 = L.pack_keys(np.array([[10, 20, 30, 40, 50]]), bits=21)
    assert int(lo1[0]) == 51 | (41 << 21) | (31 << 42) and int(hi1[0]) == 21 | (11 << 21)
    # the character LM's 16-bit layout is unchanged
    lo2, hi2 = L.pack_keys(np.array([[1, 2, 3, 4, 5]]))
    assert int(lo2[0]) == 6 | (5 << 16) | (4 << 32) | (3 << 48) and int(hi2[0]) == 2
    with pytest.raises(ValueError):
        L.pack_keys(np.array([[1] * 7]), bits=21)
    with pytest.raises(ValueError):
        L.pack_keys(np.array([[(1 << 21) - 1]]), bits=21)


def test_node_tokens_smear_and_counters(tmp_path):
    h, W = _h(), _wordlm()
    path, _ = _lm(tmp_path)
    lx = h.Lexicon.on_host(LEX_WORDS, h.CTCLabelConverter(ALPHABET, device="cpu"))
    # breadth first: 0 root; 1 = a, 2 = b; 3 = ab, 4 = ba, 5 = bb
    assert lx.words == LEX_WORDS and lx.word_node.tolist() == [1, 3, 4, 5]
    order, counts, table, node_tok, smear, kept, n_dropped, n_unk = W.WordNGramLM.host_tables(path, lx)
    assert (order, counts, kept, n_dropped, n_unk) == (3, [7, 5, 2], 12, 2, 1)
    # ids: a = 3, ab = 4, ba = 5, bb = <unk> = 0
    assert node_tok.tolist() == [-1, 3, -1, 4, 5, 0]
    f32 = np.float32
    assert smear.dtype == np.float32
    assert smear.tolist() == [f32(-0.6), f32(-0.6), f32(-0.8), f32(-0.6), f32(-0.8), f32(-1.0)]
    L = import_module("htr-vt_b200.lm")
    for ids, p in (((4,), -0.6), ((1, 4, 5), -0.2), ((0,), -1.0), ((4, 2), -0.9)):
        i = L.table_find(table, *L.pack_keys(np.array([ids]), bits=21))
        assert i[0] >= 0 and L.table_values(table, i)[0][0] == f32(p), ids
    lm = W.WordNGramLM.from_arpa(path, lx)
    assert lm.lexicon is lx and lm.device.type == "cpu" and lm.node_tok.dtype == torch.int32


def test_node_smear_on_a_random_trie():
    """the level pass equals the maximum over every node's subtree, computed word by word"""
    W = _wordlm()
    m = import_module("htr-vt_b200.lexicon")
    rs = np.random.RandomState(8)
    words = sorted({tuple(rs.randint(1, 5, size=rs.randint(1, 6))) for _ in range(200)})
    first, label, child, end = m.pack_trie(words)
    nodes = m.trie_nodes(first, label, child, words)
    p = rs.uniform(-5, 0, size=len(words)).astype(np.float32)
    node_p = np.full(len(end), -np.inf, dtype=np.float32)
    node_p[nodes] = p
    got = W.node_smear(first, child, node_p)
    want = {}
    for w, v in zip(words, p):
        for k in range(0, len(w) + 1):
            want[w[:k]] = max(want.get(w[:k], -np.inf), v)
    prefix_node = dict(zip([w[:k] for w in words for k in range(len(w) + 1)],
                           m.trie_nodes(first, label, child, [w[:k] for w in words for k in range(len(w) + 1)])))
    for pre, n in prefix_node.items():
        assert got[n] == want[pre], pre


def test_refusals(tmp_path):
    h, W = _h(), _wordlm()
    conv = h.CTCLabelConverter(ALPHABET, device="cpu")
    lx = h.Lexicon.on_host(LEX_WORDS, conv)
    text7 = "\\data\\\n" + "".join("ngram %d=1\n" % k for k in range(1, 8)) + "\n"
    for k in range(1, 8):
        text7 += "\\%d-grams:\n-0.5\t%s\n\n" % (k, " ".join(["ab"] * k))
    text7 += "\\end\\\n"
    path7, _ = _lm(tmp_path, text7, "w7.arpa")
    with pytest.raises(ValueError):
        W.WordNGramLM.host_tables(path7, lx)                                      # order 7
    path, _ = _lm(tmp_path)
    lm = W.WordNGramLM.from_arpa(path, lx)
    other = h.Lexicon.on_host(LEX_WORDS, conv)
    ops = import_module("htr-vt_b200.ops")
    x = torch.randn(4, 1, 4).log_softmax(-1)
    with pytest.raises(ValueError):
        ops.ctc_prefix_beam_lex(x, 4, other, lm, 0.5)                             # built on another lexicon
    with pytest.raises(ValueError):
        ops.ctc_prefix_beam_lm(x, 4, lm, 0.5)                                     # a word LM needs the lexicon
    with pytest.raises(ValueError):
        h.kbest_candidates(x, conv, 4, search="prefix", lm=lm, alpha=0.5)         # ... in kbest_candidates too
    with pytest.raises(ValueError):
        h.kbest_candidates(x, conv, 4, lexicon=lx, lm=lm, alpha=0.5)              # search="paths"
