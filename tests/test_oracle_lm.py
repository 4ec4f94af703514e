"""CPU: the character n-gram LM of the LM-fused CTC prefix beam search - the oracle's ARPA backoff scores against
hand-derived values, refusal of malformed files, the fused search against a brute-force enumeration, alpha = beta = 0
against the plain search, and the host-side packing of the device table (exact keys, no false matches)."""
import math
from importlib import import_module

import numpy as np
import pytest
import torch

import htrvt_lm_oracle as LO
import htrvt_oracle as O

# A 3-gram over a, b and the space.  Alphabet "ab c": classes 1 = a, 2 = b, 3 = ' ' (<space>), 4 = c (not in the LM:
# <unk>); class 5 lies beyond the alphabet (<unk> too).
HAND_ARPA = """some header text a writer may put first

\\data\\
ngram 1=6
ngram 2=5
ngram 3=2

\\1-grams:
-1.0\t<unk>
-99\t<s>\t-0.5
-0.7\t</s>
-0.4\ta\t-0.3
-0.6\tb\t-0.2
-0.9\t<space>\t-0.1

\\2-grams:
-0.3\t<s> a\t-0.25
-0.5\ta b\t-0.15
-0.2\tb a
-0.8\ta </s>
-0.45\tb <space>

\\3-grams:
-0.1\t<s> a b
-0.35\ta b a

\\end\\
"""
ALPHABET = "ab c"


def _write(tmp_path, text, name="lm.arpa"):
    p = tmp_path / name
    p.write_text(text, encoding="utf-8")
    return str(p)


def _lmmod():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200.lm")


def _converter(alphabet):
    import htrvt_b200 as h
    return h.CTCLabelConverter(alphabet, device="cpu")


@pytest.fixture
def hand(tmp_path):
    return LO.arpa_load(_write(tmp_path, HAND_ARPA), ALPHABET)


def test_hand_backoff_cases(hand):
    lm = hand
    assert lm["order"] == 3 and lm["counts"] == [6, 5, 2]
    assert lm["tokens"] == ["<blank>", "a", "b", "<space>", "<unk>"]
    lp = lambda ctx, w: LO.arpa_logprob(lm, ctx, w)          # noqa: E731
    # trigram hit: p(b | <s> a) is listed
    assert lp(("<s>", "a"), "b") == pytest.approx(-0.1, abs=1e-6)
    # bigram backoff with a non-zero bow: (a b <space>) unlisted -> bow(a b) -0.15 + p(<space> | b) -0.45
    assert lp(("<s>", "a", "b"), "<space>") == pytest.approx(-0.6, abs=1e-6)
    # two-level backoff to the unigram: bow(a b) -0.15 + bow(b) -0.2 + p(</s>) -0.7
    assert lp(("<s>", "a", "b"), "</s>") == pytest.approx(-1.05, abs=1e-6)
    # unlisted context: (<s> b) is no bigram, bow 0 -> p(a | b) -0.2
    assert lp(("<s>", "b"), "a") == pytest.approx(-0.2, abs=1e-6)
    # only the last order-1 tokens count
    assert lp(("<s>", "b", "a", "b"), "a") == pytest.approx(-0.35, abs=1e-6)
    # an alphabet character missing from the LM is <unk>: (<s> a <unk>) unlisted -> bow(<s> a) -0.25, (a <unk>)
    # unlisted -> bow(a) -0.3, p(<unk>) -1.0
    assert lp(("<s>", "a"), "<unk>") == pytest.approx(-1.55, abs=1e-6)
    # the </s> term after <unk>: bow(a <unk>) 0, bow(<unk>) 0, p(</s>) -0.7
    assert lp(("<s>", "a", "<unk>"), "</s>") == pytest.approx(-0.7, abs=1e-6)
    # <s> first: (<s> b) unlisted -> bow(<s>) -0.5 + p(b) -0.6
    assert lp(("<s>",), "b") == pytest.approx(-1.1, abs=1e-6)


def test_hand_sentence_scores(hand):
    lm = hand
    tok = lambda s: [lm["tokens"][ALPHABET.index(ch) + 1] for ch in s]  # noqa: E731
    # "ab":  p(a|<s>) -0.3 + p(b|<s> a) -0.1 + p(</s>|a b) -1.05
    assert LO.arpa_sentence_log10(lm, tok("ab")) == pytest.approx(-1.45, abs=1e-6)
    # "ab ": -0.3 - 0.1 + p(<space>|a b) -0.6 + p(</s>|b <space>): bow(b <space>) 0, (<space> </s>) unlisted,
    # bow(<space>) -0.1 + p(</s>) -0.7 = -0.8
    assert LO.arpa_sentence_log10(lm, tok("ab ")) == pytest.approx(-1.8, abs=1e-6)
    # "ba":  p(b|<s>) -1.1 + p(a|<s> b) -0.2 + p(</s>|b a): bow(b a) 0 + p(</s>|a) -0.8
    assert LO.arpa_sentence_log10(lm, tok("ba")) == pytest.approx(-2.1, abs=1e-6)
    # "ac":  -0.3 + p(<unk>|<s> a) -1.55 + p(</s>|a <unk>) -0.7
    assert LO.arpa_sentence_log10(lm, tok("ac")) == pytest.approx(-2.55, abs=1e-6)
    # "": p(</s>|<s>): (<s> </s>) unlisted -> bow(<s>) -0.5 + p(</s>) -0.7
    assert LO.arpa_sentence_log10(lm, []) == pytest.approx(-1.2, abs=1e-6)


def test_id_beyond_the_alphabet_is_unk(hand):
    """class 5 lies beyond "ab c": the search scores it as <unk>, like class 4 (c, missing from the LM)"""
    lp = np.full((2, 6), -20.0, dtype=np.float32)
    lp[0, 1] = 0.0                                            # "a" then class 5 (or 4)
    for c in (4, 5):
        x = lp.copy()
        x[1, c] = 0.0
        (lab, fused, ctc), = LO.ctc_prefix_beam_search_lm(x, 1, hand, 1.0, 0.0)
        assert lab == [1, c]
        assert fused - ctc == pytest.approx(LO.LN10 * (-0.3 - 1.55 - 0.7), abs=1e-5)


def test_no_unk_unigram_gets_minus_100(tmp_path):
    text = HAND_ARPA.replace("ngram 1=6", "ngram 1=5").replace("-1.0\t<unk>\n", "")
    lm = LO.arpa_load(_write(tmp_path, text), ALPHABET)
    assert LO.arpa_logprob(lm, ("<s>",), "<unk>") == pytest.approx(-0.5 - 100.0, abs=1e-5)
    L = _lmmod()
    order, counts, table, tmap, kept = L.CharNGramLM.host_tables(_write(tmp_path, text, "b.arpa"), _converter(ALPHABET))
    lo, hi = L.pack_keys(np.array([[L.UNK]]))
    idx = L.table_find(table, lo, hi)
    assert idx[0] >= 0 and L.table_values(table, idx)[0][0] == np.float32(-100.0)


@pytest.mark.parametrize("bad", [
    ("ngram 2=5", "ngram 2=4"),                                   # counts that do not match
    ("\\3-grams:\n-0.1\t<s> a b\n-0.35\ta b a\n\n", ""),          # a missing section
    ("\\end\\", ""),                                              # no \end\
    ("\\data\\", "\\dada\\"),                                     # no \data\
    ("-0.5\ta b\t-0.15", "-0.5\ta b\t-0.15\t7"),                   # a line with too many fields
    ("-0.5\ta b\t-0.15", "x\ta b\t-0.15"),                        # a value that is not a number
    ("-0.5\ta b\t-0.15", "nan\ta b\t-0.15"),                      # a non-finite value
])
def test_malformed_files_are_refused(tmp_path, bad):
    text = HAND_ARPA.replace(*bad)
    assert text != HAND_ARPA
    path = _write(tmp_path, text)
    with pytest.raises(ValueError):
        LO.arpa_load(path, ALPHABET)
    with pytest.raises(ValueError):
        _lmmod().CharNGramLM.from_arpa(path, _converter(ALPHABET))


def test_order_above_8_is_refused(tmp_path):
    lines = ["\\data\\"] + ["ngram %d=1" % k for k in range(1, 10)] + [""]
    for k in range(1, 10):
        lines += ["\\%d-grams:" % k, "-0.5\t" + " ".join(["a"] * k), ""]
    path = _write(tmp_path, "\n".join(lines + ["\\end\\", ""]))
    with pytest.raises(ValueError):
        LO.arpa_load(path, ALPHABET)
    with pytest.raises(ValueError):
        _lmmod().parse_arpa(path)
    # order 8 is accepted
    lines = ["\\data\\"] + ["ngram %d=1" % k for k in range(1, 9)] + [""]
    for k in range(1, 9):
        lines += ["\\%d-grams:" % k, "-0.5\t" + " ".join(["a"] * k), ""]
    path = _write(tmp_path, "\n".join(lines + ["\\end\\", ""]), "ok.arpa")
    assert LO.arpa_load(path, ALPHABET)["order"] == 8 and _lmmod().parse_arpa(path)[0] == 8


@pytest.mark.parametrize("T,C,alphabet", [(3, 3, "ab"), (2, 4, "ab "), (5, 2, "a"), (3, 3, "a"), (2, 4, "ac")])
@pytest.mark.parametrize("alpha,beta", [(0.7, 0.0), (1.5, 2.0), (0.3, -1.0)])
def test_fused_search_equals_brute_force(tmp_path, T, C, alphabet, alpha, beta):
    """A beam that holds every prefix: every labelling's fused score is its brute-force CTC log-prob + alpha ln10
    log10 P(l </s>) + beta |l|, its ctc score the brute-force value, and the order is the fused order."""
    lm = LO.arpa_load(_write(tmp_path, HAND_ARPA), alphabet)
    rs = np.random.RandomState(T * 10 + C)
    x = rs.randn(T, C).astype(np.float32) * 1.5
    lp = torch.from_numpy(x).log_softmax(-1).numpy()
    exact = O.labelling_logprobs_bruteforce(lp)
    assert len(exact) <= 16
    got = LO.ctc_prefix_beam_search_lm(lp, 16, lm, alpha, beta)
    assert set(exact) <= set(tuple(g[0]) for g in got)
    toks = lm["tokens"]
    for lab, fused, ctc in got:
        if tuple(lab) not in exact:                           # no alignment of T frames spells it
            assert ctc == -math.inf and fused == -math.inf
            continue
        assert ctc == pytest.approx(exact[tuple(lab)], abs=1e-9)
        words = [toks[c] if c < len(toks) else "<unk>" for c in lab]
        want = exact[tuple(lab)] + alpha * LO.LN10 * LO.arpa_sentence_log10(lm, words) + beta * len(lab)
        assert fused == pytest.approx(want, abs=1e-9)
    fs = [g[1] for g in got]
    assert fs == sorted(fs, reverse=True)


@pytest.mark.parametrize("T,C,K", [(20, 6, 5), (12, 4, 16), (30, 9, 3), (1, 5, 4)])
def test_zero_weights_reproduce_the_plain_search(tmp_path, T, C, K):
    lm = LO.arpa_load(_write(tmp_path, HAND_ARPA), "ab c")
    rs = np.random.RandomState(T + C + K)
    x = rs.randn(T, C).astype(np.float32) * 2.0
    x[::3] = np.round(x[::3] * 2) / 2
    lp = torch.from_numpy(x).log_softmax(-1).numpy()
    want = O.ctc_prefix_beam_search(lp, K)
    got = LO.ctc_prefix_beam_search_lm(lp, K, lm, 0.0, 0.0)
    assert [g[0] for g in got] == [w[0] for w in want]
    assert [g[1] for g in got] == [w[1] for w in want] and [g[2] for g in got] == [w[1] for w in want]


def test_table_packing_exact_keys():
    """Every packed n-gram is found with its float32 values; 10^4 random absent keys (many sharing hash slots and
    fields with present ones) are not found."""
    L = _lmmod()
    rs = np.random.RandomState(5)
    keys = set()
    for k in range(1, 9):
        for _ in range(400):
            keys.add(tuple(int(v) for v in rs.randint(0, 12, size=k)))
    keys = sorted(keys)
    lo = np.concatenate([L.pack_keys(np.array([kk]))[0] for kk in keys])
    hi = np.concatenate([L.pack_keys(np.array([kk]))[1] for kk in keys])
    p = rs.uniform(-5, 0, size=len(keys))
    b = rs.uniform(-1, 0, size=len(keys))
    table = L.pack_table(lo, hi, p, b)
    slots = table.shape[0]
    assert slots & (slots - 1) == 0 and slots >= 2 * len(keys)
    assert (table[:, 0] != 0).sum() == len(keys)
    idx = L.table_find(table, lo, hi)
    assert (idx >= 0).all() and len(set(idx.tolist())) == len(keys)
    vp, vb = L.table_values(table, idx)
    np.testing.assert_array_equal(vp, p.astype(np.float32))
    np.testing.assert_array_equal(vb, b.astype(np.float32))
    absent = []
    while len(absent) < 10000:
        kk = tuple(int(v) for v in rs.randint(0, 14, size=rs.randint(1, 9)))
        if kk not in keys:
            absent.append(kk)
    alo = np.concatenate([L.pack_keys(np.array([kk]))[0] for kk in absent])
    ahi = np.concatenate([L.pack_keys(np.array([kk]))[1] for kk in absent])
    assert (L.table_find(table, alo, ahi) == -1).all()


def test_loader_table_matches_the_oracle_dicts(tmp_path):
    """CharNGramLM's packed table and token map against the oracle's dicts on the hand 3-gram: same n-grams (those
    over the alphabet and the specials), same float32 values; c and ids beyond the alphabet map to <unk>."""
    L = _lmmod()
    path = _write(tmp_path, HAND_ARPA.replace("-0.2\tb a\n", "-0.2\tb a\n-0.6\tb x\n").replace("ngram 2=5", "ngram 2=6"))
    ref = LO.arpa_load(path, ALPHABET)
    order, counts, table, tmap, kept = L.CharNGramLM.host_tables(path, _converter(ALPHABET))
    assert order == 3 and counts == [6, 6, 2] and kept == 13                # (b x) dropped
    assert tmap[4] == L.UNK and len(tmap) == 5 and len(set(tmap[1:4])) == 3
    name = {L.UNK: "<unk>", L.BOS: "<s>", L.EOS: "</s>"}
    for c in (1, 2, 3):
        name[tmap[c]] = ref["tokens"][c]
    ids = {v: k for k, v in name.items()}
    for t, p in ref["prob"].items():
        idx = L.table_find(table, *L.pack_keys(np.array([[ids.get(w, -1) for w in t]]))) if "x" not in t else None
        if idx is None:
            continue
        vp, vb = L.table_values(table, idx)
        assert idx[0] >= 0 and float(vp[0]) == p and float(vb[0]) == ref["bow"][t], t
