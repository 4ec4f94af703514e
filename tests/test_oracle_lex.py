"""CPU: the lexicon-constrained CTC prefix beam search - the oracle against the brute-force labelling posterior
filtered to the accepted language, an empty word-character set against the plain and LM searches, hand cases (the
last-frame rule, a doubled letter inside a word, a run of free characters between words), and the host-side packing
of the trie (htr-vt_b200/lexicon.py)."""
import math
from importlib import import_module

import numpy as np
import pytest
import torch

import htrvt_lex_oracle as XO
import htrvt_lm_oracle as LO
import htrvt_oracle as O
from test_oracle_lm import ALPHABET, HAND_ARPA


def _lexmod():
    import htrvt_b200  # noqa: F401
    return import_module("htr-vt_b200.lexicon")


def _converter(alphabet):
    import htrvt_b200 as h
    return h.CTCLabelConverter(alphabet, device="cpu")


def _lp(T, C, seed, scale=1.5):
    x = np.random.RandomState(seed).randn(T, C).astype(np.float32) * scale
    return torch.from_numpy(x).log_softmax(-1).numpy()


# classes 1, 2 are word characters, 3 is free (the space); words "a", "ab", "ba", "bb"
WORDS = {(1,), (1, 2), (2, 1), (2, 2)}
IS_WORD = [0, 1, 1, 0]


@pytest.mark.parametrize("T,C", [(2, 3), (3, 3), (3, 4), (4, 4), (5, 3)])
def test_wide_beam_is_the_filtered_posterior(T, C):
    """K wider than the number of prefixes: the oracle returns exactly the accepted labellings with their exact
    posterior, best first (labellings no alignment reaches, such as "bb" in two frames, carry -inf)"""
    for seed in range(3):
        lp = _lp(T, C, 10 * T + C + seed)
        exact = {k: v for k, v in O.labelling_logprobs_bruteforce(lp).items() if XO.accepted(k, WORDS, IS_WORD)}
        got = [e for e in XO.ctc_prefix_beam_search_lex(lp, 200, WORDS, IS_WORD) if e[2] > -math.inf]
        assert {tuple(lab) for lab, _, _ in got} == set(exact)
        for lab, fused, ctc in got:
            assert fused == ctc and abs(ctc - exact[tuple(lab)]) < 1e-9
        assert [f for _, f, _ in got] == sorted((f for _, f, _ in got), reverse=True)


def test_accepted():
    assert XO.accepted([], WORDS, IS_WORD)
    assert XO.accepted([1, 3, 2, 2, 3, 3], WORDS, IS_WORD)
    assert not XO.accepted([2], WORDS, IS_WORD)                  # "b" is only a prefix
    assert not XO.accepted([1, 2, 1], WORDS, IS_WORD)            # "aba": no free character between the words
    assert XO.accepted([3, 7, 3], WORDS, IS_WORD)                # ids beyond is_word are free


@pytest.mark.parametrize("T,C,K", [(6, 4, 3), (9, 5, 5), (12, 6, 8), (7, 4, 1)])
def test_no_word_characters_is_the_plain_and_lm_search(tmp_path, T, C, K):
    lp = _lp(T, C, T * C + K, scale=2.0)
    plain = O.ctc_prefix_beam_search(lp, K)
    got = XO.ctc_prefix_beam_search_lex(lp, K, {(1, 2)}, [0] * C)
    assert [(lab, c) for lab, _, c in got] == plain
    assert all(f == c for _, f, c in got)
    path = tmp_path / "hand3.arpa"
    path.write_text(HAND_ARPA, encoding="utf-8")
    lm = LO.arpa_load(str(path), ALPHABET)
    for alpha, beta in ((0.7, 0.0), (1.5, 2.0)):
        assert XO.ctc_prefix_beam_search_lex(lp, K, set(), [0] * C, lm, alpha, beta) == \
            LO.ctc_prefix_beam_search_lm(lp, K, lm, alpha, beta)


def _peaked(rows, C):
    """one frame per entry of rows: that class at probability 0.9, the rest shared"""
    p = np.full((len(rows), C), 0.1 / (C - 1))
    for t, c in enumerate(rows):
        p[t, c] = 0.9
    return np.log(p).astype(np.float32)


def test_last_frame_rule():
    """"b" then blank: "b" alone is only the prefix of "ba" / "bb", so the line cannot end on it; inside the line the
    same prefix survives (T = 3 with an "a" after it gives "ba")"""
    lp = _peaked([2, 0], 4)
    got = XO.ctc_prefix_beam_search_lex(lp, 4, WORDS, IS_WORD)
    assert all(XO.accepted(lab, WORDS, IS_WORD) for lab, _, _ in got)
    assert [2] not in [lab for lab, _, _ in got] and got[0][0] != [2]
    assert XO.ctc_prefix_beam_search_lex(_peaked([2, 0, 1], 4), 4, WORDS, IS_WORD)[0][0] == [2, 1]
    # K = 1 and a last frame that leaves every candidate mid-word: no accepted labelling at all
    words = {(1, 2, 1)}
    assert XO.ctc_prefix_beam_search_lex(_peaked([1, 2], 4), 1, words, [0, 1, 1, 0]) == []


def test_doubled_letter_inside_a_word():
    """"ll" needs a blank between the two l; the lexicon holds "all" (classes a = 1, l = 2)"""
    words = {(1, 2, 2)}
    lp = _peaked([1, 2, 0, 2], 4)
    got = XO.ctc_prefix_beam_search_lex(lp, 8, words, [0, 1, 1, 0])
    assert got[0][0] == [1, 2, 2]
    assert all(XO.accepted(lab, words, [0, 1, 1, 0]) for lab, _, _ in got)
    assert [1, 2] not in [lab for lab, _, _ in got]               # "al" is no word


def test_free_run_between_words():
    """"ab", two spaces, "ba": a run of free characters between words is free"""
    lp = _peaked([1, 2, 3, 0, 3, 2, 1], 4)
    got = XO.ctc_prefix_beam_search_lex(lp, 8, WORDS, IS_WORD)
    assert got[0][0] == [1, 2, 3, 3, 2, 1]


# ---- host packing -------------------------------------------------------------------------------------------------
def test_pack_trie_hand():
    first, label, child, end = _lexmod().pack_trie([(1, 2), (1,), (2, 1), (1, 3)])
    # breadth first: 0 root; 1 = a, 2 = b; 3 = ab, 4 = ac, 5 = ba
    assert first.tolist() == [0, 2, 4, 5, 5, 5, 5]
    assert label.tolist() == [1, 2, 2, 3, 1]
    assert child.tolist() == [1, 2, 3, 4, 5]
    assert end.tolist() == [0, 1, 0, 1, 1, 1]
    assert first.dtype == np.int32 and label.dtype == np.int32 and end.dtype == np.uint8


def test_host_tables_skips_and_merges():
    L = _lexmod().Lexicon
    conv = _converter("abc .")
    first, label, child, end, is_word, n_words, n_skipped, wc = L.host_tables(
        ["ab", " ab ", "", "  ", "ba", "aé", "c"], conv)
    assert (n_words, n_skipped) == (3, 1)                         # ab (twice), ba, c; aé is outside the alphabet
    assert wc == "abc" and is_word.tolist() == [0, 1, 1, 1, 0, 0]
    assert len(end) == 1 + 3 + 2 and end.sum() == 3
    # an explicit word_chars: words with a free character are skipped too
    _, _, _, end, is_word, n_words, n_skipped, wc = L.host_tables(["ab", "a.b", "c"], conv, word_chars="ab")
    assert (n_words, n_skipped, wc) == (1, 2, "ab") and is_word.tolist() == [0, 1, 1, 0, 0, 0]
    # no word character at all: an empty trie
    first, label, child, end, is_word, n_words, n_skipped, wc = L.host_tables(["ab"], conv, word_chars="")
    assert (n_words, n_skipped, wc, first.tolist(), len(label)) == (0, 1, "", [0, 0], 0) and not is_word.any()


def test_from_file_errors(tmp_path):
    L = _lexmod().Lexicon
    conv = _converter("ab ")
    p = tmp_path / "words.txt"
    p.write_text("\n  \n", encoding="utf-8")
    with pytest.raises(ValueError):
        L.file_tables(str(p), conv)
    p.write_text("xyz\nzz\n", encoding="utf-8")
    with pytest.raises(ValueError):
        L.file_tables(str(p), conv)
    p.write_text("ab\n ba \nab\n", encoding="utf-8")
    t = L.file_tables(str(p), conv)
    assert t[5:] == (2, 0, "ab")
    with pytest.raises(FileNotFoundError):
        L.file_tables(str(tmp_path / "missing.txt"), conv)


def test_check_trie_refuses_bad_tries():
    m = _lexmod()
    first, label, child, end = m.pack_trie([(1, 2), (2,)])
    m.check_trie(first, label, child, end)
    with pytest.raises(ValueError):
        m.check_trie(first, label[::-1].copy(), child, end)
    with pytest.raises(ValueError):
        m.check_trie(first, label, child + 5, end)
    with pytest.raises(ValueError):
        m.check_trie(first[:-1], label, child, end)


def test_random_lexicons_pack_consistently():
    """every packed word is found by walking the trie, and nothing else ends a word"""
    m = _lexmod()
    rs = np.random.RandomState(3)
    words = {tuple(rs.randint(1, 6, size=rs.randint(1, 6))) for _ in range(300)}
    first, label, child, end = m.pack_trie(words)
    m.check_trie(first, label, child, end)
    found = set()

    def walk(n, w):
        if end[n]:
            found.add(w)
        for j in range(first[n], first[n + 1]):
            walk(child[j], w + (int(label[j]),))
    walk(0, ())
    assert found == words
    assert len(end) == 1 + len({w[:k] for w in words for k in range(1, len(w) + 1)})
