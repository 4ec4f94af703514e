"""Oracle of the lexicon-constrained CTC prefix beam search with a word n-gram LM (htr-vt_b200/wordlm.py + the word-LM
instantiation of csrc/prefix_beam.cu): plain Python, no import of the product and no trie.  The state of a prefix is
its trailing run of word characters plus its finished words.  Only tests import this file.  It restates
htrvt_lex_oracle.ctc_prefix_beam_search_lex with the same candidate numbering and tie order; only the LM term
differs: words are the LM's tokens, scored when they end, and a word being spelled ranks with its smear term."""
from __future__ import annotations

import math

import numpy as np

from htrvt_lm_oracle import LN10, arpa_logprob
from htrvt_oracle import _lae

_SPECIALS = ("<unk>", "<s>", "</s>")


def word_token(lm, word):
    """the ARPA token of a lexicon word: itself when the file lists it as a unigram, else <unk>"""
    return word if (word,) in lm["prob"] and word not in _SPECIALS else "<unk>"


def unigram(lm, tok):
    """log10 p of the unigram tok (<unk>'s when the file lists no <unk>: -100)"""
    return lm["prob"].get((tok,), -100.0)


def words_of(labels, is_word):
    """the maximal runs of word characters of labels, in order, and the trailing (possibly unfinished) run"""
    out, run = [], ()
    for c in labels:
        if c < len(is_word) and is_word[c]:
            run += (c,)
        elif run:
            out.append(run)
            run = ()
    return out, run


def sentence_terms(lm, toks, alpha, beta):
    """(sum of alpha * (LN10 * log10 p(w | <s> previous)) + beta over toks, in order; alpha * (LN10 * log10 p(</s> |
    <s> toks)))"""
    done, ctx = 0.0, ("<s>",)
    for w in toks:
        done = done + (alpha * (LN10 * arpa_logprob(lm, ctx, w)) + beta)
        ctx = ctx + (w,)
    return done, alpha * (LN10 * arpa_logprob(lm, ctx, "</s>"))


def ctc_prefix_beam_search_wordlm(log_probs: np.ndarray, beam_size: int, words, is_word, alphabet, lm, alpha, beta):
    """-> [(label list, fused score, ctc score)], fused order.  words: set of class-id tuples; is_word[c]: class c is a
    word character (ids beyond: free); alphabet[c - 1]: the character of class c (spells a word for the LM); lm: an
    htrvt_lm_oracle.arpa_load dict of word tokens.  Accepted labellings and candidates as the lexicon oracle.  Rank of
    a prefix: lae(pb', pnb') + done, done = sentence_terms(finished words)[0], plus alpha * (LN10 * smear(run)) while
    the trailing run is non-empty, smear(run) = the largest unigram log10 prob of the words that start with run.
    Survivors: fused = (lae(pb, pnb) + done) + eos with eos = completion(run) + </s> term (a finished last word) or the
    </s> term (between words), re-ranked stably."""
    T, C = log_probs.shape
    K = int(beam_size)
    prefixes = {w[:k] for w in words for k in range(1, len(w) + 1)}
    tok_of = {w: word_token(lm, "".join(alphabet[c - 1] for c in w)) for w in words}
    smear = {}
    for w in words:
        p = float(np.float32(unigram(lm, tok_of[w])))
        for k in range(1, len(w) + 1):
            smear[w[:k]] = max(smear.get(w[:k], -math.inf), p)

    def free(c):
        return not (c < len(is_word) and is_word[c])

    def state(p):
        k = len(p)
        while k > 0 and not free(p[k - 1]):
            k -= 1
        return tuple(p[k:])

    def step(s, c):
        if free(c):
            return () if (not s or s in words) else None
        return s + (c,) if s + (c,) in prefixes else None

    def final(s):
        return not s or s in words

    memo = {}

    def terms(toks):                                          # sentence_terms, memoised on the token tuple
        if toks not in memo:
            memo[toks] = sentence_terms(lm, list(toks), alpha, beta)
        return memo[toks]

    def rank_lm(p):
        fin, run = words_of(p, is_word)
        d = terms(tuple(tok_of[w] for w in fin))[0]
        return d + alpha * (LN10 * smear[run]) if run else d

    def end_terms(p):                                         # (done, eos) of a prefix that may end the line
        fin, run = words_of(p, is_word)
        toks = tuple(tok_of[w] for w in fin)
        d, e = terms(toks)
        if run:
            comp = alpha * (LN10 * arpa_logprob(lm, ("<s>",) + toks, tok_of[run])) + beta
            e = comp + terms(toks + (tok_of[run],))[1]
        return d, e

    beam = [((), 0.0, -math.inf)]
    for t in range(T):
        last = t + 1 == T
        lp = [float(v) for v in log_probs[t]]
        cand = {}                                             # prefix -> [pb', pnb', candidate number, eligible]
        for i, (p, pb, pnb) in enumerate(beam):
            tot = _lae(pb, pnb)
            cand[p] = [tot + lp[0], (pnb + lp[p[-1]]) if p else -math.inf, i, not last or final(state(p))]
        for i, (p, pb, pnb) in enumerate(beam):
            tot = _lae(pb, pnb)
            s = state(p)
            for c in range(1, C):
                v = (pb if (p and p[-1] == c) else tot) + lp[c]
                q = p + (c,)
                if q in cand:
                    cand[q][1] = _lae(cand[q][1], v)
                    continue
                s2 = step(s, c)
                if s2 is None or (last and not final(s2)):
                    continue
                cand[q] = [-math.inf, v, K + i * C + c, True]
        ranked = sorted(((-(_lae(v[0], v[1]) + rank_lm(q)), v[2], q, v[0], v[1]) for q, v in cand.items() if v[3]))
        beam = [(q, pb, pnb) for _, _, q, pb, pnb in ranked[:K]]
    out = []
    for q, pb, pnb in beam:
        ctc = _lae(pb, pnb)
        d, eos = end_terms(q)
        out.append((list(q), (ctc + d) + eos, ctc))
    return sorted(out, key=lambda e: -e[1])
