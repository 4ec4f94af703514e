"""Oracle of the lexicon-constrained CTC prefix beam search (htr-vt_b200/lexicon.py + the LEX instantiation of
csrc/prefix_beam.cu): plain Python, no import of the product and no trie: the state of a prefix is its trailing run of
word characters, checked against the set of all word prefixes.  Only tests import this file.  It restates
htrvt_lm_oracle.ctc_prefix_beam_search_lm (and, without an LM, htrvt_oracle.ctc_prefix_beam_search) with the same
candidate numbering and tie order, leaving out the candidates the lexicon forbids."""
from __future__ import annotations

import math

import numpy as np

from htrvt_lm_oracle import LN10, arpa_logprob
from htrvt_oracle import _lae


def accepted(labels, words, is_word):
    """every maximal run of word characters of labels is in words"""
    run = ()
    for c in list(labels) + [None]:
        if c is not None and c < len(is_word) and is_word[c]:
            run += (c,)
        else:
            if run and run not in words:
                return False
            run = ()
    return True


def ctc_prefix_beam_search_lex(log_probs: np.ndarray, beam_size: int, words, is_word, lm=None, alpha=0.0, beta=0.0):
    """-> [(label list, fused score, ctc score)], fused order (fused = ctc without an LM).  words: set of class-id
    tuples; is_word[c]: class c is a word character (ids beyond: free).  Between words (state ()) a free class keeps
    the state and a word class c needs (c,) to prefix a word; inside a word w a word class c needs w + (c,) to prefix a
    word, a free class needs w in words and returns to ().  In the last frame a candidate must end in () or a word."""
    T, C = log_probs.shape
    K = int(beam_size)
    prefixes = {w[:k] for w in words for k in range(1, len(w) + 1)}

    def free(c):
        return not (c < len(is_word) and is_word[c])

    def state(p):
        k = len(p)
        while k > 0 and not free(p[k - 1]):
            k -= 1
        return tuple(p[k:])

    def step(s, c):                                           # the state after c, or None when c is not allowed
        if free(c):
            return () if (not s or s in words) else None
        return s + (c,) if s + (c,) in prefixes else None

    def final(s):
        return not s or s in words

    toks = lm["tokens"] if lm is not None else []

    def tok(c):
        return toks[c] if c < len(toks) else "<unk>"

    rows = {}

    def row(p, lmp):
        if lm is None:
            return [0.0] * C, 0.0
        if p not in rows:
            ctx = ("<s>",) + tuple(tok(c) for c in p)
            r = [0.0] + [lmp + (alpha * (LN10 * arpa_logprob(lm, ctx, tok(c))) + beta) for c in range(1, C)]
            rows[p] = (r, alpha * (LN10 * arpa_logprob(lm, ctx, "</s>")))
        return rows[p]

    beam = [((), 0.0, -math.inf, 0.0)]
    for t in range(T):
        last = t + 1 == T
        lp = [float(v) for v in log_probs[t]]
        cand = {}                                             # prefix -> [pb', pnb', candidate number, lm, eligible]
        for i, (p, pb, pnb, lmp) in enumerate(beam):
            tot = _lae(pb, pnb)
            cand[p] = [tot + lp[0], (pnb + lp[p[-1]]) if p else -math.inf, i, lmp, not last or final(state(p))]
        for i, (p, pb, pnb, lmp) in enumerate(beam):
            tot = _lae(pb, pnb)
            r = row(p, lmp)[0]
            s = state(p)
            for c in range(1, C):
                v = (pb if (p and p[-1] == c) else tot) + lp[c]
                q = p + (c,)
                if q in cand:                                 # an entry of the beam: allowed, merged as before
                    cand[q][1] = _lae(cand[q][1], v)
                    continue
                s2 = step(s, c)
                if s2 is None or (last and not final(s2)):
                    continue
                cand[q] = [-math.inf, v, K + i * C + c, r[c], True]
        ranked = sorted(((-(_lae(v[0], v[1]) + v[3]), v[2], q, v[0], v[1], v[3]) for q, v in cand.items() if v[4]))
        beam = [(q, pb, pnb, lmq) for _, _, q, pb, pnb, lmq in ranked[:K]]
    out = []
    for q, pb, pnb, lmq in beam:
        ctc = _lae(pb, pnb)
        out.append((list(q), ctc if lm is None else (ctc + lmq) + row(q, lmq)[1], ctc))
    return sorted(out, key=lambda e: -e[1])
