"""Oracle of the LM-fused CTC prefix beam search (htr-vt_b200/lm.py + the LM instantiation of csrc/prefix_beam.cu):
plain numpy / Python, no import of the product.  Only tests import this file; the product never does.  It extends
htrvt_oracle.ctc_prefix_beam_search (the search without the language-model term) and shares its log-add-exp."""
from __future__ import annotations

import math

import numpy as np

from htrvt_oracle import _lae

# ----------------------------------------------------------------------------------------------
# CTC prefix beam search with a character n-gram LM inside the search (Hannun et al. 2014, algorithm 1 WITH the LM
# term; what model_window/test_with_kenlm.py:25-59 does after the search, with KenLM's score(bos=True, eos=True)).
# The ARPA backoff model restated from the format's definition on plain dicts of token tuples, independent of the
# product's packed table.  Values are rounded to float32 (KenLM stores floats) and summed in float64.
# ----------------------------------------------------------------------------------------------
LN10 = 2.302585092994046


def arpa_load(path, alphabet, space_token="<space>"):
    """ARPA file -> {"order", "counts", "prob": {token tuple: log10 p}, "bow": {token tuple: log10 bow}, "tokens":
    [class id -> ARPA token]}.  Class c >= 1 is alphabet[c - 1] (the space spelled space_token); an alphabet character
    the file does not list as a unigram is "<unk>".  ValueError on a malformed file (no \\data\\ or counts, order > 8,
    a missing \\k-grams: section, counts that do not match, a bad line or value, no \\end\\)."""
    with open(path, encoding="utf-8") as fh:
        lines = [ln.strip() for ln in fh.read().splitlines()]
    if "\\data\\" not in lines:
        raise ValueError("no \\data\\")
    i = lines.index("\\data\\") + 1
    counts = {}
    while i < len(lines) and (lines[i].startswith("ngram ") or not lines[i]):
        if lines[i]:
            k, v = lines[i][6:].split("=")
            counts[int(k)] = int(v)
        i += 1
    order = max(counts) if counts else 0
    if order < 1 or sorted(counts) != list(range(1, order + 1)):
        raise ValueError("bad counts")
    if order > 8:
        raise ValueError("order above 8")
    prob, bow = {}, {}
    for k in range(1, order + 1):
        if i >= len(lines) or lines[i] != "\\%d-grams:" % k:
            raise ValueError("missing \\%d-grams:" % k)
        i += 1
        n = 0
        while i < len(lines) and not lines[i].startswith("\\"):
            if lines[i]:
                f = lines[i].split()
                if len(f) not in (k + 1, k + 2):
                    raise ValueError("bad line")
                t = tuple(f[1:k + 1])
                p = float(f[0])
                if t == ("<s>",) and not math.isfinite(p):
                    p = -99.0
                b = float(f[k + 1]) if len(f) == k + 2 else 0.0
                if not (math.isfinite(p) and math.isfinite(b)):
                    raise ValueError("non-finite value")
                prob[t] = float(np.float32(p))
                bow[t] = float(np.float32(b))
                n += 1
            i += 1
        if n != counts[k]:
            raise ValueError("count mismatch")
    if i >= len(lines) or lines[i] != "\\end\\":
        raise ValueError("no \\end\\")
    tokens = ["<blank>"]
    for ch in alphabet:
        w = space_token if ch == " " else ch
        tokens.append(w if (w,) in prob and w not in ("<s>", "</s>", "<unk>") else "<unk>")
    return {"order": order, "counts": [counts[k] for k in range(1, order + 1)], "prob": prob, "bow": bow,
            "tokens": tokens}


def arpa_logprob(lm, context, w):
    """log10 p(w | context) by ARPA backoff, context = the whole history (starts with "<s>"), the last order-1 tokens
    used: the listed prob of the longest listed (context suffix, w), plus the bows of the longer suffixes (0 when
    unlisted); summed in float64 longest-suffix bow first, the found prob last; <unk>'s prob (-100 if unlisted) when w
    has no unigram."""
    h = tuple(context)[max(0, len(context) - (lm["order"] - 1)):] if lm["order"] > 1 else ()
    S = 0.0
    for m in range(len(h), -1, -1):
        hm = h[len(h) - m:]
        if hm + (w,) in lm["prob"]:
            return S + lm["prob"][hm + (w,)]
        if m > 0:
            S += lm["bow"].get(hm, 0.0)
    return S + lm["prob"].get(("<unk>",), -100.0)


def arpa_sentence_log10(lm, tokens):
    """log10 P(tokens </s>) from context <s> (KenLM's score(bos=True, eos=True))."""
    ctx, tot = ("<s>",), 0.0
    for w in list(tokens) + ["</s>"]:
        tot += arpa_logprob(lm, ctx, w)
        ctx = ctx + (w,)
    return tot


def ctc_prefix_beam_search_lm(log_probs: np.ndarray, beam_size: int, lm, alpha: float, beta: float):
    """ctc_prefix_beam_search with the LM inside the search -> [(label list, fused score, ctc score)], fused order.
    Entry = (prefix, pb, pnb, lm) with lm = sum over its labels of alpha * (LN10 * S) + beta, S = arpa_logprob of the
    label's token after the prefix's tokens (context <s> first); ids beyond lm["tokens"] are "<unk>".  Candidates rank
    by lae(pb', pnb') + lm' (ties by candidate number as in ctc_prefix_beam_search); an extension that spells an
    entry merges its CTC mass (lm unchanged).  At the end fused = (lae(pb, pnb) + lm) + alpha * (LN10 * S(</s>)), and
    the survivors are re-ranked by it, stably."""
    T, C = log_probs.shape
    K = int(beam_size)
    toks = lm["tokens"]

    def tok(c):
        return toks[c] if c < len(toks) else "<unk>"

    rows = {}                                                 # prefix -> [lm of prefix + c for every c], eos term

    def row(p, lmp):
        if p not in rows:
            ctx = ("<s>",) + tuple(tok(c) for c in p)
            r = [0.0] + [lmp + (alpha * (LN10 * arpa_logprob(lm, ctx, tok(c))) + beta) for c in range(1, C)]
            rows[p] = (r, alpha * (LN10 * arpa_logprob(lm, ctx, "</s>")))
        return rows[p]

    beam = [((), 0.0, -math.inf, 0.0)]
    for t in range(T):
        lp = [float(v) for v in log_probs[t]]
        cand = {}                                             # prefix -> [pb', pnb', candidate number, lm]
        for i, (p, pb, pnb, lmp) in enumerate(beam):
            tot = _lae(pb, pnb)
            cand[p] = [tot + lp[0], (pnb + lp[p[-1]]) if p else -math.inf, i, lmp]
        for i, (p, pb, pnb, lmp) in enumerate(beam):
            tot = _lae(pb, pnb)
            r = row(p, lmp)[0]
            for c in range(1, C):
                s = (pb if (p and p[-1] == c) else tot) + lp[c]
                q = p + (c,)
                if q in cand:
                    cand[q][1] = _lae(cand[q][1], s)
                else:
                    cand[q] = [-math.inf, s, K + i * C + c, r[c]]
        ranked = sorted(((-(_lae(v[0], v[1]) + v[3]), v[2], q, v[0], v[1], v[3]) for q, v in cand.items()))
        beam = [(q, pb, pnb, lmq) for _, _, q, pb, pnb, lmq in ranked[:K]]
    out = []
    for q, pb, pnb, lmq in beam:
        ctc = _lae(pb, pnb)
        out.append((list(q), (ctc + lmq) + row(q, lmq)[1], ctc))
    return sorted(out, key=lambda e: -e[1])


