"""LM-rescored CTC decoding with the reference's contract (model_window/test_with_kenlm.py:25-59).

`simple_ctc_beam_search_with_lm(log_probs[T,C], converter, lm_scorer, beam_size=5) -> str` keeps the reference's
signature and result; the per-frame beam (T * K^2 Python list operations and a D2H copy per frame per line in the
reference) runs as one kernel for the whole batch (csrc/beam.cu), one D2H copy brings back the K collapsed candidate
id rows per line, and only what must stay on the host stays there: id -> char and `lm_scorer.score(text)` (KenLM in
the reference; any object with a `.score(str) -> float` method).
`beam_search_with_lm_batch(preds_log[T,B,C], ...) -> list[str]` is the loop of validation_with_kenlm (:85-88).

`search="prefix"` (all three entry points) swaps the candidate generator for a true CTC prefix beam search
(csrc/prefix_beam.cu, SURVEY.md 8(f) row 4): the K candidates are the K most probable LABELLINGS, each scored with the
summed probability of all its alignments, instead of the K best single alignment paths (which usually collapse to two
or three distinct strings).  The default `search="paths"` is the reference's behaviour, bit for bit.

`kbest_candidates(..., search="prefix", lm=CharNGramLM, alpha=, beta=)` and `ctc_lm_decode` put a character n-gram LM
inside the prefix search (lm.py, csrc/prefix_beam.cu): every extension is ranked by CTC log-prob + alpha * ln(10) *
log10 p(char | context) + beta, and the line's end adds the </s> term, so the LM shapes which labellings survive
instead of only picking among the K the acoustic model kept.

`kbest_candidates(..., search="prefix", lexicon=Lexicon)` and `ctc_lexicon_decode` constrain that search to a word
lexicon (lexicon.py, csrc/prefix_beam.cu): every word of a candidate comes from the list, with or without the LM.  The
LM may also be a word n-gram LM built on that lexicon (WordNGramLM, wordlm.py): every finished word is then scored by
alpha * ln(10) * log10 p(word | previous words) + beta inside the search.
"""
import numpy as np
import torch

from . import ops


def _candidate_strings(ids, lens, converter, merge_repeats=True):
    """converter.decode(np.array(text), [len(text)]) of the reference (utils.py:72-86) on every already collapsed id
    row at once: decode() filters blanks / repeats / out-of-alphabet ids AGAIN (so a doubled letter that survived the
    path collapse through a blank is merged here - reference behaviour, kept).  ids [R, T], lens [R] -> R strings.
    merge_repeats=False (prefix search): the rows are LABELLINGS, a doubled label is a doubled letter and stays."""
    R, T = ids.shape
    keep = (np.arange(T)[None, :] < lens[:, None]) & (ids != 0) & (ids < len(converter.character))
    if merge_repeats:
        keep[:, 1:] &= ids[:, 1:] != ids[:, :-1]
    counts = keep.sum(1)
    ends = np.cumsum(counts)
    kept = ids[keep]                                          # row-major: row 0's survivors, then row 1's ...
    table = converter.character
    if all(len(ch) == 1 for ch in table[1:]):                 # single code points: one UTF-32 decode for the batch
        lut = np.array([32] + [ord(ch) for ch in table[1:]], dtype=np.uint32)
        flat = lut[kept].astype("<u4", copy=False).tobytes().decode("utf-32-le")
        return [flat[e - c:e] for c, e in zip(counts.tolist(), ends.tolist())]
    kept = kept.tolist()
    return ["".join(table[i] for i in kept[e - c:e]) for c, e in zip(counts.tolist(), ends.tolist())]


def kbest_candidates(log_probs, converter, beam_size=5, lengths=None, layout="tbc", search="paths", lm=None,
                     alpha=None, beta=0.0, lexicon=None):
    """-> per line: list of (string, score) for the surviving beams with a non-empty string, in the reference's
    order (test_with_kenlm.py:42-53).  search: "paths" (the reference's per-frame path beam; score = path log-prob)
    or "prefix" (CTC prefix beam search; score = log-probability of the labelling).  lm (a CharNGramLM, prefix search
    only) with weight alpha and per-character bonus beta: the candidates come from the LM-fused search, in its order,
    and score = CTC log-prob + alpha * ln(10) * log10 P(string </s>) + beta * len.  lexicon (a Lexicon, prefix search
    only, with or without lm): only labellings whose every word is in the lexicon, ranked and scored as without it.
    With lexicon, lm may be a WordNGramLM built on it: score = CTC log-prob + alpha * ln(10) * log10 P(w_1 .. w_m
    </s>) + beta * m over the string's m words (a word LM without a lexicon is a ValueError)."""
    if search not in ("paths", "prefix"):
        raise ValueError("search must be 'paths' or 'prefix'")
    if lexicon is not None:
        if search != "prefix":
            raise ValueError("lexicon= needs search='prefix' (the path beam has no lexicon constraint)")
        if lm is not None and alpha is None:
            raise ValueError("lm= needs its weight alpha")
        if lm is None:
            alpha, beta = 0.0, 0.0
        ids, lens, scores, _ = ops.ctc_prefix_beam_lex(log_probs, beam_size, lexicon, lm, alpha, beta, lengths, layout)
    elif lm is not None:
        if search != "prefix":
            raise ValueError("lm= needs search='prefix' (the path beam has no LM term)")
        if alpha is None:
            raise ValueError("lm= needs its weight alpha")
        ids, lens, scores, _ = ops.ctc_prefix_beam_lm(log_probs, beam_size, lm, alpha, beta, lengths, layout)
    else:
        fn = ops.ctc_kbest_paths if search == "paths" else ops.ctc_prefix_beam
        ids, lens, scores = fn(log_probs, beam_size, lengths, layout)
    ids, lens, scores = ids.cpu().numpy(), lens.cpu().numpy(), scores.cpu().numpy()
    B, K, T = ids.shape
    strings = _candidate_strings(ids.reshape(B * K, T), np.maximum(lens.reshape(-1), 0), converter,
                                 merge_repeats=search == "paths")
    sc = scores.tolist()
    alive = (lens >= 0).tolist()
    return [[(strings[b * K + r], sc[b][r]) for r in range(K) if alive[b][r] and strings[b * K + r]] for b in range(B)]


def _pick(cands, lm_scorer):
    if not cands:
        return ""
    lm_scores = [lm_scorer.score(c[0]) for c in cands]
    return cands[int(np.argmax(lm_scores))][0]


def simple_ctc_beam_search_with_lm(log_probs, converter, lm_scorer, beam_size=5, search="paths"):
    """Reference signature: log_probs [T, C] of ONE line -> best string by LM score."""
    if not log_probs.is_cuda:
        raise ops.HtrvtError("simple_ctc_beam_search_with_lm needs a CUDA tensor (no CPU fallback)")
    lp = log_probs.float().unsqueeze(1)                       # [T, 1, C]
    return _pick(kbest_candidates(lp, converter, beam_size, search=search)[0], lm_scorer)


def _batch_log_probs(preds_log, name):
    """preds_log on the GPU as fp32 with a contiguous class axis."""
    if not preds_log.is_cuda:
        raise ops.HtrvtError("%s needs a CUDA tensor (no CPU fallback)" % name)
    lp = preds_log.float()
    return lp if lp.stride(-1) == 1 else lp.contiguous()


def _best_strings(ids, lens, converter):
    """The best-ranked labelling of every line of a prefix search's (ids, lens) as a string."""
    return _candidate_strings(ids[:, 0].cpu().numpy(), np.maximum(lens[:, 0].cpu().numpy(), 0), converter,
                              merge_repeats=False)


def beam_search_with_lm_batch(preds_log, converter, lm_scorer, beam_size=5, lengths=None, search="paths"):
    """preds_log [T, B, C] (validation_with_kenlm's `preds_log`) -> list of B strings: one kernel, one D2H copy."""
    lp = _batch_log_probs(preds_log, "beam_search_with_lm_batch")
    return [_pick(c, lm_scorer) for c in kbest_candidates(lp, converter, beam_size, lengths, search=search)]


def ctc_lm_decode(preds_log, converter, lm, alpha, beta=0.0, beam_size=8, lengths=None):
    """preds_log [T, B, C] (validation_with_kenlm's layout) -> B strings: the best-ranked labelling of the LM-fused CTC
    prefix beam search per line ("" when that is the empty labelling).  lm: CharNGramLM on the same device."""
    lp = _batch_log_probs(preds_log, "ctc_lm_decode")
    ids, lens, _, _ = ops.ctc_prefix_beam_lm(lp, beam_size, lm, alpha, beta, lengths, "tbc")
    return _best_strings(ids, lens, converter)


def ctc_lexicon_decode(preds_log, converter, lexicon, beam_size=8, lengths=None, lm=None, alpha=0.0, beta=0.0):
    """preds_log [T, B, C] (validation_with_kenlm's layout) -> B strings: the best-ranked labelling per line of the CTC
    prefix beam search constrained to lexicon (a Lexicon on the same device), with lm (weights alpha, beta) fused in
    when given ("" for the empty labelling, and for a line with no accepted labelling).  lm: a CharNGramLM (score =
    CTC log-prob + alpha * ln(10) * log10 P(string </s>) + beta * len) or a WordNGramLM built on lexicon (score = CTC
    log-prob + alpha * ln(10) * log10 P(w_1 .. w_m </s>) + beta * m over the string's m words)."""
    lp = _batch_log_probs(preds_log, "ctc_lexicon_decode")
    ids, lens, _, _ = ops.ctc_prefix_beam_lex(lp, beam_size, lexicon, lm, alpha, beta, lengths, "tbc")
    return _best_strings(ids, lens, converter)
