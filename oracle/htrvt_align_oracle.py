"""Float64 restatement of CTC forced alignment (csrc/ctc_align.cu), blank = 0.

ctc_viterbi_align(lp[T, C], labels) is the Viterbi path of the labels through the CTC trellis:
  states S = 2L + 1, ext[2k] = 0, ext[2k+1] = labels[k];
  d_0(0) = lp(0, 0), d_0(1) = lp(0, labels[0]), every other state -inf;
  d_t(s) = m + lp(t, ext[s]), m = max(c0, c1, c2): c0 = d_{t-1}(s), c1 = d_{t-1}(s-1) (s >= 1),
           c2 = d_{t-1}(s-2) (s >= 2, ext[s] != 0, ext[s] != ext[s-2]);
  the back-pointer is the FIRST of c0, c1, c2 equal to m (stay, previous, skip) - a true maximum, where torchaudio's
  forced_align can return a path below it on exact ties;
  one float64 add per state per frame (the fp32 input widened), after the max;
  the path ends in S-1 if d(S-1) > d(S-2), else in S-2.
Vectorised over states with numpy, so it runs at T = 1024, L = 256.
"""
import collections

import numpy as np

MAX_LABELS = 256

Alignment = collections.namedtuple("Alignment", "path frame_scores spans token_scores score status")


def _fail(T, L, status):
    return Alignment(np.full(T, -1, np.int64), np.zeros(T, np.float32), np.full((L, 2), -1, np.int64),
                     np.zeros(L, np.float32), -np.inf, status)


def ctc_viterbi_align(lp, labels, input_length=None):
    """lp: [T, C] log-probs (or raw logits: the path is the same, the scores are then raw); labels: L ids in [1, C);
    input_length: frames of the line (default T).  Returns Alignment:
      path int [T] (class per frame, -1 beyond input_length), frame_scores float32 [T] (lp of that class, 0 beyond),
      spans int [L, 2] ([start, end) frames of label k), token_scores float32 [L] (float64 sum of the span's frame
      scores in frame order), score float64, status (0 aligned, 1 infeasible, 2 invalid line data).
    Failed lines: path and spans -1, scores 0, score -inf."""
    lp = np.asarray(lp, dtype=np.float64)
    T, C = lp.shape
    labels = np.asarray(labels, dtype=np.int64).reshape(-1)
    L = labels.size
    Tb = T if input_length is None else int(input_length)
    if Tb < 0 or Tb > T or L > MAX_LABELS or (L and (labels.min() < 1 or labels.max() >= C)):
        return _fail(T, L, 2)
    repeats = int(np.count_nonzero(labels[1:] == labels[:-1])) if L > 1 else 0
    if Tb < L + repeats:
        return _fail(T, L, 1)
    path = np.full(T, -1, np.int64)
    frame_scores = np.zeros(T, np.float32)
    if Tb == 0:
        return Alignment(path, frame_scores, np.zeros((0, 2), np.int64), np.zeros(0, np.float32), 0.0, 0)

    S = 2 * L + 1
    ext = np.zeros(S, np.int64)
    ext[1::2] = labels
    skip = np.zeros(S, bool)
    skip[3::2] = labels[1:] != labels[:-1]
    em = lp[:Tb, ext]                                  # [Tb, S]
    d = np.full(S, -np.inf)
    d[0] = em[0, 0]
    if S > 1:
        d[1] = em[0, 1]
    bp = np.zeros((Tb, S), np.int8)
    neg = np.full(2, -np.inf)
    for t in range(1, Tb):
        c0 = d
        c1 = np.concatenate((neg[:1], d[:-1]))
        c2 = np.concatenate((neg, d[:-2]))[:S]
        c2 = np.where(skip, c2, -np.inf)
        m = np.maximum(np.maximum(c0, c1), c2)
        # the first of c0, c1, c2 that equals the maximum (a state with every candidate -inf stays)
        bp[t] = np.where(c0 == m, 0, np.where(c1 == m, 1, 2))
        d = m + em[t]
    if S >= 2 and not d[S - 1] > d[S - 2]:
        s = S - 2
    else:
        s = S - 1
    score = float(d[s])
    states = np.empty(Tb, np.int64)
    for t in range(Tb - 1, -1, -1):
        states[t] = s
        if t > 0:
            s -= int(bp[t, s])
    path[:Tb] = ext[states]
    frame_scores[:Tb] = lp[np.arange(Tb), path[:Tb]]
    spans = np.full((L, 2), -1, np.int64)
    token_scores = np.zeros(L, np.float32)
    fs64 = lp[np.arange(Tb), path[:Tb]].astype(np.float32).astype(np.float64)
    for k in range(L):
        frames = np.nonzero(states == 2 * k + 1)[0]
        spans[k] = frames[0], frames[-1] + 1
        acc = 0.0
        for v in fs64[frames[0]:frames[-1] + 1]:         # sequential, in frame order
            acc += float(v)
        token_scores[k] = np.float32(acc)
    return Alignment(path, frame_scores, spans, token_scores, score, 0)


def collapse(path):
    """Labels a CTC path spells: repeats merged, blanks (0) dropped, -1 padding ignored."""
    out, prev = [], 0
    for c in path:
        c = int(c)
        if c < 0:
            break
        if c != 0 and c != prev:
            out.append(c)
        prev = c
    return out
