"""Record tests/golden/align_cases.npz from torchaudio.functional.forced_align (blank = 0, one line per call).

Tie-free cases (continuous random log-probs): `lp_i` fp32 [T, C], `lab_i` int32 [L], torchaudio's `ta_path_i` int32 [T]
and `ta_scores_i` fp32 [T].  They cover repeated labels, L = 1, lines with a single feasible alignment
(T = L + repeats) and T up to 256.

Tie cases (log-probs quantised to 0.5, T <= 7, C <= 4) where torchaudio's path scores BELOW the true maximum:
`qlp_j`, `qlab_j`, `qta_path_j`, the float64 score of torchaudio's path `qta_score_j` and the true maximum over all
C^T paths that collapse to the labels, `qmax_j` (brute force, independent of the oracle).  The tests pin that the
oracle does not copy torchaudio there.

Usage: python oracle/make_align_golden.py   (needs torchaudio; the tests do not)
"""
import itertools
import os

import numpy as np
import torch
import torchaudio.functional as taF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "align_cases.npz")


def log_softmax(x):
    x = np.asarray(x, np.float64)
    m = x.max(axis=1, keepdims=True)
    return (x - m - np.log(np.exp(x - m).sum(axis=1, keepdims=True))).astype(np.float32)


def ta_align(lp, lab):
    a, s = taF.forced_align(torch.from_numpy(lp)[None], torch.from_numpy(np.asarray(lab, np.int32))[None], blank=0)
    return a[0].numpy().astype(np.int32), s[0].numpy().astype(np.float32)


def collapse(p):
    out, prev = [], 0
    for c in p:
        if c != 0 and c != prev:
            out.append(int(c))
        prev = c
    return out


def brute_max(lp, lab):
    T, C = lp.shape
    best = -np.inf
    for p in itertools.product(range(C), repeat=T):
        if collapse(p) == list(lab):
            best = max(best, float(sum(float(lp[t, c]) for t, c in enumerate(p))))
    return best


def tie_free_cases(rs):
    specs = []
    for T, C, L in [(1, 2, 1), (2, 3, 1), (5, 4, 1), (7, 5, 3), (12, 6, 4), (20, 10, 6), (32, 80, 10), (64, 80, 20),
                    (128, 80, 40), (128, 40, 60), (256, 80, 90), (64, 228, 20), (200, 30, 50), (96, 12, 30)]:
        specs.append((T, C, L, "random"))
    for T, C, L in [(10, 5, 3), (40, 8, 12), (128, 40, 30), (256, 20, 64)]:
        specs.append((T, C, L, "repeats"))
    for T, C, L in [(3, 4, 1), (9, 6, 1), (64, 80, 1), (256, 8, 1)]:
        specs.append((T, C, L, "L1"))
    for L, C in [(1, 3), (3, 4), (6, 6), (12, 20), (40, 80), (90, 80)]:
        specs.append((None, C, L, "single"))
    for T, C, L in [(6, 4, 5), (30, 10, 20), (150, 40, 100), (256, 30, 127)]:
        specs.append((T, C, L, "tight"))
    for T, C, L in [(16, 3, 4), (48, 2, 1), (80, 4, 20), (256, 6, 60), (100, 80, 33), (33, 80, 32), (255, 12, 31)]:
        specs.append((T, C, L, "random"))
    cases = []
    for T, C, L, kind in specs:
        if kind == "repeats":
            base = rs.randint(1, C, size=L)
            lab = base.copy()
            lab[1::3] = lab[0::3][:len(lab[1::3])]         # every third pair doubled
        elif kind == "single":
            lab = rs.randint(1, C, size=L)
            lab[1::2] = lab[0::2][:len(lab[1::2])] if L > 1 else lab[1::2]
            T = L + int(np.count_nonzero(lab[1:] == lab[:-1]))
        else:
            lab = rs.randint(1, C, size=L)
            while T < L + int(np.count_nonzero(lab[1:] == lab[:-1])):
                lab = rs.randint(1, C, size=L)
        reps = int(np.count_nonzero(lab[1:] == lab[:-1]))
        assert T >= L + reps, (T, L, reps)
        lp = log_softmax(rs.randn(T, C) * 3.0)
        cases.append((lp, lab.astype(np.int32)))
    return cases


def tie_cases(rs, want=4):
    out = []
    while len(out) < want:
        T, C = rs.randint(3, 8), rs.randint(2, 5)
        L = rs.randint(1, min(T, 4) + 1)
        lab = rs.randint(1, C, size=L).astype(np.int32)
        if T < L + int(np.count_nonzero(lab[1:] == lab[:-1])):
            continue
        lp = (np.round(rs.uniform(-3.0, 0.0, size=(T, C)) * 2.0) / 2.0).astype(np.float32)
        path, _ = ta_align(lp, lab)
        got = float(sum(float(lp[t, c]) for t, c in enumerate(path)))
        best = brute_max(lp, lab)
        if got < best:
            out.append((lp, lab, path, got, best))
    return out


def main():
    rs = np.random.RandomState(20261021)
    arrays = {}
    cases = tie_free_cases(rs)
    for i, (lp, lab) in enumerate(cases):
        path, scores = ta_align(lp, lab)
        arrays["lp_%02d" % i], arrays["lab_%02d" % i] = lp, lab
        arrays["ta_path_%02d" % i], arrays["ta_scores_%02d" % i] = path, scores
    for j, (lp, lab, path, got, best) in enumerate(tie_cases(rs)):
        arrays["qlp_%d" % j], arrays["qlab_%d" % j], arrays["qta_path_%d" % j] = lp, lab, path
        arrays["qta_score_%d" % j], arrays["qmax_%d" % j] = np.float64(got), np.float64(best)
    arrays["n_cases"] = np.int64(len(cases))
    arrays["n_ties"] = np.int64(sum(1 for k in arrays if k.startswith("qlp_")))
    np.savez_compressed(OUT, **arrays)
    print("wrote %s: %d tie-free cases, %d tie cases" % (OUT, int(arrays["n_cases"]), int(arrays["n_ties"])))


if __name__ == "__main__":
    main()
