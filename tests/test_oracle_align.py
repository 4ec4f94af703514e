"""CPU: the float64 forced-alignment oracle (oracle/htrvt_align_oracle.py) against brute force, hand-built ties,
torchaudio's recorded outputs and the CTC likelihood."""
import itertools
import math
import os

import numpy as np
import pytest

import htrvt_align_oracle as A
import htrvt_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "align_cases.npz")


def _path_sum(lp, path):
    return sum(float(lp[t, c]) for t, c in enumerate(path))


def _brute(lp, labels):
    """max over all C^T paths that collapse to the labels (None when there is none)"""
    T, C = lp.shape
    best = None
    for p in itertools.product(range(C), repeat=T):
        if A.collapse(p) == list(labels):
            v = _path_sum(lp, p)
            best = v if best is None or v > best else best
    return best


def _log_softmax(x):
    m = x.max(axis=1, keepdims=True)
    return (x - m - np.log(np.exp(x - m).sum(axis=1, keepdims=True))).astype(np.float32)


def _check_consistent(lp, labels, r):
    T = lp.shape[0]
    assert r.status == 0
    assert A.collapse(r.path) == list(labels)
    assert _path_sum(lp, r.path[:T]) == r.score                 # float64 sum of the path equals the Viterbi score
    for k in range(len(labels)):
        a, z = r.spans[k]
        assert 0 <= a < z <= T and all(r.path[t] == labels[k] for t in range(a, z))
    assert np.array_equal(r.frame_scores, lp[np.arange(T), r.path].astype(np.float32))


@pytest.mark.parametrize("seed", range(40))
def test_brute_force_tiny(seed):
    rs = np.random.RandomState(seed)
    T, C = rs.randint(1, 8), rs.randint(2, 5)
    if C ** T > 20000:
        T = 6
    L = rs.randint(0, min(T + 2, 5))
    labels = rs.randint(1, C, size=L).tolist()
    quantised = seed % 2 == 1
    x = rs.uniform(-3.0, 0.0, size=(T, C))
    lp = (np.round(x * 2.0) / 2.0).astype(np.float32) if quantised else _log_softmax(rs.randn(T, C) * 2.0)
    r = A.ctc_viterbi_align(lp, labels)
    best = _brute(lp, labels)
    if best is None:
        assert r.status == 1 and r.score == -math.inf and (r.path == -1).all()
        return
    assert r.status == 0
    assert r.score == best
    _check_consistent(lp, labels, r)


def test_infeasible_is_exactly_too_few_frames():
    for labels in ([1], [1, 1], [1, 2, 1], [2, 2, 2], [1, 2]):
        reps = sum(1 for a, b in zip(labels, labels[1:]) if a == b)
        for T in range(1, 7):
            lp = np.log(np.full((T, 3), 1.0 / 3.0)).astype(np.float32)
            r = A.ctc_viterbi_align(lp, labels)
            assert (r.status == 1) == (T < len(labels) + reps) == (_brute(lp, labels) is None)


def test_tie_stay_beats_previous():
    # frame 1, state 1 (label): stay (from state 1) and previous (from blank) both -1: stay wins -> label at frames 0, 1
    lp = np.array([[-1.0, -1.0], [-5.0, -1.0]], np.float32)
    r = A.ctc_viterbi_align(lp, [1])
    assert r.path.tolist() == [1, 1] and r.score == -2.0


def test_tie_previous_beats_skip():
    # labels a b: state 3 (b) at frame 2 from state 2 (blank, previous) or state 1 (a, skip), both -2: previous wins
    lp = np.array([[-9.0, -1.0, -9.0],
                   [-1.0, -1.0, -9.0],
                   [-9.0, -9.0, -1.0]], np.float32)
    r = A.ctc_viterbi_align(lp, [1, 2])
    assert r.path.tolist() == [1, 0, 2]
    assert r.score == -3.0


def test_tie_end_on_last_label():
    # d(S-1) == d(S-2): the path ends on the last label, not on the trailing blank
    lp = np.array([[-9.0, -1.0], [-1.0, -1.0]], np.float32)
    r = A.ctc_viterbi_align(lp, [1])
    assert r.path.tolist() == [1, 1] and r.score == -2.0


def test_golden_tie_free_cases_match_torchaudio():
    g = np.load(GOLDEN)
    n = int(g["n_cases"])
    assert n >= 35
    for i in range(n):
        lp, lab = g["lp_%02d" % i], g["lab_%02d" % i]
        r = A.ctc_viterbi_align(lp, lab)
        assert r.status == 0
        assert np.array_equal(r.path, g["ta_path_%02d" % i]), i
        np.testing.assert_allclose(r.frame_scores, g["ta_scores_%02d" % i], atol=1e-5)
        assert abs(r.score - float(g["ta_scores_%02d" % i].astype(np.float64).sum())) < 1e-3


def test_golden_ties_oracle_finds_the_true_maximum():
    g = np.load(GOLDEN)
    nq = int(g["n_ties"])
    assert nq >= 3
    for j in range(nq):
        lp, lab = g["qlp_%d" % j], g["qlab_%d" % j]
        r = A.ctc_viterbi_align(lp, lab)
        assert float(g["qta_score_%d" % j]) < float(g["qmax_%d" % j])      # torchaudio's path is below the maximum
        assert r.score == float(g["qmax_%d" % j])
        assert not np.array_equal(r.path, g["qta_path_%d" % j])
        _check_consistent(lp, lab, r)


@pytest.mark.parametrize("seed", range(8))
def test_viterbi_below_ctc_likelihood(seed):
    rs = np.random.RandomState(100 + seed)
    T, C, L = rs.randint(3, 16), rs.randint(3, 8), rs.randint(1, 5)
    labels = rs.randint(1, C, size=L)
    reps = int(np.count_nonzero(labels[1:] == labels[:-1]))
    if T < L + reps:
        T = L + reps
    single = seed % 2 == 1
    if single:                                          # only one alignment exists: Viterbi = likelihood
        T = L + reps
    logits = rs.randn(1, T, C)
    nll, _ = O.ctc_loss_grad(logits, labels, np.array([T]), np.array([L]))
    lp = logits[0] - np.log(np.exp(logits[0]).sum(axis=1, keepdims=True))
    r = A.ctc_viterbi_align(lp, labels)
    assert r.status == 0
    assert r.score <= -nll[0] + 1e-9
    if single:
        assert abs(r.score + nll[0]) < 1e-9


def test_invalid_and_padding():
    lp = np.log(np.full((5, 4), 0.25))
    assert A.ctc_viterbi_align(lp, [0]).status == 2
    assert A.ctc_viterbi_align(lp, [4]).status == 2
    assert A.ctc_viterbi_align(lp, [1], input_length=6).status == 2
    assert A.ctc_viterbi_align(lp, [1] * 257).status == 2
    r = A.ctc_viterbi_align(lp, [1, 2], input_length=3)
    assert r.status == 0 and r.path[3:].tolist() == [-1, -1] and r.frame_scores[3:].tolist() == [0.0, 0.0]
    r = A.ctc_viterbi_align(lp, [], input_length=0)
    assert r.status == 0 and r.score == 0.0 and (r.path == -1).all()
    r = A.ctc_viterbi_align(lp, [])
    assert r.status == 0 and r.path.tolist() == [0] * 5
