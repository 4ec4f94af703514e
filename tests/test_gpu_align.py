"""GPU: CTC forced alignment (csrc/ctc_align.cu; ops.ctc_align, forced_align, align_text) against the float64 oracle
`ctc_viterbi_align` (pinned to brute force and torchaudio in tests/test_oracle_align.py): path, spans, status and score
bit-equal, frame and token scores equal in log-prob mode; the logits mode, a 4096-line batch, the public entry points
and the refusals."""
import math
import os

import numpy as np
import pytest
import torch

import htrvt_align_oracle as A
import htrvt_oracle as O

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "align_cases.npz")


def _h():
    import htrvt_b200
    return htrvt_b200


def _log_softmax(x):
    x = np.asarray(x, np.float64)
    m = x.max(axis=-1, keepdims=True)
    return x - m - np.log(np.exp(x - m).sum(axis=-1, keepdims=True))


def _labels(rs, L, C, kind):
    if C == 2 or kind == "run":
        return np.full(L, 1 if C == 2 else rs.randint(1, C), np.int64)       # one repeated letter
    return rs.randint(1, C, size=L)


def _run(x_btc, labels, in_len, *, layout, padded, host_lengths, is_logprob=True, lengths_override=None):
    """x_btc: fp32 numpy [B, T, C]; labels: list of int arrays; in_len: list of frame counts (None = T)."""
    B, T, C = x_btc.shape
    tl = np.array([len(l) for l in labels] if lengths_override is None else lengths_override, np.int32)
    if padded:
        w = max([len(l) for l in labels] + [1])
        tg = np.zeros((B, w), np.int32)
        for b, l in enumerate(labels):
            tg[b, :len(l)] = l
    else:
        tg = np.concatenate([np.asarray(l, np.int32) for l in labels] + [np.zeros(0, np.int32)])
    xt = torch.from_numpy(np.ascontiguousarray(x_btc)).cuda()
    if layout == "tbc":
        xt = xt.transpose(0, 1).contiguous()
    tl_t = torch.from_numpy(tl) if host_lengths else torch.from_numpy(tl).cuda()
    il = None if in_len is None else torch.tensor(in_len, dtype=torch.int32).cuda()
    r = _h().ctc_align(xt, torch.from_numpy(tg).cuda(), tl_t, il, layout=layout, is_logprob=is_logprob)
    torch.cuda.synchronize()
    return type(r)(*[t.cpu().numpy() for t in r])


def _check_line(r, b, want, L, exact_scores=True):
    assert int(r.status[b]) == want.status, (b, int(r.status[b]), want.status)
    assert np.array_equal(r.path[b], want.path), b
    if want.status == 0:
        assert r.score[b] == want.score, (b, r.score[b], want.score)
    else:
        assert r.score[b] == -math.inf
    n = r.spans.shape[1]
    sp = np.full((n, 2), -1, np.int64)
    ts = np.zeros(n, np.float32)
    if want.status == 0:
        sp[:L] = want.spans
        ts[:L] = want.token_scores
    assert np.array_equal(r.spans[b], sp), b
    if exact_scores:
        assert np.array_equal(r.frame_scores[b], want.frame_scores), b
        assert np.array_equal(r.token_scores[b], ts), b


SHAPES = [(T, C) for T in (1, 2, 7, 128, 256, 1024) for C in (2, 80, 228)]
LS = (0, 1, 31, 32, 33, 64, 127, 200, 256)


@pytest.mark.parametrize("T,C", SHAPES)
def test_kernel_matches_oracle(T, C):
    rs = np.random.RandomState(T * 1000 + C)
    labels, in_len = [], []
    for i, L in enumerate(LS):
        labels.append(_labels(rs, L, C, "run" if i % 4 == 3 else "random"))
        in_len.append(T if i % 3 == 0 else max(T - i, 0))
    labels.append(np.zeros(0, np.int64)); in_len.append(0)                          # empty line, no frames
    labels.append(_labels(rs, 3, C, "random")); in_len.append(0)                     # labels, no frames: infeasible
    B = len(labels)
    quantised = (T + C) % 2 == 1
    if quantised:                                                                      # exact ties everywhere
        x = (np.round(rs.uniform(-4.0, 0.0, size=(B, T, C)) * 2.0) / 2.0).astype(np.float32)
    else:
        x = _log_softmax(rs.randn(B, T, C) * 3.0).astype(np.float32)
    want = [A.ctc_viterbi_align(x[b], labels[b], in_len[b]) for b in range(B)]
    for layout in ("btc", "tbc"):
        for padded in (False, True):
            for host in (False, True):
                r = _run(x, labels, in_len, layout=layout, padded=padded, host_lengths=host)
                for b in range(B):
                    _check_line(r, b, want[b], len(labels[b]))


@pytest.mark.parametrize("lmax", [0, 1, 31, 32, 33, 63, 64, 127, 128, 200, 255, 256])
def test_states_per_lane_instantiations(lmax):
    """The host-side hint (longest label) picks 2, 4, 8, 16 or 17 states per lane: every boundary, both sides."""
    rs = np.random.RandomState(500 + lmax)
    T, C = 520, 80
    Ls = sorted(set([lmax, lmax // 2, max(lmax - 1, 0), 0]))
    labels = [_labels(rs, L, C, "run" if L == lmax // 2 and L > 1 else "random") for L in Ls]
    labels = [l if len(l) + int(np.count_nonzero(l[1:] == l[:-1])) <= T else l[:T // 2] for l in labels]
    labels[-1] = rs.randint(1, C, size=lmax)                               # the longest line sets the hint
    in_len = [T - 3 * i for i in range(len(Ls))]
    x = _log_softmax(rs.randn(len(Ls), T, C) * 3.0).astype(np.float32)
    want = [A.ctc_viterbi_align(x[b], labels[b], in_len[b]) for b in range(len(Ls))]
    for host in (True, False):
        r = _run(x, labels, in_len, layout="tbc", padded=not host, host_lengths=host)
        for b in range(len(Ls)):
            _check_line(r, b, want[b], len(labels[b]))


def test_ties_runs_and_small_alphabets():
    rs = np.random.RandomState(7)
    for T, C, Ls in [(7, 2, (1, 2, 3, 4)), (40, 3, (5, 10, 19, 20)), (128, 5, (30, 60, 63, 64)),
                     (300, 4, (100, 149, 150, 151))]:
        labels = [_labels(rs, L, C, "run" if j % 2 else "random") for j, L in enumerate(Ls)]
        x = (np.round(rs.uniform(-2.0, 0.0, size=(len(Ls), T, C)) * 2.0) / 2.0).astype(np.float32)
        x[:, :, 0] = -1.0                                                              # blank ties with labels
        want = [A.ctc_viterbi_align(x[b], labels[b]) for b in range(len(Ls))]
        r = _run(x, labels, None, layout="btc", padded=True, host_lengths=True)
        for b in range(len(Ls)):
            _check_line(r, b, want[b], len(labels[b]))


@pytest.mark.parametrize("padded", [False, True])
def test_mixed_batch_infeasible_and_invalid(padded):
    rs = np.random.RandomState(11)
    T, C = 64, 20
    x = _log_softmax(rs.randn(10, T, C) * 2.0).astype(np.float32)
    labels = [rs.randint(1, C, size=10),                      # fine
              np.array([3, 3, 3, 3]),                         # infeasible at 6 frames (needs 7)
              np.array([1, 2, C]),                            # label == C: invalid
              rs.randint(1, C, size=30),                      # fine
              np.array([4, 0, 5]),                            # blank inside the labels: invalid
              rs.randint(1, C, size=5),                       # T_b > T: invalid
              rs.randint(1, C, size=40),                      # infeasible: 40 labels in 30 frames
              np.array([], np.int64),                         # empty, fine
              rs.randint(1, C, size=8),                       # fine, after the invalid lines
              np.array([7])]                                  # fine at one frame
    in_len = [T, 6, T, 50, T, T + 1, 30, 0, T, 1]
    r = _run(x, labels, in_len, layout="btc", padded=padded, host_lengths=False)
    for b in range(10):
        if b == 5:                                            # (the oracle takes no lines longer than their rows)
            assert int(r.status[b]) == 2 and (r.path[b] == -1).all() and (r.frame_scores[b] == 0).all()
            assert r.score[b] == -math.inf and (r.spans[b] == -1).all() and (r.token_scores[b] == 0).all()
            continue
        want = A.ctc_viterbi_align(x[b], labels[b], in_len[b])
        _check_line(r, b, want, len(labels[b]))
    assert r.status.tolist() == [0, 1, 2, 0, 2, 2, 1, 0, 0, 0]


def test_negative_length_and_label_limit():
    rs = np.random.RandomState(12)
    T, C = 600, 30
    x = _log_softmax(rs.randn(4, T, C)).astype(np.float32)
    labels = [rs.randint(1, C, size=12), np.zeros(0, np.int64), rs.randint(1, C, size=257), rs.randint(1, C, size=9)]
    # concatenated targets: a negative length counts as 0 when later lines' labels are located
    r = _run(x, labels, None, layout="btc", padded=False, host_lengths=False, lengths_override=[12, -3, 257, 9])
    assert r.status.tolist() == [0, 2, 2, 0]
    for b in (0, 3):
        _check_line(r, b, A.ctc_viterbi_align(x[b], labels[b]), len(labels[b]))


def test_logits_mode():
    rs = np.random.RandomState(21)
    for T, C in [(1, 2), (7, 80), (256, 80), (1024, 228)]:
        Ls = [min(L, T) for L in (0, 1, 33, 127, 200)]
        labels = [rs.randint(1, C, size=L) for L in Ls]
        labels = [l if T >= len(l) + int(np.count_nonzero(l[1:] == l[:-1])) else np.zeros(0, np.int64)
                  for l in labels]
        x = (rs.randn(len(Ls), T, C) * 3.0 + 5.0).astype(np.float32)
        r = _run(x, labels, None, layout="btc", padded=False, host_lengths=True, is_logprob=False)
        for b in range(len(Ls)):
            raw = A.ctc_viterbi_align(x[b], labels[b])
            assert np.array_equal(r.path[b], raw.path) and int(r.status[b]) == 0
            want = A.ctc_viterbi_align(_log_softmax(x[b]), labels[b])
            assert np.array_equal(want.path, raw.path)
            np.testing.assert_allclose(r.frame_scores[b], want.frame_scores, atol=1e-5, rtol=0)
            np.testing.assert_allclose(r.token_scores[b, :len(labels[b])], want.token_scores, atol=1e-5, rtol=0)
            assert abs(r.score[b] - want.score) < 1e-5, (b, r.score[b], want.score)


def test_scale_greedy_targets_and_ctc_likelihood():
    """4096 lines at T = 256 aligned to their own greedy decode: the argmax path is feasible and scores the sum of the
    frame maxima, which bounds every path, so the Viterbi score must equal it."""
    from importlib import import_module
    ops = import_module("htr-vt_b200.ops")
    g = torch.Generator(device="cuda").manual_seed(5)
    B, T, C = 4096, 256, 80
    z = torch.randn(B, T, C, device="cuda", generator=g) * 2.0
    z[:, :, 0] += 3.0                                                      # blank-heavy, like a trained model
    lp = torch.log_softmax(z, dim=-1)
    lpn = lp.cpu().numpy()
    am = lpn.argmax(axis=-1)
    labels, lens = [], []
    for b in range(B):
        lab = [int(c) for i, c in enumerate(am[b]) if c != 0 and (i == 0 or c != am[b, i - 1])]
        labels.extend(lab)
        lens.append(len(lab))
    tg = torch.tensor(labels, dtype=torch.int32)
    tl = torch.tensor(lens, dtype=torch.int32)
    r = _h().ctc_align(lp, tg, tl, layout="btc")
    status, score, path = r.status.cpu().numpy(), r.score.cpu().numpy(), r.path.cpu().numpy()
    assert (status == 0).all()
    mx = np.cumsum(lpn.max(axis=-1).astype(np.float64), axis=1)[:, -1]    # sequential float64 sum per line
    assert np.all(np.abs(score - mx) <= 1e-12 * np.maximum(1.0, np.abs(mx))), np.abs(score - mx).max()
    top2 = np.partition(lpn, C - 2, axis=-1)[:, :, -2:]                    # [runner-up, maximum]
    clear = (top2[:, :, 1] - top2[:, :, 0]) > 1e-6
    assert np.array_equal(path[clear], am[clear])
    nll, _ = ops.ctc_loss_grad(lp, tg, None, tl, layout="btc", is_logprob=True, want_grad=False,
                               max_target_len=int(max(lens)))
    nll = nll.double().cpu().numpy()
    assert np.all(score <= -nll + 1e-4 * np.maximum(1.0, np.abs(nll)))


def test_forced_align_matches_torchaudio_golden():
    g = np.load(GOLDEN)
    n = int(g["n_cases"])
    groups = {}
    for i in range(n):
        groups.setdefault(g["lp_%02d" % i].shape[1], []).append(i)
    for C, ids in groups.items():                                          # one padded batch per alphabet size
        T = max(g["lp_%02d" % i].shape[0] for i in ids)
        Lw = max(len(g["lab_%02d" % i]) for i in ids)
        x = np.zeros((len(ids), T, C), np.float32)
        tg = np.zeros((len(ids), Lw), np.int32)
        il, tl = [], []
        for j, i in enumerate(ids):
            lp, lab = g["lp_%02d" % i], g["lab_%02d" % i]
            x[j, :lp.shape[0]] = lp
            tg[j, :len(lab)] = lab
            il.append(lp.shape[0]); tl.append(len(lab))
        al, sc = _h().forced_align(torch.from_numpy(x).cuda(), torch.from_numpy(tg).cuda(),
                                   torch.tensor(il, dtype=torch.int32), torch.tensor(tl, dtype=torch.int32))
        al, sc = al.cpu().numpy(), sc.cpu().numpy()
        for j, i in enumerate(ids):
            Tb = il[j]
            assert np.array_equal(al[j, :Tb], g["ta_path_%02d" % i]), i
            assert np.array_equal(sc[j, :Tb], g["ta_scores_%02d" % i]), i
            assert (al[j, Tb:] == -1).all() and (sc[j, Tb:] == 0).all()


def test_align_text_on_model_output():
    H = __import__("importlib").import_module("htr-vt_b200.model.HTR_VT")
    h = _h()
    nb_cls, W = 80, 512
    m = H.create_model(nb_cls, [64, W])
    m.load_state_dict(O.init_state_dict(nb_cls, [64, W], seed=31), strict=True)
    m = m.cuda().eval()
    rs = np.random.RandomState(32)
    x = torch.from_numpy(rs.rand(4, 1, 64, W).astype(np.float32)).cuda()
    with torch.no_grad():
        logits = m(x).float()
    alphabet = "".join(chr(ord("a") + i) for i in range(26)) + "".join(chr(ord("A") + i) for i in range(26)) + \
        "0123456789 .,;:!?'\"()-+*/=&%#@<>[]_"
    alphabet = alphabet[:nb_cls - 1]
    conv = h.CTCLabelConverter(alphabet)
    texts = ["".join(alphabet[i] for i in rs.randint(0, len(alphabet), size=n)) for n in (1, 17, 40, 60)]
    texts[2] = texts[2][:10] + "ll" + texts[2][12:]                      # a doubled letter
    T = logits.shape[1]
    out = h.align_text(logits, conv, texts, image_width=W)
    assert len(out) == 4
    for text, boxes in zip(texts, out):
        assert "".join(c for c, _, _, _ in boxes) == text
        prev = 0
        for ch, x0, x1, lpv in boxes:
            assert prev <= x0 < x1 <= W and x0 % (W // T) == 0
            assert lpv <= 0.0
            prev = x1
    r = h.ctc_align(logits, *conv.encode(texts), layout="btc", is_logprob=False)
    assert out[1][3][1] == 4 * int(r.spans[1, 3, 0]) and (r.status == 0).all().item()
    assert h.align_text(logits, conv, texts, px_per_frame=4) == out


def test_refusals():
    h = _h()
    HtrvtError = h._lib.HtrvtError
    lp = torch.log_softmax(torch.randn(2, 16, 5), -1)
    tg = torch.tensor([[1, 2], [3, 3]], dtype=torch.int32)
    with pytest.raises(HtrvtError):
        h.forced_align(lp, tg)                                            # CPU tensors
    with pytest.raises(HtrvtError):
        h.ctc_align(lp.cuda().half(), tg, torch.tensor([2, 2]), layout="btc")
    with pytest.raises(ValueError):
        h.forced_align(lp.cuda(), tg, blank=1)
    with pytest.raises(ValueError):
        h.forced_align(lp.cuda(), torch.tensor([[1, 5], [1, 2]], dtype=torch.int32))   # label id == C
    with pytest.raises(HtrvtError, match=r"\[1\]"):
        h.forced_align(lp.cuda(), tg, torch.tensor([16, 1], dtype=torch.int32))       # [3, 3] needs 3 frames
    big = torch.log_softmax(torch.randn(1, 600, 5), -1).cuda()
    with pytest.raises(HtrvtError):
        h.ctc_align(big, torch.ones(257, dtype=torch.int32), torch.tensor([257]), layout="btc")   # L > 256
    r = h.ctc_align(big, torch.ones(257, dtype=torch.int32).cuda(), torch.tensor([257]).cuda(), layout="btc")
    assert int(r.status[0]) == 2                                          # the same line with device-side lengths
    with pytest.raises(ValueError, match="'ß'"):
        h.align_text(torch.randn(1, 8, 4).cuda(), h.CTCLabelConverter("abc"), ["aß"], image_width=32)
    # whole-call refusals of the C ABI: nothing is launched
    from importlib import import_module
    L = import_module("htr-vt_b200._lib")
    lib = L.lib()
    x = lp.cuda().contiguous()
    path, spans, status = (torch.empty(n, dtype=torch.int32, device="cuda") for n in (32, 8, 2))
    fs, ts = (torch.empty(n, dtype=torch.float32, device="cuda") for n in (32, 4))
    score = torch.empty(2, dtype=torch.float64, device="cuda")
    tgc, tlc = tg.cuda(), torch.tensor([2, 2], dtype=torch.int32).cuda()
    need = lib.htrvt_ctc_align_workspace_bytes(2, 16, 2)
    ws = torch.empty(need + 16, dtype=torch.uint8, device="cuda")
    p = lambda t: t.data_ptr()                                            # noqa: E731

    def call(T=16, C=5, sb=80, st=5, hint=2, wsb=need, wsp=None):
        return lib.htrvt_ctc_align(p(x), sb, st, 1, p(tgc), 2, None, p(tlc), 2, T, C, hint, p(path), p(fs),
                                   p(spans), 2, p(ts), p(score), p(status), wsp or p(ws), wsb, None)
    assert call() == 0
    torch.cuda.synchronize()
    assert status.tolist() == [0, 0]                                      # T_b = T = 16 for both lines
    assert call(T=0) == -1 and call(C=1) == -1 and call(sb=-1) == -1 and call(hint=257) == -1
    assert call(wsb=need - 1) == -5
    assert call(wsp=p(ws) + 4) == -2
    torch.cuda.synchronize()
