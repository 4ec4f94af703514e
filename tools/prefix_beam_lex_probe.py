"""Timing probe: the lexicon-constrained CTC prefix beam search (ops.ctc_prefix_beam_lex) against the plain and the
LM-fused searches (ops.ctc_prefix_beam, ops.ctc_prefix_beam_lm) in the same run.

512 lines (the inference batch), T = 128 and 256, C = 80, K = 5 / 8 / 16, on random logits and on "trained-like"
logits (blank-dominated, one peaked character every few frames), with seeded synthetic lexicons of 10^4 and 10^5
words (2-10 letters over 52 letters; digits, punctuation and the space are free) and a seeded random 3-gram.  CUDA
events, median of several windows.  Also reports the lexicon build time, and the card name and power limit of the run.

    python tools/prefix_beam_lex_probe.py [--windows 5] [--reps 5] [--json OUT.json]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch  # noqa: E402
from importlib import import_module  # noqa: E402

from prefix_beam_lm_probe import ALPHABET, C, card, logits, time_ms, write_arpa  # noqa: E402

h = import_module("htrvt_b200")
ops = import_module("htr-vt_b200.ops")
LETTERS = "".join(ch for ch in ALPHABET if ch.isalpha())[:52]


def synthetic_words(n, seed):
    """n distinct seeded words of 2-10 letters over LETTERS"""
    rs = np.random.RandomState(seed)
    out = set()
    while len(out) < n:
        k = rs.randint(2, 11, size=n)
        idx = rs.randint(0, len(LETTERS), size=int(k.sum()))
        s = "".join(LETTERS[i] for i in idx)
        ends = np.cumsum(k)
        out.update(s[e - m:e] for e, m in zip(ends.tolist(), k.tolist()))
    return sorted(out)[:n]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "the probe times the kernels on a CUDA device"
    out = {"card": card(), "torch": torch.__version__, "lexicons": {}, "runs": []}
    print("card:", out["card"])
    conv = h.CTCLabelConverter(ALPHABET)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "3gram.arpa")
        write_arpa(path, [0, 6400, 150000], 1)
        lm = h.CharNGramLM.from_arpa(path, conv)
    lexs = {}
    for name, n in (("10k", 10 ** 4), ("100k", 10 ** 5)):
        words = synthetic_words(n, seed=n)
        t0 = time.perf_counter()
        lx = h.Lexicon.from_words(words, conv)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        lexs[name] = lx
        out["lexicons"][name] = {"words": lx.n_words, "nodes": lx.n_nodes, "build_s": dt}
        print("lexicon %s: %d words, %d trie nodes, build %.2f s" % (name, lx.n_words, lx.n_nodes, dt))
    B = 512
    cols = ["plain", "lex10k", "lex100k", "3gram", "lex10k+3g", "lex100k+3g"]
    print("%-8s %4s %3s " % ("logits", "T", "K") + " ".join("%11s" % c for c in cols) + "  (ms)")
    for kind in ("random", "trained"):
        for T in (128, 256):
            lp = logits(kind, T, B, seed=T)
            for K in (5, 8, 16):
                r = {"logits": kind, "B": B, "T": T, "C": C, "K": K}
                r["plain"] = time_ms(lambda: ops.ctc_prefix_beam(lp, K), a.windows, a.reps)
                r["3gram"] = time_ms(lambda: ops.ctc_prefix_beam_lm(lp, K, lm, 0.8, 1.0), a.windows, a.reps)
                for name, lx in lexs.items():
                    r["lex" + name] = time_ms(lambda: ops.ctc_prefix_beam_lex(lp, K, lx), a.windows, a.reps)
                    r["lex%s+3g" % name] = time_ms(lambda: ops.ctc_prefix_beam_lex(lp, K, lx, lm, 0.8, 1.0),
                                                   a.windows, a.reps)
                out["runs"].append(r)
                print("%-8s %4d %3d " % (kind, T, K) + " ".join("%11.3f" % r[c][0] for c in cols))
    print("card:", card())
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
