"""Timing probe: the lexicon-constrained CTC prefix beam search with a word n-gram LM (ops.ctc_prefix_beam_lex with a
WordNGramLM) beside the lexicon-only search and the lexicon + character 3-gram search, in the same run.

512 lines (the inference batch), T = 128 and 256, C = 80, K = 5 / 8 / 16, on random and "trained-like" logits (blank-
dominated, one peaked character every few frames), with the seeded synthetic lexicons of tools/prefix_beam_lex_probe.py
(10^4 and 10^5 words), a seeded random character 3-gram and, per lexicon, a seeded random word 3-gram (every lexicon
word a unigram, 2 bigrams and 1 trigram per word).  CUDA events, median of several windows.  Also reports the word-LM
build time, and the card name and power limit of the run.

    python tools/prefix_beam_wordlm_probe.py [--windows 5] [--reps 5] [--json OUT.json]
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

from prefix_beam_lex_probe import synthetic_words  # noqa: E402
from prefix_beam_lm_probe import ALPHABET, C, card, logits, time_ms, write_arpa  # noqa: E402

h = import_module("htrvt_b200")
ops = import_module("htr-vt_b200.ops")


def write_word_arpa(path, words, seed):
    """seeded random word 3-gram: every word a unigram; per word two bigrams (one after <s> for a fifth of them) and
    one trigram extending a listed bigram; a fifth of the bigrams and trigrams end in </s>"""
    rs = np.random.RandomState(seed)
    n = len(words)
    w = np.array(words + ["</s>"], dtype=object)
    big = set()
    for i, j in zip(np.repeat(np.arange(n), 2).tolist(), rs.randint(0, n + 1, size=2 * n).tolist()):
        big.add((("<s>" if rs.rand() < 0.1 else w[i]), w[j if rs.rand() > 0.2 else n]))
    big = sorted(big)
    ext = [g for g in big if g[1] != "</s>"]
    tri = sorted({ext[k] + (w[rs.randint(0, n + 1)],) for k in rs.randint(0, len(ext), size=n).tolist()})
    uni = [(x,) for x in words] + [("<s>",), ("</s>",), ("<unk>",)]
    with open(path, "w", encoding="utf-8") as fh:
        fh.write("\\data\\\nngram 1=%d\nngram 2=%d\nngram 3=%d\n\n" % (len(uni), len(big), len(tri)))
        for k, gk in enumerate((uni, big, tri)):
            fh.write("\\%d-grams:\n" % (k + 1))
            p = -rs.uniform(0.05, 4.0, size=len(gk))
            b = -rs.uniform(0.0, 1.0, size=len(gk))
            fh.write("".join(("%.6f\t%s\t%.6f\n" % (-99.0 if g == ("<s>",) else pp, " ".join(g), bb))
                             if (k < 2 and g[-1] != "</s>") else ("%.6f\t%s\n" % (pp, " ".join(g)))
                             for pp, g, bb in zip(p, gk, b)))
            fh.write("\n")
        fh.write("\\end\\\n")
    return len(uni) + len(big) + len(tri)


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
    lexs, wlms = {}, {}
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "3gram.arpa")
        write_arpa(path, [0, 6400, 150000], 1)
        clm = h.CharNGramLM.from_arpa(path, conv)
        for name, n in (("10k", 10 ** 4), ("100k", 10 ** 5)):
            lx = h.Lexicon.from_words(synthetic_words(n, seed=n), conv)
            wpath = os.path.join(d, "w3_%s.arpa" % name)
            grams = write_word_arpa(wpath, lx.words, seed=n + 1)
            t0 = time.perf_counter()
            wlm = h.WordNGramLM.from_arpa(wpath, lx)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            lexs[name], wlms[name] = lx, wlm
            out["lexicons"][name] = {"words": lx.n_words, "nodes": lx.n_nodes, "word_ngrams": grams,
                                     "word_lm_build_s": dt}
            print("lexicon %s: %d words, %d trie nodes; word 3-gram of %d n-grams built in %.2f s"
                  % (name, lx.n_words, lx.n_nodes, grams, dt))
    B = 512
    cols = ["lex10k", "lex10k+c3", "lex10k+w3", "lex100k", "lex100k+c3", "lex100k+w3"]
    print("%-8s %4s %3s " % ("logits", "T", "K") + " ".join("%11s" % c for c in cols) + "  (ms)")
    for kind in ("random", "trained"):
        for T in (128, 256):
            lp = logits(kind, T, B, seed=T)
            for K in (5, 8, 16):
                r = {"logits": kind, "B": B, "T": T, "C": C, "K": K}
                for name, lx in lexs.items():
                    r["lex" + name] = time_ms(lambda: ops.ctc_prefix_beam_lex(lp, K, lx), a.windows, a.reps)
                    r["lex%s+c3" % name] = time_ms(lambda: ops.ctc_prefix_beam_lex(lp, K, lx, clm, 0.8, 1.0),
                                                   a.windows, a.reps)
                    r["lex%s+w3" % name] = time_ms(lambda: ops.ctc_prefix_beam_lex(lp, K, lx, wlms[name], 0.8, 1.0),
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
