"""Timing probe: the LM-fused CTC prefix beam search (ops.ctc_prefix_beam_lm) against the plain one (ops.ctc_prefix_beam).

512 lines (the inference batch), T = 128 and 256, C = 80, K = 5 / 8 / 16, on random logits and on "trained-like" logits
(blank-dominated, one peaked character every few frames), with a seeded random 3-gram and a 6-gram of about 10^6
n-grams (its table, 32 MB+ of slots, outgrows L1 and most of L2).  CUDA events, median of several windows.  Also
reports the ARPA parse + table build time, and the card name and power limit of the run.

    python tools/prefix_beam_lm_probe.py [--windows 5] [--reps 5] [--json OUT.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from importlib import import_module  # noqa: E402

h = import_module("htrvt_b200")
ops = import_module("htr-vt_b200.ops")

C = 80
ALPHABET = "".join(chr(0x21 + i) for i in range(C - 2)) + " "           # 79 characters, the space last


def write_arpa(path, counts, seed):
    """Seeded random ARPA file over ALPHABET (the space as <space>), n-gram set closed under prefixes: level k
    extends random level k-1 n-grams by random tokens (duplicates dropped, so levels come out a little smaller)."""
    rs = np.random.RandomState(seed)
    words = np.array([("<space>" if ch == " " else ch) for ch in ALPHABET] + ["</s>", "<s>", "<unk>"])
    V = len(ALPHABET)
    levels = [np.arange(V + 3).reshape(-1, 1)]
    for k, n in enumerate(counts[1:], start=2):
        prev = levels[-1]
        prev = prev[(prev[:, -1] < V) | (prev[:, -1] == V + 1)] if k == 2 else prev[prev[:, -1] < V]
        par = prev[rs.randint(0, len(prev), size=int(n * 1.1))]
        nxt = rs.randint(0, V + 1, size=(len(par), 1))                   # a character or </s>
        g = np.unique(np.concatenate([par, nxt], axis=1), axis=0)
        levels.append(g[rs.permutation(len(g))[:n]])
    order = len(levels)
    with open(path, "w", encoding="utf-8") as fh:
        fh.write("\\data\\\n" + "".join("ngram %d=%d\n" % (k + 1, len(g)) for k, g in enumerate(levels)) + "\n")
        for k, g in enumerate(levels):
            fh.write("\\%d-grams:\n" % (k + 1))
            p = -rs.uniform(0.05, 3.0, size=len(g))
            b = -rs.uniform(0.0, 1.0, size=len(g))
            toks = [" ".join(r) for r in words[g]]
            has_bow = (k + 1 < order) & (g[:, -1] != V)
            fh.write("".join(("%.6f\t%s\t%.6f\n" % (pp, t, bb)) if hb else ("%.6f\t%s\n" % (pp, t))
                             for pp, t, bb, hb in zip(p, toks, b, has_bow)))
            fh.write("\n")
        fh.write("\\end\\\n")
    return sum(len(g) for g in levels)


def logits(kind, T, B, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn(T, B, C, generator=g) * 2.0
    if kind == "trained":                      # blank-dominated, one peaked character every 3-5 frames
        x = torch.randn(T, B, C, generator=g)
        x[:, :, 0] += 9.0
        t = 0
        rs = np.random.RandomState(seed)
        while t < T:
            ch = torch.from_numpy(rs.randint(1, C, size=B))
            x[t, torch.arange(B), ch] += 14.0
            x[t, :, 0] -= 9.0
            t += rs.randint(3, 6)
    return x.log_softmax(-1).cuda()


def time_ms(fn, windows, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    res = []
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        res.append(e0.elapsed_time(e1) / reps)
    return float(np.median(res)), float(min(res)), float(max(res))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except Exception as e:                     # the measurement stands without it, but say so
        return "%s (nvidia-smi unavailable: %s)" % (torch.cuda.get_device_name(), e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "the probe times the kernels on a CUDA device"
    out = {"card": card(), "torch": torch.__version__, "lms": {}, "runs": []}
    print("card:", out["card"])
    conv = h.CTCLabelConverter(ALPHABET)
    lms = {}
    with tempfile.TemporaryDirectory() as d:
        for name, counts, seed in (("3gram", [0, 6400, 150000], 1),
                                   ("6gram", [0, 6000, 60000, 200000, 330000, 420000], 2)):
            path = os.path.join(d, name + ".arpa")
            n = write_arpa(path, counts, seed)
            t0 = time.perf_counter()
            lm = h.CharNGramLM.from_arpa(path, conv)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            lms[name] = lm
            info = {"ngrams": n, "kept": lm.kept, "slots": lm.slots, "table_MB": lm.slots * 32 / 2 ** 20,
                    "parse_build_s": dt, "arpa_MB": os.path.getsize(path) / 2 ** 20}
            out["lms"][name] = info
            print("%s: %d n-grams (%.1f MB ARPA) -> %d slots (%.0f MB table): parse + build %.2f s"
                  % (name, n, info["arpa_MB"], lm.slots, info["table_MB"], dt))
    B = 512
    print("%-8s %4s %3s %10s %10s %10s %8s %8s" % ("logits", "T", "K", "plain ms", "3-gram ms", "6-gram ms",
                                                  "x 3g", "x 6g"))
    for kind in ("random", "trained"):
        for T in (128, 256):
            lp = logits(kind, T, B, seed=T)
            for K in (5, 8, 16):
                r = {"logits": kind, "B": B, "T": T, "C": C, "K": K}
                r["plain"] = time_ms(lambda: ops.ctc_prefix_beam(lp, K), a.windows, a.reps)
                for name, lm in lms.items():
                    r[name] = time_ms(lambda: ops.ctc_prefix_beam_lm(lp, K, lm, 0.8, 1.0), a.windows, a.reps)
                out["runs"].append(r)
                print("%-8s %4d %3d %10.3f %10.3f %10.3f %8.2f %8.2f" % (
                    kind, T, K, r["plain"][0], r["3gram"][0], r["6gram"][0], r["3gram"][0] / r["plain"][0],
                    r["6gram"][0] / r["plain"][0]))
    print("card:", card())
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
