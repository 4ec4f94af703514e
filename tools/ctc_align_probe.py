"""Time CTC forced alignment (csrc/ctc_align.cu) on the GPU, beside ctc_loss_grad on the same shapes (the same trellis
with sums, forward and backward) and torchaudio's host forced_align per line, the alternative without this kernel.

Shapes: B in {512, 4096}, T in {128, 256}, C = 80, label lengths drawn like IAM lines (mean ~40, max 90), blank-heavy
log-probs.  CUDA events around each call after warm-up; the median of --reps calls.  The card's name and power limit
are read in the same run.

Usage: python tools/ctc_align_probe.py [--reps 30] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()
    except Exception:
        return torch.cuda.get_device_name() + " (power limit not readable)"


def iam_lengths(rs, B):
    return np.clip(np.round(rs.normal(40.0, 15.0, size=B)), 1, 90).astype(np.int32)


def batch(rs, B, T, C):
    z = torch.from_numpy(rs.randn(B, T, C).astype(np.float32) * 2.0)
    z[:, :, 0] += 2.0
    lp = torch.log_softmax(z, -1).cuda()
    tl = iam_lengths(rs, B)
    tg = rs.randint(1, C, size=int(tl.sum())).astype(np.int32)
    return lp, z.cuda(), torch.from_numpy(tg), torch.from_numpy(tl)


def time_ms(fn, reps, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    a = ap.parse_args()
    import htrvt_b200 as h
    from importlib import import_module
    ops = import_module("htr-vt_b200.ops")
    assert torch.cuda.is_available(), "the probe times the GPU kernel: it needs a CUDA device"
    rs = np.random.RandomState(0)
    res = {"card": card(), "rows": []}
    print("card:", res["card"])
    print("%5s %4s %3s | %12s %12s %14s | %12s %12s" % ("B", "T", "C", "align ms", "lines/s", "align logits ms",
                                                        "ctc f+b ms", "ratio"))
    for B in (512, 4096):
        for T in (128, 256):
            C = 80
            lp, z, tg, tl = batch(rs, B, T, C)
            tgd = tg.cuda()
            al = time_ms(lambda: h.ctc_align(lp, tgd, tl, layout="btc"), a.reps)
            al_lg = time_ms(lambda: h.ctc_align(z, tgd, tl, layout="btc", is_logprob=False), a.reps)
            mtl = int(tl.max())
            ctc = time_ms(lambda: ops.ctc_loss_grad(lp, tgd, None, tl, layout="btc", is_logprob=True, want_grad=True,
                                                    max_target_len=mtl), a.reps)
            r = h.ctc_align(lp, tgd, tl, layout="btc")
            assert int((r.status != 0).sum()) == 0
            row = dict(B=B, T=T, C=C, mean_L=float(tl.float().mean()), max_L=mtl, align_ms=al, align_logits_ms=al_lg,
                       ctc_loss_grad_ms=ctc, lines_per_s=B / (al[0] * 1e-3))
            res["rows"].append(row)
            print("%5d %4d %3d | %12.3f %12.0f %14.3f | %12.3f %12.2f" % (B, T, C, al[0], row["lines_per_s"], al_lg[0],
                                                                        ctc[0], al[0] / ctc[0]))
    try:
        import torchaudio.functional as taF
        lpc = torch.log_softmax(torch.randn(1, 128, 80) * 2.0, -1)
        tgc = torch.randint(1, 80, (1, 40), dtype=torch.int32)
        for _ in range(5):
            taF.forced_align(lpc, tgc, blank=0)
        n = 200
        t0 = time.perf_counter()
        for _ in range(n):
            taF.forced_align(lpc, tgc, blank=0)
        res["torchaudio_cpu_us_per_line"] = (time.perf_counter() - t0) / n * 1e6
        print("torchaudio forced_align on the host, T = 128, C = 80, L = 40: %.1f us per line (%d threads)"
              % (res["torchaudio_cpu_us_per_line"], torch.get_num_threads()))
    except ImportError:
        res["torchaudio_cpu_us_per_line"] = None
        print("torchaudio not installed: host timing not measured")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
