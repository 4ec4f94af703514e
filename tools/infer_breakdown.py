"""Per-op breakdown of the eval-mode forward + greedy decode at 512 lines (BASELINE config 4 share).

Usage: infer_breakdown.py [B] [--variant {v1,window}] [--precision {bf16,fp32}] [--reps R]
  v1: bench.py's model (80 classes, W = 512); window: the windowed variant (90 classes, W = 1024, T = 256).
  --reps R times R windows of 5 forwards each (after 3 warm-up forwards) and prints each one's rate and the spread.
"""
import argparse
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from importlib import import_module
import bench
import htrvt_b200 as h
ops = import_module("htr-vt_b200.ops")
ap = argparse.ArgumentParser()
ap.add_argument("B", nargs="?", type=int, default=512)
ap.add_argument("--variant", choices=("v1", "window"), default="v1")
ap.add_argument("--precision", choices=("bf16", "fp32"), default="bf16")
ap.add_argument("--reps", type=int, default=1)
args = ap.parse_args()
dev = torch.device("cuda", 0)
B = args.B
torch.manual_seed(123)
if args.variant == "v1":
    H = import_module("htr-vt_b200.model.HTR_VT")
    nb_cls = bench.NB_CLS
    model = H.create_model(nb_cls, [bench.IMG_H, bench.IMG_W]).to(dev).eval()
    img = bench.synth_batch(B, 1)[0].to(dev)
else:
    Wm = import_module("htr-vt_b200.model_window.HTR_VT")
    nb_cls, W = 90, 1024
    model = Wm.create_model(nb_cls, [W, bench.IMG_H]).to(dev).eval()          # img_size = [W, H] for this variant
    img = torch.from_numpy(np.random.RandomState(1).rand(B, 1, bench.IMG_H, W).astype("float32")).to(dev)
model.set_precision(args.precision)
conv = h.CTCLabelConverter("".join(chr(33 + i) for i in range(nb_cls - 1)))
def once():
    with torch.no_grad():
        return conv.decode_logits(model(img).float())
for _ in range(3): once()
torch.cuda.synchronize()
rates = []
for _ in range(args.reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): once()
    e1.record(); torch.cuda.synchronize()
    rates.append(B / (e0.elapsed_time(e1) / 5) * 1e3)
    print("eval forward + decode: %.3f ms per %d lines = %.0f img/s" % (e0.elapsed_time(e1) / 5, B, rates[-1]))
if args.reps > 1:
    print("%s %s: %d windows of 5 forwards, lines/s min %.0f median %.0f max %.0f" % (
        args.variant, args.precision, args.reps, min(rates), float(np.median(rates)), max(rates)))
ops.PROFILE = []
once()
torch.cuda.synchronize()
prof, ops.PROFILE = ops.PROFILE, None
by = {}
for name, fl, a, b in prof:
    d = by.setdefault(name, [0.0, 0.0, 0]); d[0] += a.elapsed_time(b); d[1] += fl; d[2] += 1
tot = sum(v[0] for v in by.values())
for k, v in sorted(by.items(), key=lambda kv: -kv[1][0]):
    print("%-20s %3d launches %8.3f ms %5.1f%%  %s" % (k, v[2], v[0], 100 * v[0] / tot, ("%.0f TFLOP/s" % (v[1] / v[0] / 1e9)) if v[1] else ""))
print("sum of ops %.3f ms" % tot)
