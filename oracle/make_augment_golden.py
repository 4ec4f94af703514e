"""Golden vectors for the augmentation (SURVEY.md 8(f) row 2), produced by the reference's OWN code:
model_v1/data/dataset.py::SameTrCollate and model_v1/data/transform.py are imported UNMODIFIED from /root/reference
(dev container only) and run with the real cv2, PIL and torchvision of this image; the one missing dependency,
scikit-image, is replaced by oracle/skimage_stub (a restatement of the four symbols RandomTransform touches - the
projective-warp leg is therefore "parity unpinned", oracle/augment_oracle.py header).

Writes tests/golden/augment_cases.npz: inputs, per-case (numpy, torch) seeds and the collate's outputs for seeds that
cover all eight gate combinations; and tests/golden/augment_rng_after.json: per seed, the next np.random.rand() and
torch.rand(1) after the collate (checked against the same draws after draw_collate_params).
Usage: python oracle/make_augment_golden.py
"""
import importlib
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden")
REF = os.environ.get("HTRVT_REFERENCE", "/root/reference")


def load_reference_collate():
    for name in [m for m in sys.modules if m.split(".")[0] in ("data", "utils", "skimage")]:
        del sys.modules[name]
    sys.path.insert(0, os.path.join(HERE, "skimage_stub"))
    sys.path.insert(0, os.path.join(REF, "model_v1"))
    try:
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ds = importlib.import_module("data.dataset")
    finally:
        sys.path.remove(os.path.join(REF, "model_v1"))
    return ds.SameTrCollate


def synthetic_lines(rs, B, H, W):
    """White paper (1.0), grey-to-black pen strokes, a little paper noise: float32 [B, 1, H, W] in [0, 1]."""
    x = np.ones((B, H, W), dtype=np.float32)
    for b in range(B):
        x[b] -= rs.rand(H, W).astype(np.float32) * 0.06
        for _ in range(rs.randint(20, 40)):
            r0, c0 = rs.randint(8, H - 8), rs.randint(4, W - 12)
            hh, ww = rs.randint(2, 20), rs.randint(1, 9)
            ink = 0.05 + 0.5 * rs.rand()
            x[b, max(0, r0 - hh // 2):r0 + hh // 2 + 1, c0:c0 + ww] = ink
        k = rs.randint(W // 2, W)                      # right padding with 1.0 like the loader (dataset.py:129-130)
        x[b, :, k:] = 1.0
    return np.clip(x, 0, 1)[:, None]


def default_args():
    return types.SimpleNamespace(proj=8.0, dila_ero_max_kernel=3, dila_ero_iter=1, jitter_contrast=0.4,
                                 jitter_brightness=0.4, jitter_saturation=0.4, jitter_hue=0.2)


def main():
    sys.path.insert(0, HERE)
    sys.path.insert(0, ROOT)
    import augment_oracle as A
    aug = importlib.import_module("htr-vt_b200.augment")
    collate = load_reference_collate()
    args = default_args()
    rs = np.random.RandomState(99)
    B, H, W = 3, 64, 256
    imgs = synthetic_lines(rs, B, H, W)
    batch = [(imgs[i], "label%d" % i) for i in range(B)]
    seen, seeds, outs, after = set(), [], [], []
    seed = 0
    while len(seen) < 8 and seed < 400:
        seed += 1
        np.random.seed(seed); torch.manual_seed(seed)
        p = aug.draw_collate_params(B, H, W, args)
        mine = [np.random.rand(), float(torch.rand(1))]
        combo = tuple(p[k] is not None for k in ("warp", "morph", "jitter"))
        if combo in seen and not (combo[1] and len(seeds) < 14):
            continue
        np.random.seed(seed); torch.manual_seed(seed)
        out, labels = collate(batch, args)
        # the next draw of each global generator: where the collate leaves them, including draws that do not change
        # the output (saturation / hue factors on grey images)
        nxt = [np.random.rand(), float(torch.rand(1))]
        assert mine == nxt, (seed, combo, mine, nxt)
        after.append(nxt)
        assert list(labels) == ["label%d" % i for i in range(B)]
        got = np.round(out.numpy()[:, 0] * 255).astype(np.uint8)
        # the product's draw order + the oracle's pixel arithmetic reproduce the reference's output
        want = A.apply_params(np.uint8(imgs[:, 0] * 255), p)
        assert np.array_equal(got, want), (seed, combo, int((got != want).sum()))
        seen.add(combo); seeds.append(seed); outs.append(got)
        print("seed", seed, "gates", combo, "morph", p["morph"])
    np.savez_compressed(os.path.join(OUT, "augment_cases.npz"), images=imgs.astype(np.float32),
                        seeds=np.array(seeds, dtype=np.int64), outputs=np.stack(outs),
                        args=np.array([args.proj, args.dila_ero_max_kernel, args.dila_ero_iter, args.jitter_brightness,
                                       args.jitter_contrast, args.jitter_saturation, args.jitter_hue]))
    with open(os.path.join(OUT, "augment_rng_after.json"), "w") as fh:
        json.dump({"source": "the reference SameTrCollate (oracle/make_augment_golden.py)", "seeds": seeds,
                   "next_np_torch": after}, fh, indent=1)
        fh.write("\n")
    print(len(seeds), "cases, all", len(seen), "gate combinations")


if __name__ == "__main__":
    main()
