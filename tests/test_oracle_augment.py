"""CPU tests of the augmentation oracle (oracle/augment_oracle.py) and of the product's host logic
(htr-vt_b200/augment.py): restatements pinned bit for bit to cv2 / PIL / torchvision / scipy where those are
importable and committed goldens produced by the reference's own SameTrCollate (oracle/make_augment_golden.py)."""
import os
import sys
import types
from importlib import import_module

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import augment_oracle as A  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")


def _args(g=None):
    v = [8.0, 3, 1, 0.4, 0.4, 0.4, 0.2] if g is None else list(g["args"])
    return types.SimpleNamespace(proj=float(v[0]), dila_ero_max_kernel=int(v[1]), dila_ero_iter=int(v[2]),
                                 jitter_brightness=float(v[3]), jitter_contrast=float(v[4]),
                                 jitter_saturation=float(v[5]), jitter_hue=float(v[6]))


def _img(rs, H=64, W=200):
    x = rs.randint(0, 256, (H, W)).astype(np.uint8)
    x[:, : W // 3] = np.clip(x[:, : W // 3].astype(int) + 150, 0, 255)
    x[H // 4: H // 2, W // 2:] = 255
    return x


def test_morph_restatement_matches_cv2():
    cv2 = pytest.importorskip("cv2")
    rs = np.random.RandomState(0)
    x = _img(rs)
    for kr in (1, 2, 3, 4):
        for kc in (1, 2, 3):
            for it in (1, 2, 3):
                k = np.ones((kr, kc), np.uint8)
                assert np.array_equal(A.morph(x, kr, kc, it, True), cv2.erode(x, k, iterations=it)), (kr, kc, it)
                assert np.array_equal(A.morph(x, kr, kc, it, False), cv2.dilate(x, k, iterations=it)), (kr, kc, it)


def test_jitter_restatement_matches_torchvision_on_grey_images():
    TF = pytest.importorskip("torchvision.transforms.functional")
    from PIL import Image
    rs = np.random.RandomState(1)
    x = _img(rs)
    pim = Image.fromarray(x)
    for f in list(rs.uniform(0.6, 1.4, 30)) + [1.0, 0.6, 1.4, 0.0, 2.0, float(np.float32(1.0)) + 1e-9]:
        assert np.array_equal(A.jitter_L(x, [0], [f, None, None, None]), np.array(TF.adjust_brightness(pim, f))), f
        assert np.array_equal(A.jitter_L(x, [1], [None, f, None, None]), np.array(TF.adjust_contrast(pim, f))), f
        assert np.array_equal(np.array(TF.adjust_saturation(pim, f)), x)
        assert np.array_equal(np.array(TF.adjust_hue(pim, max(-0.5, min(0.5, f - 1.0)))), x)
    # a full ColorJitter call with the same torch seed
    from torchvision.transforms import ColorJitter
    cj = ColorJitter(0.4, 0.4, 0.4, 0.2)
    for seed in range(6):
        torch.manual_seed(seed)
        want = np.array(cj(pim))
        torch.manual_seed(seed)
        order, b, c, s, h = ColorJitter.get_params(cj.brightness, cj.contrast, cj.saturation, cj.hue)
        assert np.array_equal(A.jitter_L(x, [int(v) for v in order], [b, c, s, h]), want)


def test_zoom_and_antialias_restatements_match_scipy():
    ndi = pytest.importorskip("scipy.ndimage")
    rs = np.random.RandomState(2)
    for ih, iw, oh, ow in [(70, 37, 64, 32), (60, 30, 64, 32), (64, 32, 64, 32), (81, 45, 64, 40), (1, 9, 4, 9),
                           (34, 76, 33, 77), (63, 509, 64, 512), (50, 500, 64, 512), (9, 1, 9, 5), (2, 3, 7, 11),
                           (30, 40, 33, 47), (20, 31, 33, 30), (33, 20, 30, 31), (5, 7, 9, 13)]:
        for x in (rs.randint(0, 256, (ih, iw)).astype(np.float64), rs.rand(ih, iw) * 255):
            want = ndi.zoom(x, [oh / ih, ow / iw], order=1, mode="mirror", cval=0, grid_mode=True)
            assert np.array_equal(A.zoom_linear_mirror(x, oh, ow), want), (ih, iw, oh, ow)
    # the three-tap anti-aliasing filter of the CUDA kernel: centre * w0 + (up + down) * w1, rows mirrored
    x = rs.randint(0, 256, (81, 50)).astype(np.float64)
    x[:, :20] = 255.0
    sig = A.antialias_sigma((81, 50), (64, 50))
    assert 0.125 < sig[0] < 0.375 and sig[1] == 0
    want = ndi.gaussian_filter(x, sig, cval=0, mode="mirror")
    k = np.exp(-0.5 / (sig[0] * sig[0]) * np.arange(-1, 2) ** 2)
    k = k / k.sum()
    up = x[[1] + list(range(0, 80))]
    dn = x[list(range(1, 81)) + [79]]
    assert np.array_equal(x * k[1] + (up + dn) * k[0], want)


def test_goldens_from_the_reference_collate():
    """The product's host logic (RNG order, parameter derivation) + the oracle's pixel arithmetic reproduce what the
    reference's own SameTrCollate returned for the same seeds (all eight gate combinations), and the draws leave numpy's
    and torch's global generators where augment_rng_after.json records them (its "source" says where that came from),
    draws that do not change a grey image (saturation / hue factors) included."""
    import json
    aug = import_module("htr-vt_b200.augment")
    g = np.load(os.path.join(G, "augment_cases.npz"))
    with open(os.path.join(G, "augment_rng_after.json")) as fh:
        nxt = json.load(fh)
    assert nxt["seeds"] == g["seeds"].tolist()
    args = _args(g)
    u8 = np.uint8(g["images"][:, 0] * 255)
    B, H, W = u8.shape
    combos = set()
    for seed, want, after in zip(g["seeds"], g["outputs"], nxt["next_np_torch"]):
        np.random.seed(int(seed)); torch.manual_seed(int(seed))
        p = aug.draw_collate_params(B, H, W, args)
        assert [np.random.rand(), float(torch.rand(1))] == after, int(seed)
        combos.add(tuple(p[k] is not None for k in ("warp", "morph", "jitter")))
        assert np.array_equal(A.apply_params(u8, p), want), int(seed)
    assert len(combos) == 8


def test_parameter_records():
    aug = import_module("htr-vt_b200.augment")
    ops = import_module("htr-vt_b200.ops")
    args = _args()
    np.random.seed(7); torch.manual_seed(7)                    # seed 7: all three gates (golden list)
    p = aug.draw_collate_params(3, 64, 256, args)
    assert all(p[k] is not None for k in ("warp", "morph", "jitter"))
    rec, morph = aug.pack_params(p, 3, 64, 256)
    assert rec.shape == (3, 128) and rec.dtype == np.uint8
    r = rec.view(aug._REC).reshape(3)
    assert (r["warp"] == 1).all() and (r["rows"] > 40).all() and (r["cols"] > 200).all()
    assert np.allclose(r["m"][:, 8], 1.0) and (r["jit_n"] <= 2).all()
    assert morph[0] in (1, 2) and 1 <= morph[1] <= 3 and 1 <= morph[2] <= 3 and morph[3] == 1
    # a projection value whose anti-aliasing filter needs more than three taps is refused, not approximated
    M, _ = p["warp"][0]
    with pytest.raises(ops.HtrvtError):
        aug.pack_params({"warp": [(M, (120, 256))] * 3, "morph": None, "jitter": None}, 3, 64, 256)
    # jitter strength 0 switches an op off without consuming a draw (torchvision _check_input)
    assert aug._jitter_range(0.0) is None and aug._jitter_range(0.4) == (0.6, 1.4)
    assert aug._jitter_range(0.2, center=0.0, bound=(-0.5, 0.5), clip_first_on_zero=False) == (-0.2, 0.2)
