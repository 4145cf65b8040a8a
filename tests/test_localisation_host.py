"""CPU tests of the localisation metrics' reference (oracle/localisation_oracle.py: AU-PRO and pixel AUROC over a whole set) and of
the host side of the `--au-pro` option of the evaluator."""
import importlib

import numpy as np
import pytest
import torch
from scipy.ndimage import label

from oracle import localisation_oracle as L

PKG = "anomaly-detection-super-resolution_b200"


def brute_force_au_pro(maps, masks, alpha):
    """Every distinct score as a threshold: FPR = share of defect-free pixels >= t, PRO = mean over the regions of the share of the
    region's pixels >= t; (0, 0) first; trapezoids up to alpha with the crossing segment interpolated."""
    s = np.concatenate([np.asarray(a, np.float32).ravel() for a in maps]).astype(np.float64) + 0.0
    ok = np.concatenate([(np.asarray(m) == 0).ravel() for m in masks])
    regs = []
    off = 0
    for a, m in zip(maps, masks):
        lab, n = label(np.asarray(m) != 0, structure=np.ones((3, 3), int))
        regs += [off + np.flatnonzero(lab.ravel() == k) for k in range(1, n + 1)]
        off += np.asarray(a).size
    xs, ys = [0.0], [0.0]
    for t in np.unique(s)[::-1]:
        xs.append(float((s[ok] >= t).mean()))
        ys.append(float(np.mean([(s[r] >= t).mean() for r in regs])))
    tot = 0.0
    for i in range(len(xs) - 1):
        x0, x1, y0, y1 = xs[i], xs[i + 1], ys[i], ys[i + 1]
        if x0 >= alpha:
            break
        if x1 > alpha:
            y1 = y0 + (y1 - y0) * (alpha - x0) / (x1 - x0)
            x1 = alpha
        tot += (x1 - x0) * (y0 + y1) / 2
    return tot / alpha


def _tiny_set(seed):
    rng = np.random.default_rng(seed)
    maps, masks = [], []
    for i in range(4):
        h, w = rng.integers(5, 10), rng.integers(5, 10)
        maps.append((rng.integers(-6, 7, (h, w)) / 3.0).astype(np.float32))       # few distinct values: many ties, negatives, zeros
        m = np.zeros((h, w), np.uint8)
        if i:
            for _ in range(rng.integers(1, 4)):
                y, x = rng.integers(0, h), rng.integers(0, w)
                m[y:y + rng.integers(1, 4), x:x + rng.integers(1, 4)] = 255
        masks.append(m)
    return maps, masks


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("alpha", [0.05, 0.3, 1.0])
def test_oracle_matches_brute_force(seed, alpha):
    maps, masks = _tiny_set(seed)
    assert abs(L.au_pro(maps, masks, alpha) - brute_force_au_pro(maps, masks, alpha)) <= 1e-12


def test_oracle_pixel_auroc_is_sklearn():
    from sklearn.metrics import roc_auc_score

    maps, masks = _tiny_set(9)
    want = roc_auc_score(np.concatenate([(m != 0).ravel() for m in masks]), np.concatenate([a.ravel() for a in maps]))
    assert L.pixel_auroc(maps, masks) == want


def test_eight_connectivity():
    diag = np.eye(5, dtype=np.uint8)
    _, sizes = L.regions([diag])
    assert sizes.tolist() == [5]                                    # diagonal neighbours join one region
    checker = (np.indices((6, 6)).sum(0) % 2).astype(np.uint8)
    _, sizes = L.regions([checker])
    assert sizes.tolist() == [18]                                   # a checkerboard is one region
    two = np.zeros((4, 6), np.uint8)
    two[0, 0] = two[3, 5] = 1
    reg, sizes = L.regions([two, two])
    assert sizes.tolist() == [1, 1, 1, 1] and reg[1].max() == 3     # numbered across the images


def test_area_cut():
    fpr, pro = np.array([0.0, 0.2, 0.5, 1.0]), np.array([0.0, 0.6, 0.9, 1.0])
    # 0 .. 0.2: 0.06; 0.2 .. 0.3 with PRO(0.3) = 0.7 interpolated: 0.065
    assert L.area(fpr, pro, 0.3) == pytest.approx((0.06 + 0.065) / 0.3, abs=1e-15)
    assert L.area(fpr, pro, 1.0) == pytest.approx(0.06 + 0.225 + 0.475, abs=1e-15)
    assert L.area(fpr, pro, 0.5) == pytest.approx((0.06 + 0.225) / 0.5, abs=1e-15)   # alpha on a curve point: no cut
    # vertical segments add nothing
    assert L.area(np.array([0.0, 0.0, 1.0]), np.array([0.0, 0.5, 1.0]), 1.0) == pytest.approx(0.75, abs=1e-15)


def test_alpha_equal_to_a_curve_point():
    # 10 defect-free pixels, one 4-pixel region: alpha = 0.2 is the FPR after the two highest defect-free scores
    a = np.array([[9, 8, 8, 7, 6, 5, 4, 3, 2, 1, 0, -1, -2, -3]], np.float32)
    m = np.zeros_like(a, dtype=np.uint8)
    m[0, [0, 3, 4, 12]] = 1
    fpr, pro = L.curve([a], [m])
    assert 0.2 in fpr
    for alpha in (0.2, 0.25, 0.3, 1.0):
        assert L.au_pro([a], [m], alpha) == pytest.approx(brute_force_au_pro([a], [m], alpha), abs=1e-15)


def test_expected_values():
    rng = np.random.default_rng(1)
    masks = [(rng.random((16, 16)) < 0.2).astype(np.uint8) for _ in range(3)]
    flat = [np.full((16, 16), 0.5, np.float32) for _ in range(3)]
    assert L.au_pro(flat, masks, 0.3) == pytest.approx(0.15, abs=1e-15)   # one point (1, 1): area 0.045 / 0.3
    assert L.pixel_auroc(flat, masks) == 0.5
    sep = [np.where(m != 0, 2.0 + rng.random(m.shape), rng.random(m.shape)).astype(np.float32) for m in masks]
    assert L.au_pro(sep, masks, 0.3) == pytest.approx(1.0, abs=1e-12)
    assert L.pixel_auroc(sep, masks) == 1.0


def test_negative_zero_ties_positive_zero():
    a = np.array([[0.0, -0.0, 1.0, -1.0]], np.float32)
    m = np.array([[1, 0, 0, 1]], np.uint8)
    fpr, pro = L.curve([a], [m])
    assert len(fpr) == 4                                             # 1.0, 0.0 (both signs), -1.0


def test_oracle_errors():
    a = np.zeros((4, 4), np.float32)
    with pytest.raises(ValueError):
        L.au_pro([a], [np.zeros((4, 4))])                            # no defect region
    with pytest.raises(ValueError):
        L.au_pro([a], [np.ones((4, 4))])                             # no defect-free pixel
    m = np.zeros((4, 4))
    m[0, 0] = 1
    b = a.copy()
    b[1, 1] = np.nan
    with pytest.raises(ValueError):
        L.au_pro([b], [m])


def test_cli_au_pro_flag():
    evaluate = importlib.import_module(PKG + ".evaluate")
    assert evaluate.parse_args([]).au_pro is None
    assert evaluate.parse_args(["--mask-dir", "gt"]).au_pro is None
    assert evaluate.parse_args(["--mask-dir", "gt", "--au-pro"]).au_pro == 0.3
    assert evaluate.parse_args(["--au-pro", "--mask-dir", "gt"]).au_pro == 0.3
    assert evaluate.parse_args(["--mask-dir", "gt", "--au-pro", "0.05"]).au_pro == 0.05
    assert evaluate.parse_args(["--mask-dir", "gt", "--au-pro", "1"]).au_pro == 1.0
    for bad in (["--au-pro"], ["--au-pro", "0.3"], ["--mask-dir", "gt", "--au-pro", "0"], ["--mask-dir", "gt", "--au-pro", "1.5"],
                ["--mask-dir", "gt", "--au-pro", "-0.1"], ["--mask-dir", "gt", "--au-pro", "x"]):
        with pytest.raises(SystemExit):
            evaluate.parse_args(bad)


def test_evaluate_on_test_checks_au_pro_first():
    evaluate = importlib.import_module(PKG + ".evaluate")
    with pytest.raises(ValueError, match="mask_dir"):
        evaluate.evaluate_on_test(None, None, "", False, au_pro=0.3)
    with pytest.raises(ValueError, match=r"\(0, 1\]"):
        evaluate.evaluate_on_test(None, None, "", False, mask_dir="gt", au_pro=0.0)


def test_device_metrics_refuse_host_tensors():
    metrics = importlib.import_module(PKG + ".metrics")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.au_pro(torch.zeros(2, 4, 4), np.zeros((2, 4, 4)))
    acc = metrics.LocalisationAccumulator(1)
    with pytest.raises(ValueError, match="fpr_limit"):
        acc.finish(0.0)
    with pytest.raises(ValueError, match="defect region"):
        acc.finish(0.3)
