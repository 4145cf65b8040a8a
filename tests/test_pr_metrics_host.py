"""CPU tests of the precision-recall reference (oracle/pr_oracle.py: pixel AP and F1-max with its threshold over a whole set) and of the
host side of the `--pr-metrics` / `--save-segmentation` options and of LocalisationAccumulator.results / segmentation."""
import importlib
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import pr_oracle as P

PKG = "anomaly-detection-super-resolution_b200"


def _tiny_set(seed):
    """4 small images, few distinct scores (many ties, negatives, both zeros), one image without defects."""
    rng = np.random.default_rng(seed)
    maps, masks = [], []
    for i in range(4):
        h, w = rng.integers(4, 9), rng.integers(4, 9)
        a = (rng.integers(-4, 5, (h, w)) / 2.0).astype(np.float32)
        a[rng.random((h, w)) < 0.2] = -0.0
        maps.append(a)
        m = np.zeros((h, w), np.uint8)
        if i:
            for _ in range(rng.integers(1, 4)):
                y, x = rng.integers(0, h), rng.integers(0, w)
                m[y:y + rng.integers(1, 4), x:x + rng.integers(1, 4)] = 255
        masks.append(m)
    return maps, masks


def brute_force_f1(maps, masks):
    """Every distinct score t, highest first, as a threshold: F1 of `score >= t` from TP / FP / FN, exact fractions; the first
    (highest) t of the best F1 wins."""
    s = np.concatenate([a.ravel() for a in maps]).astype(np.float64) + 0.0
    y = np.concatenate([(m != 0).ravel() for m in masks])
    best, best_t = Fraction(-1), None
    for t in np.unique(s)[::-1]:
        pred = s >= t
        tp, fp, fn = int((pred & y).sum()), int((pred & ~y).sum()), int((~pred & y).sum())
        f = Fraction(2 * tp, 2 * tp + fp + fn)
        if f > best:
            best, best_t = f, float(t)
    return best, best_t


def hand_ap(maps, masks):
    """Run by run: sum over the distinct scores (highest first) of (new defect pixels / N_def) * precision at that score."""
    s = np.concatenate([a.ravel() for a in maps]).astype(np.float64) + 0.0
    y = np.concatenate([(m != 0).ravel() for m in masks])
    n_def, ap, d_prev = int(y.sum()), 0.0, 0
    for t in np.unique(s)[::-1]:
        d, o = int((y & (s >= t)).sum()), int((~y & (s >= t)).sum())
        ap += (d - d_prev) / n_def * d / (d + o)
        d_prev = d
    return ap


@pytest.mark.parametrize("seed", range(8))
def test_oracle_f1_max_matches_brute_force(seed):
    maps, masks = _tiny_set(seed)
    want, want_t = brute_force_f1(maps, masks)
    f1, thr = P.f1_max(maps, masks)
    assert f1 == float(want) and thr == want_t
    assert not (thr == 0 and np.signbit(thr))                   # -0.0 is reported as +0.0


def test_oracle_f1_max_tie_goes_to_the_higher_threshold():
    # N_def = 2: at 5 F1 = 2 / (1 + 0 + 2) = 2/3, at 2 F1 = 4 / (2 + 2 + 2) = 2/3 as well; 5 wins
    a = np.array([[5, 4, 3, 2, 1]], np.float32)
    m = np.array([[1, 0, 0, 1, 0]], np.uint8)
    assert P.f1_max([a], [m]) == (2 / 3, 5.0)
    assert brute_force_f1([a], [m]) == (Fraction(2, 3), 5.0)
    # a defect run of -0.0 and +0.0 pixels: one threshold, +0.0
    z = np.array([[1.0, -0.0, 0.0, -0.0, -1.0]], np.float32)
    k = np.array([[0, 1, 1, 1, 0]], np.uint8)
    f1, thr = P.f1_max([z], [k])
    assert f1 == 2 * 3 / (3 + 1 + 3) and thr == 0.0 and not np.signbit(thr)


@pytest.mark.parametrize("seed", range(6))
def test_oracle_pixel_ap_matches_hand_computation(seed):
    maps, masks = _tiny_set(seed)
    assert abs(P.pixel_ap(maps, masks) - hand_ap(maps, masks)) <= 1e-12


def test_oracle_expected_values():
    masks = [np.zeros((4, 4), np.uint8), np.zeros((4, 4), np.uint8)]
    masks[1][1:3, 1:3] = 1
    flat = [np.full((4, 4), 0.5, np.float32) for _ in masks]
    assert P.pixel_ap(flat, masks) == pytest.approx(4 / 32, abs=1e-15)     # one run: the precision of everything
    assert P.f1_max(flat, masks) == (2 * 4 / (4 + 28 + 4), 0.5)
    sep = [np.where(m != 0, 2.0, 1.0).astype(np.float32) for m in masks]
    assert P.pixel_ap(sep, masks) == 1.0
    assert P.f1_max(sep, masks) == (1.0, 2.0)


def test_oracle_errors():
    a = np.zeros((4, 4), np.float32)
    with pytest.raises(ValueError):
        P.f1_max([a], [np.zeros((4, 4))])                               # no defect pixel
    m = np.zeros((4, 4))
    m[0, 0] = 1
    b = a.copy()
    b[1, 1] = np.nan
    with pytest.raises(ValueError):
        P.f1_max([b], [m])


def test_cli_pr_flags():
    evaluate = importlib.import_module(PKG + ".evaluate")
    a = evaluate.parse_args([])
    assert a.pr_metrics is False and a.save_segmentation is False
    a = evaluate.parse_args(["--mask-dir", "gt", "--pr-metrics", "--save-segmentation"])
    assert a.pr_metrics and a.save_segmentation
    assert evaluate.parse_args(["--save-segmentation", "--mask-dir", "gt"]).save_segmentation
    for bad in (["--pr-metrics"], ["--save-segmentation"], ["--pr-metrics", "--au-pro"], ["--save-segmentation", "--save-maps"]):
        with pytest.raises(SystemExit):
            evaluate.parse_args(bad)


def test_evaluate_on_test_checks_pr_flags_first():
    evaluate = importlib.import_module(PKG + ".evaluate")
    for kw in (dict(pr_metrics=True), dict(save_segmentation=True)):
        with pytest.raises(ValueError, match="mask_dir"):
            evaluate.evaluate_on_test(None, None, "", False, **kw)


def test_accumulator_results_errors_and_empty_segmentation():
    metrics = importlib.import_module(PKG + ".metrics")
    assert metrics.LocalisationMetrics._fields == ("pixel_auroc", "au_pro", "pixel_ap", "f1_max", "f1_threshold")
    acc = metrics.LocalisationAccumulator(2)
    for call in (acc.results, acc.finish):
        with pytest.raises(ValueError, match="fpr_limit"):
            call(0.0)
        with pytest.raises(ValueError, match="defect region"):
            call()
    assert acc.segmentation(1, 0.5) == []
    with pytest.raises(IndexError):
        acc.segmentation(2, 0.5)


def test_device_metrics_refuse_host_tensors():
    metrics = importlib.import_module(PKG + ".metrics")
    for fn in (metrics.pixel_ap, metrics.f1_max):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(torch.zeros(2, 4, 4), np.zeros((2, 4, 4)))
