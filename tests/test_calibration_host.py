"""CPU tests of the calibrated-threshold reference (oracle/threshold_oracle.py: the inverted_cdf quantile, TP / FP / FN / TN and PRO
at a threshold), of the host side of LocalisationAccumulator.append(maps, masks=None) / quantile / at_threshold, and of the
`--calibration-dir` / `--calibration-quantile` / `--save-calibrated-masks` options."""
import importlib
import math
import os
from fractions import Fraction

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import threshold_oracle as T

PKG = "anomaly-detection-super-resolution_b200"
metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")
ops = importlib.import_module(PKG + ".ops")


def test_inverted_cdf_rank_matches_numpy():
    rng = np.random.default_rng(0)
    qs = [0.0, 1e-9, 0.1, 0.14, 0.2, 0.28, 0.3, 0.5, 0.56, 0.7, 0.9, 0.999, 1.0] + list(rng.random(40))
    for n in [1, 2, 3, 7, 10, 25, 50, 100, 1000, 1001, 12345, 2 ** 24 + 3]:
        x = np.arange(n, dtype=np.float64) if n < 100000 else None
        for q in qs:
            k = metrics.inverted_cdf_rank(n, q)
            assert 1 <= k <= n
            if x is not None:
                assert np.quantile(x, q, method="inverted_cdf") == k - 1, (n, q, k)
    assert metrics.inverted_cdf_rank(25, 0.28) == 8        # 0.28 * 25 rounds to 7.000000000000001 in float64, as numpy forms it
    assert metrics.inverted_cdf_rank(10, 0.3) == 3 and metrics.inverted_cdf_rank(10, 0.7) == 7
    assert metrics.inverted_cdf_rank(5, 0.0) == 1 and metrics.inverted_cdf_rank(5, 1.0) == 5


def test_oracle_quantile_forms_the_rank_in_float64():
    """numpy forms q n in the input's dtype: the oracle converts fp32 scores to float64 (exact) so that the rank is formed in float64."""
    x = np.arange(2880, dtype=np.float32).reshape(48, 60)
    assert np.quantile(x, 0.3, method="inverted_cdf") == 864                # fp32: 0.3 * 2880 rounds above 864, rank 865
    assert T.quantile([x], 0.3) == 863 == metrics.inverted_cdf_rank(2880, 0.3) - 1


def test_fp32_at_least():
    for t in (0.1, -0.1, 1.0, 3e38, -3e38, 1e-45, 0.0, 2.5):
        f = metrics.fp32_at_least(t)
        assert f.dtype == np.float32 and float(f) >= t
        assert float(np.nextafter(f, np.float32(-np.inf))) < t or float(f) == t


@pytest.mark.parametrize("seed", range(6))
def test_oracle_quantile_matches_brute_force(seed):
    rng = np.random.default_rng(seed)
    maps = [(rng.integers(-5, 6, (rng.integers(1, 6), rng.integers(1, 6))) / 2).astype(np.float32) for _ in range(3)]
    maps[0][0, 0] = -0.0
    s = sorted(float(v) + 0.0 for a in maps for v in a.ravel())
    n = len(s)
    for q in (0.0, 0.25, 0.3, 0.5, 0.7, 1.0, rng.random()):
        k = max(1, math.ceil(Fraction(q) * n))              # exact arithmetic on the double q
        want = s[k - 1]
        got = T.quantile(maps, q)
        assert got == s[metrics.inverted_cdf_rank(n, q) - 1] and not (got == 0 and np.signbit(got))
        if metrics.inverted_cdf_rank(n, q) == k:
            assert got == want


def brute_force_counts(maps, masks, t):
    """Pixel by pixel, regions by a flood fill over the 8 neighbours; PRO as an exact fraction."""
    tp = fp = fn = tn = 0
    hits, sizes = [], []
    for a, m in zip(maps, masks):
        h, w = m.shape
        lab = -np.ones((h, w), int)
        for y in range(h):
            for x in range(w):
                if m[y, x] and lab[y, x] < 0:
                    lab[y, x] = len(sizes)
                    stack, size, hit = [(y, x)], 0, 0
                    while stack:
                        cy, cx = stack.pop()
                        size += 1
                        hit += float(a[cy, cx]) >= t
                        for dy in (-1, 0, 1):
                            for dx in (-1, 0, 1):
                                ny, nx = cy + dy, cx + dx
                                if 0 <= ny < h and 0 <= nx < w and m[ny, nx] and lab[ny, nx] < 0:
                                    lab[ny, nx] = len(sizes)
                                    stack.append((ny, nx))
                    sizes.append(size)
                    hits.append(hit)
                pred, d = float(a[y, x]) >= t, bool(m[y, x])
                tp += pred and d
                fp += pred and not d
                fn += d and not pred
                tn += not pred and not d
    pro = float(sum(Fraction(h, s) for h, s in zip(hits, sizes)) / len(sizes)) if sizes else float("nan")
    return tp, fp, fn, tn, pro


@pytest.mark.parametrize("seed", range(6))
def test_oracle_counts_match_brute_force(seed):
    rng = np.random.default_rng(seed + 10)
    maps, masks = [], []
    for i in range(3):
        h, w = rng.integers(3, 10), rng.integers(3, 10)
        maps.append((rng.integers(-4, 5, (h, w)) / 4).astype(np.float32))
        m = np.zeros((h, w), np.uint8)
        if i:
            m[rng.random((h, w)) < 0.3] = 1
        masks.append(m)
    values = np.unique(np.concatenate([a.ravel() for a in maps]).astype(np.float64))
    for t in list(values) + [values.min() - 1, values.max() + 1, (values[0] + values[1]) / 2, 0.1]:
        got = T.counts(maps, masks, t)
        want = brute_force_counts(maps, masks, t)
        assert got[:4] == want[:4], t
        assert (math.isnan(got[4]) and math.isnan(want[4])) or abs(got[4] - want[4]) <= 1e-15, t
    empty = [np.zeros(a.shape, np.uint8) for a in maps]
    assert math.isnan(T.counts(maps, empty, 0.0)[4])


def test_oracle_refuses_nan():
    a = np.zeros((3, 3), np.float32)
    a[1, 1] = np.nan
    for call in (lambda: T.quantile([a], 0.5), lambda: T.counts([a], [np.zeros((3, 3))], 0.0)):
        with pytest.raises(ValueError):
            call()


# ------------------------------------------------------------------------------------------------------------- accumulator
def test_append_without_masks_bookkeeping(monkeypatch):
    """masks=None: every pixel defect-free, no regions, n_ok grows by the pixel count; a later masked append labels as before.
    (The device check is lifted so that the bookkeeping runs on host tensors.)"""
    monkeypatch.setattr(ops, "_cuda", lambda t, name: None)
    acc = metrics.LocalisationAccumulator(2)
    a = torch.arange(2 * 3 * 4, dtype=torch.float32).reshape(2, 3, 4)
    acc.append([a, -a])
    assert (acc.n, acc.n_ok, acc.n_regions) == (24, 24, 0) and acc._shapes == [(3, 4), (3, 4)]
    assert torch.equal(acc._regions[:24], torch.full((24,), -1, dtype=torch.int32))
    assert torch.equal(acc._maps[0][:24], a.reshape(-1)) and torch.equal(acc._maps[1][:24], -a.reshape(-1))
    b = [torch.ones(2, 5), torch.zeros(4, 4)]
    acc.append([b, b])                                       # a sequence of mixed sizes
    assert (acc.n, acc.n_ok) == (24 + 26, 24 + 26) and acc._shapes[2:] == [(2, 5), (4, 4)]
    m = np.zeros((3, 4), np.uint8)
    m[0, 0] = m[2, 3] = 1
    acc.append([a[:1], a[:1]], [m])
    assert (acc.n, acc.n_ok, acc.n_regions) == (62, 60, 2)
    assert acc._regions[50:62].tolist() == [0] + [-1] * 10 + [1]
    with pytest.raises(ValueError, match="same images"):
        acc.append([a, a[:1]])
    with pytest.raises(ValueError, match="3 maps given"):
        acc.append([a, a, a])


def test_quantile_and_at_threshold_argument_errors():
    assert metrics.ThresholdMetrics._fields == ("threshold", "tp", "fp", "fn", "tn", "precision", "recall", "fpr", "f1", "iou", "pro")
    acc = metrics.LocalisationAccumulator(2)
    for q in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError, match="q must be"):
            acc.quantile(0, q)
    with pytest.raises(ValueError, match="no scores"):
        acc.quantile(1, 0.5)
    with pytest.raises(ValueError, match="NaN"):
        acc.at_threshold(0, float("nan"))
    with pytest.raises(ValueError, match="no scores"):
        acc.at_threshold(0, 0.5)
    for call in (acc.quantile, acc.at_threshold):
        with pytest.raises(IndexError):
            call(2, 0.5)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.score_quantile(torch.zeros(2, 4, 4), 0.5)


# ------------------------------------------------------------------------------------------------------------- CLI
def test_cli_calibration_flags():
    a = evaluate.parse_args([])
    assert a.calibration_dir is None and a.calibration_quantile == 0.999 and a.save_calibrated_masks is False
    a = evaluate.parse_args(["--calibration-dir", "cal", "--calibration-quantile", "0.99", "--save-calibrated-masks"])
    assert a.calibration_dir == "cal" and a.calibration_quantile == 0.99 and a.save_calibrated_masks
    assert evaluate.parse_args(["--calibration-dir", "cal", "--calibration-quantile", "1"]).calibration_quantile == 1.0
    for bad in (["--save-calibrated-masks"], ["--calibration-dir", "cal", "--calibration-quantile", "0"],
                ["--calibration-dir", "cal", "--calibration-quantile", "1.5"], ["--calibration-quantile", "-0.5"],
                ["--calibration-dir", "cal", "--calibration-quantile", "nan"]):
        with pytest.raises(SystemExit):
            evaluate.parse_args(bad)


def test_evaluate_on_test_checks_calibration_flags_first():
    with pytest.raises(ValueError, match="calibration_quantile"):
        evaluate.evaluate_on_test(None, None, "", False, calibration_dir="cal", calibration_quantile=0.0)
    with pytest.raises(ValueError, match="calibration_dir"):
        evaluate.evaluate_on_test(None, None, "", False, save_calibrated_masks=True)


def _write_split(d, n, side, scale=4):
    rng = np.random.default_rng(n + side)
    for sub in ("HR", f"LR_{scale}"):
        os.makedirs(os.path.join(d, sub), exist_ok=True)
    for i in range(n):
        Image.fromarray(rng.integers(0, 256, (side, side), dtype=np.uint8)).save(os.path.join(d, "HR", f"{i:03d}.png"))
        Image.fromarray(rng.integers(0, 256, (side // scale, side // scale), dtype=np.uint8)).save(
            os.path.join(d, f"LR_{scale}", f"{i:03d}.png"))


def test_calibration_images_must_have_the_test_size(tmp_path):
    """The size check runs on the PNG headers before any model is built (no GPU needed to reach it)."""
    root = str(tmp_path / "data")
    _write_split(os.path.join(root, "grid", "test", "good"), 2, 32)
    _write_split(os.path.join(root, "grid", "test", "bad"), 2, 32)
    _write_split(str(tmp_path / "cal_bad"), 2, 48)
    os.makedirs(str(tmp_path / "empty" / "HR"))

    class Opt:
        scale, data_root, classe = 4, root, "grid"

    with pytest.raises(ValueError, match=r"calibration image .*000\.png is 48x48, the test images are 32x32"):
        evaluate.evaluate_on_test(Opt(), None, str(tmp_path / "out"), False, calibration_dir=str(tmp_path / "cal_bad"))
    with pytest.raises(ValueError, match="no calibration images"):
        evaluate.evaluate_on_test(Opt(), None, str(tmp_path / "out"), False, calibration_dir=str(tmp_path / "empty"))
    assert not os.path.exists(str(tmp_path / "out"))
