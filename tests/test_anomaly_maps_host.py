"""CPU tests of the host side of the anomaly maps: pixel-level AUROC, the ground-truth mask lookup of the evaluator, the new command
line flags, and the up-front argument checks of ops.anomaly_maps."""
import importlib
import os

import numpy as np
import pytest
import torch
from PIL import Image

PKG = "anomaly-detection-super-resolution_b200"


@pytest.fixture(scope="module")
def metrics():
    return importlib.import_module(PKG + ".metrics")


@pytest.fixture(scope="module")
def evaluate():
    return importlib.import_module(PKG + ".evaluate")


def test_pixel_auroc_matches_sklearn_with_ties(metrics):
    from sklearn.metrics import roc_auc_score

    rng = np.random.default_rng(0)
    maps = rng.integers(0, 20, (5, 32, 48)).astype(np.float32) / 7.0      # few distinct values: many ties
    masks = (rng.random((5, 32, 48)) < 0.1).astype(np.uint8) * 255
    want = roc_auc_score((masks != 0).ravel(), maps.ravel())
    assert abs(metrics.pixel_auroc(maps, masks) - want) <= 1e-12
    # a list of per-image arrays of different sizes counts every pixel once
    lst_maps, lst_masks = [maps[0], maps[1, :16]], [masks[0], masks[1, :16]]
    want = roc_auc_score(np.concatenate([(m != 0).ravel() for m in lst_masks]), np.concatenate([m.ravel() for m in lst_maps]))
    assert abs(metrics.pixel_auroc(lst_maps, lst_masks) - want) <= 1e-12
    with pytest.raises(ValueError):
        metrics.pixel_auroc(maps, masks[:, :16])
    with pytest.raises(ValueError):
        metrics.pixel_auroc([maps[0]], [masks[0, :16]])


def test_mask_lookup_rules(tmp_path, evaluate):
    d = tmp_path / "masks"
    d.mkdir()
    Image.fromarray(np.zeros((8, 8), np.uint8)).save(d / "000.png")
    Image.fromarray(np.zeros((8, 8), np.uint8)).save(d / "001_mask.png")
    hr = lambda stem: str(tmp_path / "HR" / f"{stem}.png")
    assert evaluate.find_mask(str(d), hr("000"), 1) == str(d / "000.png")
    assert evaluate.find_mask(str(d), hr("001"), 1) == str(d / "001_mask.png")
    assert evaluate.find_mask(str(d), hr("002"), 0) is None          # good image without a mask: all clear
    with pytest.raises(FileNotFoundError) as e:                      # defective image without a mask
        evaluate.find_mask(str(d), hr("002"), 1)
    assert str(d / "002.png") in str(e.value) and str(d / "002_mask.png") in str(e.value)


def test_load_mask_crops_like_hr(tmp_path, evaluate):
    m = np.zeros((20, 22, 3), np.uint8)
    m[3, 4, 1] = 7                                                   # any non-zero channel marks a defect
    m[19, 21] = 255                                                  # outside the crop
    Image.fromarray(m).save(tmp_path / "m.png")
    got = evaluate.load_mask(str(tmp_path / "m.png"), (16, 20), (16, 20))
    assert got.shape == (16, 20) and got.dtype == bool and got.sum() == 1 and got[3, 4]
    assert not evaluate.load_mask(None, (16, 20), (16, 20)).any()
    with pytest.raises(ValueError):
        evaluate.load_mask(str(tmp_path / "m.png"), (16, 16), (16, 20))


def test_cli_parses_map_flags(evaluate):
    a = evaluate.parse_args([])
    assert (a.anomaly_maps, a.map_window_size, a.map_sigma, a.mask_dir, a.save_maps) == (False, 11, 4.0, None, False)
    a = evaluate.parse_args(["--anomaly-maps", "--map-window-size", "7", "--map-sigma", "0", "--mask-dir", "gt", "--save-maps"])
    assert (a.anomaly_maps, a.map_window_size, a.map_sigma, a.mask_dir, a.save_maps) == (True, 7, 0.0, "gt", True)


def test_anomaly_maps_refuses_cpu_and_bad_inputs():
    ops = importlib.import_module(PKG + ".ops")
    a = torch.zeros(1, 8, 8, 3, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.anomaly_maps(a, a, 3, 0.0)
