"""CPU tests of the MSGMS map's host side: the numpy reference (oracle/gms_oracle.py) against a torch fp64 transcription of RIAD's
formulation and against hand-computed values, the workspace size of the C side, the `--gms-map` option and ops.gms_map's refusal of
CPU tensors."""
import importlib
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from PIL import Image

from oracle import gms_oracle as G
from oracle import scoring_oracle as S

PKG = "anomaly-detection-super-resolution_b200"
ops = importlib.import_module(PKG + ".ops")
evaluate = importlib.import_module(PKG + ".evaluate")


def riad_msgms_torch(sr_u8: np.ndarray, hr_u8: np.ndarray) -> np.ndarray:
    """RIAD's MSGMS in torch fp64 on the gray planes of the 1 - SSIM map: F.conv2d with the Prewitt kernels and padding=1,
    F.avg_pool2d(2, 2), F.interpolate(bilinear, align_corners=False), c = 0.0026, 1e-12 under the square root."""
    x = torch.from_numpy(S.to_gray01(hr_u8).astype(np.float64))[None, None]
    y = torch.from_numpy(S.to_gray01(sr_u8).astype(np.float64))[None, None]
    hx = torch.tensor([[1 / 3, 0, -1 / 3]] * 3, dtype=torch.float64)[None, None]
    hy = hx.transpose(-1, -2)
    size = x.shape[-2:]

    def grad(p):
        return torch.sqrt(F.conv2d(p, hx, padding=1) ** 2 + F.conv2d(p, hy, padding=1) ** 2 + 1e-12)

    total = torch.zeros_like(x)
    for k in range(4):
        if k:
            x, y = F.avg_pool2d(x, kernel_size=2, stride=2), F.avg_pool2d(y, kernel_size=2, stride=2)
        gx, gy = grad(x), grad(y)
        gms = (2 * gx * gy + 0.0026) / (gx ** 2 + gy ** 2 + 0.0026)
        total = total + F.interpolate(1 - gms, size=size, mode="bilinear", align_corners=False)
    return (total / 4)[0, 0].numpy()


@pytest.mark.parametrize("c", [1, 3])
@pytest.mark.parametrize("h,w", [(128, 128), (64, 96), (100, 84)])
def test_oracle_matches_torch_riad(h, w, c):
    rng = np.random.default_rng(h * w + c)
    hr = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
    sr = np.clip(hr.astype(np.int16) + rng.integers(-40, 41, (h, w, c)), 0, 255).astype(np.uint8)
    for a, b in ((sr, hr), (rng.integers(0, 256, (h, w, c), dtype=np.uint8), hr)):
        want = riad_msgms_torch(a, b)
        got = G.gms_map(a, b)
        assert got.shape == (h, w)
        assert np.abs(got - want).max() <= 1e-12
    assert [d.shape for d in G.level_maps(sr, hr)] == [(h >> k, w >> k) for k in range(4)]   # 100 x 84: 50x42, 25x21, 12x10


def test_identical_pair_is_exactly_zero():
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (40, 56, 3), dtype=np.uint8)
    assert not G.gms_map(img, img).any()
    assert not G.gms_map(img, img, sigma=4.0).any()


def test_step_edge_level0_value():
    """HR: a vertical step 0 -> 1 at column j0, SR: flat 0.  Left of the edge gx(HR) = (0 - 1) * 3 / 3 = -1 and gy = 0, so
    g(HR) = sqrt(1 + 1e-12); g(SR) = sqrt(1e-12) everywhere."""
    h, w, j0 = 32, 32, 16
    hr = np.zeros((h, w, 1), np.uint8)
    hr[:, j0:] = 255
    sr = np.zeros_like(hr)
    a, b = math.sqrt(1.0 + 1e-12), math.sqrt(1e-12)
    want = 1.0 - (2 * a * b + 0.0026) / (a * a + b * b + 0.0026)
    d0 = G.level_maps(sr, hr)[0]
    for i in (5, 16, 26):
        assert abs(d0[i, j0 - 1] - want) <= 1e-15 and abs(d0[i, j0] - want) <= 1e-15
    assert abs(d0[16, 3] - 0.0) <= 1e-15                     # flat on both sides: g = 1e-6 in both images
    assert abs(G.gms_map(sr, hr)[16, j0 - 1] - riad_msgms_torch(sr, hr)[16, j0 - 1]) <= 1e-12


def test_workspace_bytes_cover_both_pyramids_and_the_level_planes():
    for b, h, w in ((256, 128, 128), (128, 256, 256), (3, 100, 84), (1, 8, 8), (0, 64, 64)):
        coarse = sum((h >> k) * (w >> k) for k in range(1, 4))
        assert ops.gms_workspace_bytes(b, h, w) == 4 * b * (2 * h * w + 3 * coarse)
    with pytest.raises(ValueError):
        ops.gms_workspace_bytes(-1, 8, 8)


def test_gms_map_refuses_cpu_tensors():
    a = torch.zeros(1, 8, 8, 3, dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.gms_map(a, a)


def test_cli_parses_gms_flag():
    assert evaluate.parse_args([]).gms_map is False
    a = evaluate.parse_args(["--gms-map", "--map-sigma", "2"])
    assert a.gms_map is True and a.map_sigma == 2.0 and a.anomaly_maps is False   # implied later, by evaluate_on_test


def test_evaluate_on_test_gms_map_implies_anomaly_maps(tmp_path, monkeypatch):
    """The evaluator is built with the maps and the MSGMS map on; stopped there, before any device work."""
    root = str(tmp_path / "data")
    rng = np.random.default_rng(0)
    for split in ("good", "bad"):
        for sub, side in (("HR", 32), ("LR_4", 8)):
            d = os.path.join(root, "grid", "test", split, sub)
            os.makedirs(d)
            Image.fromarray(rng.integers(0, 256, (side, side), dtype=np.uint8)).save(os.path.join(d, "000.png"))

    class Stop(Exception):
        pass

    seen = {}

    def fake_evaluator(model, rgb_range, window_sizes=None, maps=None, gms=False):
        seen.update(maps=maps, gms=gms)
        raise Stop

    model_mod = importlib.import_module(PKG + ".model")
    monkeypatch.setattr(model_mod, "Model", lambda opt, ckp: None)
    monkeypatch.setattr(evaluate, "BatchedEvaluator", fake_evaluator)

    class Opt:
        scale, data_root, classe, rgb_range = 4, root, "grid", 255

    with pytest.raises(Stop):
        evaluate.evaluate_on_test(Opt(), None, str(tmp_path / "out"), False, map_sigma=2.0, gms_map=True)
    assert seen == dict(maps=(11, 2.0), gms=True)
    with pytest.raises(Stop):
        evaluate.evaluate_on_test(Opt(), None, str(tmp_path / "out"), False)
    assert seen == dict(maps=None, gms=False)
