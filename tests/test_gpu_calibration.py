"""GPU tests of the calibrated thresholds (csrc/localisation.cu adsr_score_quantile / adsr_threshold_metrics through
metrics.LocalisationAccumulator.quantile / at_threshold and metrics.score_quantile): the quantile equals numpy's inverted_cdf quantile
of the scores as float64 exactly (ties, negative scores, +-3e38, -0.0, n = 1, mixed sizes, more than 2^24 pixels), the counts at a threshold equal the oracle
exactly and PRO within 1e-12, F1 at the F1-max threshold equals F1-max bit for bit, results do not depend on the batching; then
`--calibration-dir --save-calibrated-masks` end to end."""
import importlib
import math
import os
import shutil

import numpy as np
import pytest
import torch
from PIL import Image
from scipy.ndimage import gaussian_filter

from gpu_common import PKG
from oracle import drct_oracle as O
from oracle import threshold_oracle as T
from test_gpu_anomaly_maps import _dataset_with_masks
from test_gpu_pr_metrics import _blob_masks, _device

pytestmark = pytest.mark.gpu

metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")

QS = (0.0, 1e-9, 0.3, 0.5, 0.999, 1.0)


def check_quantiles(maps, acc=None):
    """Every q of QS: the device quantile of host maps (list input) equals numpy's inverted_cdf quantile, +0.0 for a zero."""
    if acc is None:
        acc = metrics.LocalisationAccumulator(1)
        acc.append([_device(maps)])
    got = [acc.quantile(0, q) for q in QS]
    for q, g in zip(QS, got):
        assert g == T.quantile(maps, q), (q, g, T.quantile(maps, q))
        assert not (g == 0 and np.signbit(g)), q
    return got


def test_quantile_heavy_ties():
    rng = np.random.default_rng(20)
    maps = [(np.round(rng.random((50, 20)) * 6) / 4).astype(np.float32) for _ in range(4)]   # n = 4000: q n integer for 0.3, 0.5, 0.999
    check_quantiles(maps)


def test_quantile_negative_huge_and_signed_zeros():
    rng = np.random.default_rng(21)
    maps = []
    for _ in range(5):
        a = (rng.integers(-4, 5, (40, 25)) / 2.0).astype(np.float32)
        a[rng.random(a.shape) < 0.3] = -0.0
        a[rng.random(a.shape) < 0.05] = np.float32(3e38)
        a[rng.random(a.shape) < 0.05] = np.float32(-3e38)
        maps.append(a)
    check_quantiles(maps)
    zeros = [np.where(rng.random((10, 10)) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32) for _ in range(3)]
    assert set(check_quantiles(zeros)) == {0.0}
    neg = [np.full((3, 3), -0.0, np.float32)]                  # only -0.0: reported as +0.0
    assert check_quantiles(neg) == [0.0] * len(QS)


def test_quantile_single_pixel_and_mixed_sizes():
    assert check_quantiles([np.array([[-2.5]], np.float32)]) == [-2.5] * len(QS)
    rng = np.random.default_rng(22)
    shapes = [(17, 33), (64, 40), (5, 7), (1, 1), (128, 96)]
    maps = [rng.standard_normal(s).astype(np.float32) for s in shapes]
    check_quantiles(maps)
    stack = torch.from_numpy(np.stack([rng.random((24, 24)).astype(np.float32) for _ in range(5)])).cuda()
    for q in QS:
        assert metrics.score_quantile(stack, q) == metrics.score_quantile(list(stack.unbind(0)), q) == T.quantile(list(stack.cpu()), q)


def test_quantile_beyond_torch_quantile_limit():
    n_img, h, w = 264, 256, 256
    g = torch.Generator(device="cuda").manual_seed(23)
    maps = torch.round(torch.rand(n_img, h, w, generator=g, device="cuda") * 5000) / 1000
    assert maps.numel() > 2 ** 24
    with pytest.raises(RuntimeError, match="too large"):
        torch.quantile(maps.reshape(-1), 0.5)
    acc = metrics.LocalisationAccumulator(1)
    for s in range(0, n_img, 64):
        acc.append([maps[s:s + 64]])
    check_quantiles(list(maps.cpu().numpy()), acc)


def test_quantile_nan_raises():
    a = np.zeros((8, 8), np.float32)
    a[3, 4] = np.nan
    with pytest.raises(ValueError, match="NaN"):
        metrics.score_quantile(_device([a]), 0.5)


# ------------------------------------------------------------------------------------------------------------- threshold metrics
def check_threshold(maps, masks, acc, t):
    r = acc.at_threshold(0, t)
    tp, fp, fn, tn, pro = T.counts(maps, masks, t)
    assert (r.tp, r.fp, r.fn, r.tn) == (tp, fp, fn, tn), (t, r, (tp, fp, fn, tn))
    assert (math.isnan(pro) and math.isnan(r.pro)) or abs(r.pro - pro) <= 1e-12, (t, r.pro, pro)
    assert r.threshold == t and r.precision == (tp / (tp + fp) if tp + fp else 0.0)
    if tp + fn:
        assert r.recall == tp / (tp + fn) and r.f1 == 2 * tp / (2 * tp + fp + fn) and r.iou == tp / (tp + fp + fn)
    assert r.fpr == fp / (fp + tn)
    return r


def _thresholds(maps, rng):
    v = np.unique(np.concatenate([a.ravel() for a in maps]).astype(np.float64))
    picks = list(rng.choice(v, min(8, len(v)), replace=False)) + [v.min(), v.max()]
    between = [(v[i] + v[i + 1]) / 2 for i in rng.integers(0, len(v) - 1, 4)] if len(v) > 1 else []
    return picks + between + [v.min() - 1.0, v.max() + 1.0, float(np.nextafter(np.float32(v[len(v) // 2]), np.float32(np.inf))) - 1e-12]


@pytest.mark.parametrize("kind", ["ties", "smoothed", "negative"])
def test_threshold_metrics_match_oracle(kind):
    rng = np.random.default_rng({"ties": 30, "smoothed": 31, "negative": 32}[kind])
    masks = _blob_masks(rng, 10, 48, 40)
    if kind == "ties":
        maps = [(np.round(rng.random((48, 40)) * 12 + 4 * (m != 0)) / 8).astype(np.float32) for m in masks]
    elif kind == "smoothed":
        maps = [gaussian_filter((rng.random((48, 40)) + 0.8 * (m != 0)).astype(np.float32), 3.0) for m in masks]
    else:
        maps = [np.where(rng.random((48, 40)) < 0.2, np.float32(-0.0), (rng.integers(-3, 4, (48, 40)) / 2.0)).astype(np.float32)
                for _ in masks]
    acc = metrics.LocalisationAccumulator(1)
    acc.append([_device(maps)], masks)
    for t in _thresholds(maps, rng):
        check_threshold(maps, masks, acc, t)
    r = check_threshold(maps, masks, acc, -1e30)               # everything predicted
    assert r.recall == 1.0 and r.fpr == 1.0 and abs(r.pro - 1.0) <= 1e-12   # floor(2^63 / |r|) weights: 1 to within 2^-60
    r = check_threshold(maps, masks, acc, 1e30)                # nothing predicted
    assert r.tp == r.fp == 0 and r.precision == 0.0 and r.pro == 0.0


def test_threshold_metrics_mixed_sizes_and_no_regions():
    rng = np.random.default_rng(33)
    shapes = [(17, 33), (64, 40), (5, 7), (128, 96)]
    masks = [_blob_masks(rng, 1, h, w, 1.0)[0] for h, w in shapes]
    maps = [(np.round(rng.random(s) * 30) / 7).astype(np.float32) for s in shapes]
    acc = metrics.LocalisationAccumulator(1)
    acc.append([_device(maps)], masks)
    for t in _thresholds(maps, rng):
        check_threshold(maps, masks, acc, t)
    clean = metrics.LocalisationAccumulator(1)                 # defect-free images only: no region, PRO and recall are NaN
    clean.append([_device(maps)])
    empty = [np.zeros(s, np.uint8) for s in shapes]
    r = check_threshold(maps, empty, clean, 2.0)
    assert math.isnan(r.pro) and math.isnan(r.recall) and r.tp == r.fn == 0


def test_f1_at_the_f1_max_threshold_and_segmentation():
    rng = np.random.default_rng(34)
    masks = _blob_masks(rng, 16, 64, 64)
    ssim = [gaussian_filter((rng.random((64, 64)) + 0.6 * (m != 0)).astype(np.float32), 2.0) for m in masks]
    se = [(np.round(rng.random((64, 64)) * 50 + 20 * (m != 0)) / 100).astype(np.float32) for m in masks]
    acc = metrics.LocalisationAccumulator(2)
    acc.append([_device(ssim), _device(se)], masks)
    for j, res in enumerate(acc.results()):
        r = acc.at_threshold(j, res.f1_threshold)
        assert r.f1 == res.f1_max, (j, r.f1, res.f1_max)
        seg = acc.segmentation(j, res.f1_threshold)
        assert r.tp + r.fp == sum(int(s.sum()) for s in seg)
        t = res.f1_threshold + 1e-9                            # not an fp32 value: rounded up like segmentation()
        assert acc.at_threshold(j, t).tp + acc.at_threshold(j, t).fp == sum(int(s.sum()) for s in acc.segmentation(j, t))


def test_bitwise_deterministic_and_batch_independent():
    rng = np.random.default_rng(35)
    n = 128
    masks = _blob_masks(rng, n, 64, 64)
    ssim = np.stack([gaussian_filter(rng.random((64, 64)).astype(np.float32), 2.0) for _ in range(n)])
    se = (np.round(rng.random((n, 64, 64)) * 100) / 100).astype(np.float32)
    d_ssim, d_se = torch.from_numpy(ssim).cuda(), torch.from_numpy(se).cuda()
    ts = (0.25, 0.5, float(np.float32(0.37)))
    results = []
    for bs in (8, 64, 128, 8):
        acc, cal = metrics.LocalisationAccumulator(2), metrics.LocalisationAccumulator(2)
        for s in range(0, n, bs):
            acc.append([d_ssim[s:s + bs], d_se[s:s + bs]], masks[s:s + bs])
            cal.append([d_ssim[s:s + bs], d_se[s:s + bs]])
        results.append(([acc.at_threshold(j, t) for j in range(2) for t in ts], [cal.quantile(j, q) for j in range(2) for q in QS]))
    assert all(r == results[0] for r in results), results
    assert results[0][1] == [T.quantile(list(m), q) for m in (ssim, se) for q in QS]


# ------------------------------------------------------------------------------------------------------------- evaluator
def test_evaluate_cli_calibration(tmp_path, capsys, monkeypatch):
    n, q = 16, 0.99
    root = str(tmp_path / "mvtec_128")
    _, _, labels, masks = _dataset_with_masks(root, "carpet", 3, n, seed=78)
    other = str(tmp_path / "other")
    _dataset_with_masks(other, "carpet", 3, 12, seed=79)       # its 6 good images become the defect-free calibration split
    cal_dir = os.path.join(root, "carpet", "train", "good")
    shutil.move(os.path.join(other, "carpet", "test", "good"), cal_dir)
    sd = O.make_state_dict(O.DrctCfg(num_layers=1), seed=4)
    ckpt = str(tmp_path / "model_best.pt")
    torch.save(sd, ckpt)
    orig = evaluate.setup_opt_drct

    def one_rdg(*a, **k):
        opt = orig(*a, **k)
        opt.depths, opt.num_heads = (6,), (6,)
        return opt

    monkeypatch.setattr(evaluate, "setup_opt_drct", one_rdg)
    built = []

    class Recording(evaluate.BatchedEvaluator):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            built.append(self)

    monkeypatch.setattr(evaluate, "BatchedEvaluator", Recording)
    out_dir = str(tmp_path / "out")
    mask_dir = os.path.join(root, "masks")
    argv = ["--model-type", "drct", "--classe", "carpet", "--scale", "4", "--resolution", "128", "--data-root", root,
            "--checkpoint", ckpt, "--batch-size", "8", "--output-dir", out_dir, "--mask-dir", mask_dir]
    plain = evaluate.main(argv)
    plain_lines = capsys.readouterr().out.strip().splitlines()
    res = evaluate.main(argv + ["--calibration-dir", cal_dir, "--calibration-quantile", str(q), "--save-calibrated-masks",
                                "--save-maps"])
    lines = capsys.readouterr().out.strip().splitlines()

    cal_keys = {f"calib_{k}_{m}" for k in ("pixel_threshold", "image_threshold", "image_tpr", "image_fpr", "pixel_precision",
                                           "pixel_recall", "pixel_fpr", "pixel_f1", "pixel_iou", "pixel_pro") for m in ("ssim", "se")}
    assert cal_keys <= set(res) and not cal_keys & set(plain)
    assert not any(l.startswith("Map CAL") for l in plain_lines)
    cal_at = [i for i, l in enumerate(lines) if l.startswith("Map CAL - ")]
    assert len(cal_at) == 1 and not any(l.startswith("Map ") for l in lines[:cal_at[0]])
    after = lines[cal_at[0] + 1:]
    assert after == plain_lines[-len(after):]                 # every line after Map CAL is that of the run without it
    assert np.array_equal(res["scores"], plain["scores"]) and np.array_equal(res["map_max"], plain["map_max"])

    # the calibration maps, recomputed with the evaluator's own model on the same batch: the thresholds are their numpy quantiles
    ev = evaluate.BatchedEvaluator(built[-1].model, 255.0, built[-1].window_sizes, maps=(11, 4.0))
    ev.use_graph = False
    pairs = [evaluate.load_pair(h, l, 4, 3, 255.0, raw_u8=True) for h, l in zip(*evaluate.scan_split(cal_dir, 4))]
    assert len(pairs) == 6
    with torch.no_grad():
        ev.step(torch.stack([p[0] for p in pairs]), torch.stack([p[1] for p in pairs]))
    cal_maps = [ev.last_maps[j].cpu().numpy() for j in range(2)]
    cal_max = ev.last_maps[2].cpu().numpy()

    order = np.argsort(labels, kind="stable")                  # evaluator order: good first, then bad; names sorted
    mk = [masks[i] for i in order]
    y = labels[order]
    split = lambda i: "good" if labels[i] == 0 else "bad"
    parts = []
    for j, (kind, label) in enumerate((("ssim", "1-SSIM"), ("se", "SE"))):
        t_px, t_img = res[f"calib_pixel_threshold_{kind}"], res[f"calib_image_threshold_{kind}"]
        assert t_px == T.quantile(list(cal_maps[j]), q) == float(np.quantile(cal_maps[j].astype(np.float64), q, method="inverted_cdf"))
        assert t_img == float(np.quantile(cal_max[:, j], q, method="inverted_cdf")), kind
        assert (cal_maps[j] > t_px).mean() <= 1 - q + 1e-12 and (cal_max[:, j] > t_img).mean() <= 1 - q + 1e-12

        maps = [np.load(os.path.join(out_dir, "maps", split(i), f"{i:03d}_{kind}.npy")) for i in order]
        for i, m in zip(order, maps):
            png = np.array(Image.open(os.path.join(out_dir, "calibrated", split(i), f"{i:03d}_{kind}.png")))
            assert png.dtype == np.uint8 and set(np.unique(png)) <= {0, 255}
            assert np.array_equal(png == 255, m > np.float32(t_px)), (kind, i)
        flagged = np.array([m.max() > t_img for m in maps])
        tpr, fpr = flagged[y == 1].mean(), flagged[y == 0].mean()
        assert (res[f"calib_image_tpr_{kind}"], res[f"calib_image_fpr_{kind}"]) == (tpr, fpr), kind
        tp, fp, fn, tn, pro = T.counts(maps, mk, float(np.nextafter(np.float32(t_px), np.float32(np.inf))))
        assert tp + fp == sum(int((m > np.float32(t_px)).sum()) for m in maps)
        want = dict(precision=tp / (tp + fp) if tp + fp else 0.0, recall=tp / (tp + fn), fpr=fp / (fp + tn),
                    f1=2 * tp / (2 * tp + fp + fn), iou=tp / (tp + fp + fn))
        for k, v in want.items():
            assert res[f"calib_pixel_{k}_{kind}"] == v, (kind, k)
        assert abs(res[f"calib_pixel_pro_{kind}"] - pro) <= 1e-12, kind
        parts.append(f"{label} t_px {t_px:g}, t_img {t_img:g}, image TPR {tpr:.4f}, FPR {fpr:.4f}, pixel precision "
                     f"{want['precision']:.4f}, recall {want['recall']:.4f}, FPR {want['fpr']:.4f}, F1 {want['f1']:.4f}, "
                     f"IoU {want['iou']:.4f}, PRO {res[f'calib_pixel_pro_{kind}']:.4f}")
    assert lines[cal_at[0]] == f"Map CAL - q={q:g} on 6 defect-free images: " + "; ".join(parts)

    # without masks: the thresholds and the image decisions only, the same values
    no_masks = [a for a in argv if a not in ("--mask-dir", mask_dir)]
    res2 = evaluate.main(no_masks + ["--calibration-dir", cal_dir, "--calibration-quantile", str(q)])
    lines2 = capsys.readouterr().out.strip().splitlines()
    keys2 = {k for k in cal_keys if "calib_pixel_threshold" in k or "calib_image" in k}
    assert {k for k in res2 if k.startswith("calib_")} == keys2 and all(res2[k] == res[k] for k in keys2)
    assert lines2[-3].startswith("Map CAL - ") and "pixel precision" not in lines2[-3]
