"""GPU tests of the precision-recall half of the localisation metrics (csrc/localisation.cu through
metrics.LocalisationAccumulator.results / segmentation, metrics.pixel_ap / f1_max): pixel AP against sklearn (|d| <= 1e-9), F1-max
against oracle/pr_oracle.py (|d| <= 1e-12) and its threshold equal, on ties, smoothed maps, negative scores and -0.0, tiny and border
regions, defect-free and all-defect images, mixed image sizes and more than 2^24 pixels; the threshold's masks recount F1-max exactly;
results() agrees with finish() bit for bit; determinism and batch independence; then `--pr-metrics --save-segmentation` end to end."""
import importlib
import os

import numpy as np
import pytest
import torch
from PIL import Image
from scipy.ndimage import gaussian_filter

from gpu_common import PKG
from oracle import drct_oracle as O
from oracle import pr_oracle as P
from test_gpu_anomaly_maps import _dataset_with_masks

pytestmark = pytest.mark.gpu

metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")


def _device(maps):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in maps]


def _f1_of(pred, masks):
    """F1 of predicted bool masks against ground-truth masks, recounted from TP / FP / FN."""
    tp = sum(int((p & (m != 0)).sum()) for p, m in zip(pred, masks))
    fp = sum(int((p & (m == 0)).sum()) for p, m in zip(pred, masks))
    fn = sum(int((~p & (m != 0)).sum()) for p, m in zip(pred, masks))
    return 2 * tp / (2 * tp + fp + fn)


def check(maps, masks, acc=None):
    """Device results of host maps / masks (list input) against sklearn and the oracle; returns the LocalisationMetrics."""
    if acc is None:
        acc = metrics.LocalisationAccumulator(1)
        acc.append([_device(maps)], masks)
    r, = acc.results()
    want_ap = P.pixel_ap(maps, masks)
    want_f1, want_t = P.f1_max(maps, masks)
    assert abs(r.pixel_ap - want_ap) <= 1e-9, (r.pixel_ap, want_ap)
    assert abs(r.f1_max - want_f1) <= 1e-12, (r.f1_max, want_f1)
    assert r.f1_threshold == want_t and not (r.f1_threshold == 0 and np.signbit(r.f1_threshold)), (r.f1_threshold, want_t)
    assert acc.finish() == [(r.pixel_auroc, r.au_pro)]                  # the same bits through both entry points
    seg = acc.segmentation(0, r.f1_threshold)
    assert [s.shape for s in seg] == [np.shape(m) for m in masks] and all(s.dtype == bool for s in seg)
    assert all(np.array_equal(s, np.asarray(a, np.float32) >= np.float32(r.f1_threshold)) for s, a in zip(seg, maps))
    assert _f1_of(seg, masks) == r.f1_max
    return r


def _blob_masks(rng, n, h, w, p_defect=0.7):
    masks = []
    for _ in range(n):
        m = np.zeros((h, w), np.uint8)
        if rng.random() < p_defect:
            for _ in range(rng.integers(1, 4)):
                y, x = rng.integers(0, h), rng.integers(0, w)
                m[y:y + rng.integers(1, max(2, h // 3)), x:x + rng.integers(1, max(2, w // 3))] = 255
            yy, xx = np.mgrid[:h, :w]
            cy, cx, r = rng.integers(0, h), rng.integers(0, w), rng.integers(2, 8)
            m[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = 255
        masks.append(m)
    if not any(m.any() for m in masks):
        masks[0][0, 0] = 255
    return masks


def test_many_ties():
    rng = np.random.default_rng(10)
    masks = _blob_masks(rng, 12, 64, 64)
    maps = [(np.round(rng.random((64, 64)) * 12 + 4 * (m != 0)) / 8).astype(np.float32) for m in masks]
    check(maps, masks)


def test_smoothed_maps():
    rng = np.random.default_rng(11)
    masks = _blob_masks(rng, 10, 96, 80)
    maps = [gaussian_filter((rng.random((96, 80)) + 0.8 * (m != 0)).astype(np.float32), 4.0, mode="reflect") for m in masks]
    check(maps, masks)


def test_negative_scores_and_negative_zero():
    rng = np.random.default_rng(12)
    masks = _blob_masks(rng, 6, 40, 40)
    maps = []
    for m in masks:
        a = (rng.integers(-3, 4, (40, 40)) / 2.0).astype(np.float32)
        a[rng.random((40, 40)) < 0.3] = -0.0
        a[rng.random((40, 40)) < 0.1] = np.float32(-3.0e38)
        maps.append(a)
    assert any(np.signbit(a[a == 0]).any() for a in maps)
    r = check(maps, masks)
    flipped = [np.where(a == 0, np.float32(0.0), a) for a in maps]
    assert check(flipped, masks) == r
    # every defect pixel at -0.0 or +0.0, every other pixel at 1.5 or -2.0: the zero run attains F1-max and is reported as +0.0
    zero = [np.where(m != 0, np.where(rng.random(m.shape) < 0.5, np.float32(-0.0), np.float32(0.0)),
                     np.where(rng.random(m.shape) < 0.5, np.float32(1.5), np.float32(-2.0))).astype(np.float32) for m in masks]
    r = check(zero, masks)
    assert r.f1_threshold == 0.0 and not np.signbit(r.f1_threshold) and r.f1_max < 1.0   # the ok pixels at 1.5 come first


def test_single_pixel_and_border_regions():
    rng = np.random.default_rng(13)
    masks = []
    for _ in range(5):
        m = np.zeros((32, 48), np.uint8)
        m[rng.integers(0, 32, 6), rng.integers(0, 48, 6)] = 1
        m[0, :5] = m[-1, -3:] = m[10:14, 0] = m[:2, -1] = 1
        masks.append(m)
    maps = [(rng.random((32, 48)) + 0.3 * (m != 0)).astype(np.float32) for m in masks]
    check(maps, masks)


def test_defect_free_and_all_defect_images():
    rng = np.random.default_rng(14)
    masks = [np.zeros((32, 32), np.uint8), np.ones((32, 32), np.uint8) * 255, np.zeros((32, 32), np.uint8)]
    masks[2][5:9, 20:30] = 1
    maps = [np.round(rng.random((32, 32)) * 50).astype(np.float32) / 10 for _ in masks]
    check(maps, masks)


def test_mixed_image_sizes_and_tensor_input():
    rng = np.random.default_rng(15)
    shapes = [(17, 33), (64, 40), (5, 7), (128, 96)]
    masks = [_blob_masks(rng, 1, h, w, 1.0)[0] for h, w in shapes]
    maps = [(np.round(rng.random(s) * 30) / 7).astype(np.float32) for s in shapes]
    check(maps, masks)
    same = [np.zeros((24, 24), np.uint8) for _ in range(4)]
    same[1][3:8, 3:8] = same[3][20:, 10:12] = 1
    stack = np.stack([rng.random((24, 24)).astype(np.float32) for _ in range(4)])
    d = torch.from_numpy(stack).cuda()
    assert metrics.pixel_ap(d, np.stack(same)) == metrics.pixel_ap(list(d.unbind(0)), same)
    assert abs(metrics.pixel_ap(d, same) - P.pixel_ap(list(stack), same)) <= 1e-9
    assert metrics.f1_max(d, np.stack(same)) == P.f1_max(list(stack), same)


def test_more_than_2_pow_24_pixels():
    rng = np.random.default_rng(16)
    n_img, h, w = 264, 256, 256
    masks = np.zeros((n_img, h, w), np.uint8)
    for i in range(0, n_img, 3):
        y, x = rng.integers(0, h - 40, 2)
        masks[i, y:y + rng.integers(4, 40), x:x + rng.integers(4, 40)] = 1
    maps = (np.round(rng.random((n_img, h, w)) * 4000) / 1000 + 0.5 * masks).astype(np.float32)
    assert maps.size > 2 ** 24
    acc = metrics.LocalisationAccumulator(1)
    for s in range(0, n_img, 64):
        acc.append([torch.from_numpy(maps[s:s + 64]).cuda()], masks[s:s + 64])
    check(list(maps), list(masks), acc)


def test_bitwise_deterministic_and_batch_independent():
    rng = np.random.default_rng(17)
    n = 128
    masks = _blob_masks(rng, n, 64, 64)
    ssim = np.stack([gaussian_filter(rng.random((64, 64)).astype(np.float32), 2.0) for _ in range(n)])
    se = (np.round(rng.random((n, 64, 64)) * 100) / 100).astype(np.float32)
    d_ssim, d_se = torch.from_numpy(ssim).cuda(), torch.from_numpy(se).cuda()
    results = []
    for bs in (8, 64, 128, 8):
        acc = metrics.LocalisationAccumulator(2)
        for s in range(0, n, bs):
            acc.append([d_ssim[s:s + bs], d_se[s:s + bs]], masks[s:s + bs])
        results.append(acc.results(0.3))
    assert all(r == results[0] for r in results), results
    for j, maps in enumerate((ssim, se)):
        assert abs(results[0][j].pixel_ap - P.pixel_ap(list(maps), masks)) <= 1e-9
        assert results[0][j].f1_threshold == P.f1_max(list(maps), masks)[1]


# ------------------------------------------------------------------------------------------------------------- evaluator
def test_evaluate_cli_pr_metrics_and_segmentation(tmp_path, capsys, monkeypatch):
    n = 16
    root = str(tmp_path / "mvtec_128")
    _, _, labels, masks = _dataset_with_masks(root, "carpet", 3, n, seed=78)
    sd = O.make_state_dict(O.DrctCfg(num_layers=1), seed=4)
    ckpt = str(tmp_path / "model_best.pt")
    torch.save(sd, ckpt)
    orig = evaluate.setup_opt_drct

    def one_rdg(*a, **k):
        opt = orig(*a, **k)
        opt.depths, opt.num_heads = (6,), (6,)
        return opt

    monkeypatch.setattr(evaluate, "setup_opt_drct", one_rdg)
    out_dir = str(tmp_path / "out")
    mask_dir = os.path.join(root, "masks")
    argv = ["--model-type", "drct", "--classe", "carpet", "--scale", "4", "--resolution", "128", "--data-root", root,
            "--checkpoint", ckpt, "--batch-size", "8", "--output-dir", out_dir, "--mask-dir", mask_dir]
    plain = evaluate.main(argv)
    plain_lines = capsys.readouterr().out.strip().splitlines()
    assert not os.path.isdir(os.path.join(out_dir, "segmentation"))
    res = evaluate.main(argv + ["--pr-metrics", "--au-pro", "--save-segmentation", "--save-maps"])
    lines = capsys.readouterr().out.strip().splitlines()

    new_keys = {f"{k}_{m}" for k in ("pixel_ap", "f1_max", "f1_threshold") for m in ("ssim", "se")}
    assert not any(l.startswith("Map PR ") for l in plain_lines) and not new_keys & set(plain)
    assert new_keys <= set(res)
    # PR line, PRO line, then the two lines of a plain --mask-dir run
    assert lines[-2:] == plain_lines[-2:]
    assert lines[-3].startswith("Map PRO - AU-PRO@0.3 1-SSIM: ")
    assert lines[-4] == (f"Map PR - pixel AP 1-SSIM: {res['pixel_ap_ssim']:.4f}, pixel AP SE: {res['pixel_ap_se']:.4f}, "
                         f"F1-max 1-SSIM: {res['f1_max_ssim']:.4f} (thr {res['f1_threshold_ssim']:g}), "
                         f"F1-max SE: {res['f1_max_se']:.4f} (thr {res['f1_threshold_se']:g})")
    for k in ("pixel_auroc_ssim", "pixel_auroc_se"):
        assert res[k] == plain[k]

    # evaluator order: good first, then bad; names sorted
    order = np.argsort(labels, kind="stable")
    mk = [masks[i] for i in order]
    split = lambda i: "good" if labels[i] == 0 else "bad"
    for kind in ("ssim", "se"):
        maps = [np.load(os.path.join(out_dir, "maps", split(i), f"{i:03d}_{kind}.npy")) for i in order]
        assert abs(res[f"pixel_ap_{kind}"] - P.pixel_ap(maps, mk)) <= 1e-9, kind
        assert (res[f"f1_max_{kind}"], res[f"f1_threshold_{kind}"]) == P.f1_max(maps, mk), kind
        pngs = [np.array(Image.open(os.path.join(out_dir, "segmentation", split(i), f"{i:03d}_{kind}.png"))) for i in order]
        assert all(p.dtype == np.uint8 and p.shape == (128, 128) and set(np.unique(p)) <= {0, 255} for p in pngs)
        pred = [p == 255 for p in pngs]
        assert all(np.array_equal(p, m >= np.float32(res[f"f1_threshold_{kind}"])) for p, m in zip(pred, maps))
        assert _f1_of(pred, mk) == res[f"f1_max_{kind}"], kind

    # --pr-metrics without --au-pro: the PR line right before the Map AUCs line
    res2 = evaluate.main(argv + ["--pr-metrics"])
    lines2 = capsys.readouterr().out.strip().splitlines()
    assert lines2[-2:] == plain_lines[-2:] and lines2[-3] == lines[-4]
    assert all(res2[k] == res[k] for k in new_keys)
