"""GPU tests of the defect regions (csrc/regions.cu adsr_label_regions / adsr_region_stats through ops.label_regions / region_stats and
metrics.defect_regions): labels equal scipy.ndimage.label (8-connectivity) exactly on random masks at every density, around the
percolation point, on serpentines and spirals that cross every tile border, on checkerboards, stripes, full and empty images, at odd
sizes and in batches; every table field equals oracle/region_oracle.py exactly, on the threshold and the mask path and for several
minimum areas; the region metrics equal the oracle; results are bitwise deterministic and batch independent; then
`--calibration-dir --defect-regions --min-region-area --mask-dir` end to end."""
import csv
import importlib
import math
import os
import shutil

import numpy as np
import pytest
import torch

from gpu_common import PKG
from oracle import drct_oracle as O
from oracle import region_oracle as R
from test_gpu_anomaly_maps import _dataset_with_masks
from test_gpu_pr_metrics import _blob_masks

pytestmark = pytest.mark.gpu

ops = importlib.import_module(PKG + ".ops")
metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")

SIZES = (1, 2, 31, 33, 127, 128, 129, 256, 257)


def gpu_label_masks(masks, min_area=1):
    """ops.label_regions on the mask path -> (labels [B, H, W], counts [B]) on the host."""
    m = torch.from_numpy(np.ascontiguousarray(np.asarray(masks) != 0).astype(np.uint8)).cuda()
    b, h, w = m.shape
    ws = torch.empty(ops.regions_workspace_bytes(b, h, w), dtype=torch.uint8, device="cuda")
    labels = torch.empty(b, h, w, dtype=torch.int32, device="cuda")
    counts = torch.empty(b, dtype=torch.int32, device="cuda")
    ops.label_regions(None, 0.0, m, min_area, ws, labels, counts)
    assert int(ws[:4].view(torch.int32).item()) == 0
    return labels.cpu().numpy(), counts.cpu().numpy(), (m, ws, labels, counts)


def check_mask_labels(masks, min_area=1):
    got, counts, _ = gpu_label_masks(masks, min_area)
    for i, m in enumerate(masks):
        want, n = R.label_image(np.asarray(m) != 0, min_area)
        assert counts[i] == n, (i, counts[i], n)
        assert np.array_equal(got[i], want), (i, np.argwhere(got[i] != want)[:5])
    return got


def rows_equal(table, rows):
    assert len(table) == len(rows), (len(table), len(rows))
    for name in table.dtype.names:
        got = table[name]
        want = np.array([r[name] for r in rows], dtype=table.dtype[name])
        if name == "peak":
            assert np.array_equal(got, want, equal_nan=True), (got[got != want][:5], want[got != want][:5])
            assert not np.any(np.signbit(got) & (got == 0))
        else:
            assert np.array_equal(got, want), (name, np.flatnonzero(got != want)[:5])


def check_regions(maps, t, min_area=1, masks=None):
    d = metrics.defect_regions(torch.from_numpy(np.ascontiguousarray(maps)).cuda(), t, min_area, masks)
    labs, rows, n, gt_n, gt_det = R.defect_regions(list(maps), t, min_area, masks)
    assert np.array_equal(d.labels.cpu().numpy(), np.stack(labs))
    assert np.array_equal(d.n_regions, n)
    rows_equal(d.regions, rows)
    if masks is not None:
        assert np.array_equal(d.gt_regions, gt_n) and np.array_equal(d.gt_detected, gt_det)
    centroid = d.regions["sum_y"] / d.regions["area"]
    assert np.array_equal(centroid, np.array([r["sum_y"] / r["area"] for r in rows]))
    return d


# ------------------------------------------------------------------------------------------------------------- labels
@pytest.mark.parametrize("density", [0.05, 0.2, 0.40, 0.42, 0.44, 0.45, 0.47, 0.6, 0.8, 0.95])
def test_random_masks_all_densities(density):
    rng = np.random.default_rng(int(density * 1000))
    check_mask_labels(rng.random((8, 200, 300)) < density)
    check_mask_labels(rng.random((4, 129, 257)) < density, min_area=3)


def _serpentine(h, w, period=4):
    m = np.zeros((h, w), bool)
    m[::period] = True                                        # rows joined alternately at the right and the left end
    for k, y in enumerate(range(0, h - period, period)):
        m[y:y + period, w - 1 if k % 2 == 0 else 0] = True
    return m


def _spiral(n):
    m = np.zeros((n, n), bool)
    y0, x0, y1, x1 = 0, 0, n - 1, n - 1
    while y0 <= y1 and x0 <= x1:
        m[y0, x0:x1 + 1] = True
        m[y0:y1 + 1, x1] = True
        if y1 - y0 >= 2:
            m[y1, x0:x1 + 1] = True
        if x1 - x0 >= 2 and y1 - y0 >= 4:
            m[y0 + 2:y1 + 1, x0] = True
        y0, x0, y1, x1 = y0 + 2, x0 + 2, y1 - 2, x1 - 2
    return m


def test_serpentines_and_spirals():
    shapes = [_serpentine(256, 257), _serpentine(257, 256, 2), _serpentine(129, 500, 3), _serpentine(300, 33, 2)]
    for s in shapes:
        lab = check_mask_labels([s])
        assert lab.max() == 1                                 # one component winding over every tile border
    diag = np.eye(300, dtype=bool) | np.eye(300, k=1, dtype=bool)[:, ::-1]
    for m in (_spiral(255), _spiral(256), _spiral(301), diag, np.eye(257, dtype=bool)):
        check_mask_labels([m])
    # diagonal staircases: 8-connected only through corners, across tile borders
    stair = np.zeros((200, 200), bool)
    for k in range(0, 200, 7):
        idx = np.arange(200 - k)
        stair[idx, idx + k] = True
    check_mask_labels([stair, stair[::-1], stair[:, ::-1], stair.T])


def test_checkerboards_stripes_full_and_empty():
    yy, xx = np.mgrid[:130, :260]
    cases = [(yy + xx) % 2 == 0, (yy + xx) % 2 == 1, (yy // 2 + xx // 2) % 2 == 0, yy % 2 == 0, xx % 2 == 0, yy % 3 == 0,
             np.ones((130, 260), bool), np.zeros((130, 260), bool), (yy % 32 == 31) | (xx % 32 == 0)]
    lab = check_mask_labels(cases)
    assert lab[0].max() == 1 and lab[1].max() == 1            # a checkerboard is one component under 8-connectivity
    assert lab[6].max() == 1 and lab[7].max() == 0


def test_every_size_pair():
    rng = np.random.default_rng(5)
    for h in SIZES:
        for w in SIZES:
            masks = [rng.random((h, w)) < d for d in (0.3, 0.45, 0.7)]
            check_mask_labels(masks)
            maps = rng.random((3, h, w)).astype(np.float32)
            check_regions(maps, 0.55, 1)


def test_batch_of_64_distinct_images():
    rng = np.random.default_rng(6)
    masks = [rng.random((97, 143)) < rng.uniform(0.05, 0.95) for _ in range(64)]
    masks[3][:] = False
    masks[7][:] = True
    check_mask_labels(masks)
    check_mask_labels(masks, min_area=5)


def test_large_batch_near_percolation():
    rng = np.random.default_rng(7)
    masks = rng.random((256, 256, 256)) < 0.43
    check_mask_labels(masks)


# ------------------------------------------------------------------------------------------------------------- tables
def test_threshold_path_ties_nan_and_signed_zeros():
    rng = np.random.default_rng(8)
    maps = (np.round(rng.random((6, 70, 90)) * 8) / 8).astype(np.float32)          # heavy ties, also at the threshold
    maps[0, rng.random((70, 90)) < 0.05] = np.nan
    maps[1] = np.where(rng.random((70, 90)) < 0.5, np.float32(-0.0), np.float32(0.0))
    maps[2] = -maps[2]
    for t in (0.5, 0.625, 0.0, -0.0, -0.5, float(np.nextafter(np.float32(0.5), np.float32(1))), 0.5 - 1e-12, 2.0):
        for min_area in (1, 2, 7):
            d = check_regions(maps, t, min_area)
            if t == 2.0:
                assert d.regions.size == 0 and not d.n_regions.any()
    z = check_regions(maps[1:2], 0.0)                         # -0.0 >= 0.0: every pixel, one region, peak +0.0 at the first pixel
    assert z.n_regions.tolist() == [1] and z.regions["peak"][0] == 0 and (z.regions["peak_y"][0], z.regions["peak_x"][0]) == (0, 0)
    nan = np.full((1, 5, 5), np.nan, np.float32)
    assert check_regions(nan, -1e30).regions.size == 0        # NaN is never foreground


def test_threshold_path_with_masks_and_min_areas():
    rng = np.random.default_rng(9)
    masks = _blob_masks(rng, 12, 96, 80)
    from scipy.ndimage import gaussian_filter
    maps = np.stack([gaussian_filter((rng.random((96, 80)) + 0.9 * (m != 0)).astype(np.float32), 1.5) for m in masks])
    for t in (0.55, 0.6, 0.7):
        for min_area in (1, 4, 30):
            d = check_regions(maps, t, min_area, masks)
            on_dev = metrics.defect_regions(torch.from_numpy(maps).cuda(), t, min_area, torch.from_numpy(np.stack(masks)).cuda())
            assert torch.equal(on_dev.labels, d.labels) and on_dev.regions.tobytes() == d.regions.tobytes()   # device masks: the same
            assert np.array_equal(on_dev.gt_regions, d.gt_regions) and np.array_equal(on_dev.gt_detected, d.gt_detected)


def test_mask_path_table():
    rng = np.random.default_rng(10)
    masks = np.stack([rng.random((65, 129)) < d for d in (0.1, 0.4, 0.6)])
    for min_area in (1, 3, 10):
        got, counts, (m, ws, labels, cnt) = gpu_label_masks(masks, min_area)
        off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        table = torch.empty(int(off[-1]), 9, dtype=torch.int64, device="cuda")
        ops.region_stats(labels, None, None, torch.from_numpy(off).cuda(), None, ws, table)
        tab = table.cpu().numpy()
        assert int(ws[:4].view(torch.int32).item()) == 0
        rows = []
        for i in range(len(masks)):
            lab, n = R.label_image(masks[i], min_area)
            rows += R.region_rows(lab, n, i)
        want = np.array([[r["area"], r["y0"], r["x0"], r["y1"] - 1, r["x1"] - 1, r["sum_y"], r["sum_x"], 0, 0] for r in rows],
                        dtype=np.int64).reshape(-1, 9)
        assert np.array_equal(tab, want)


def test_region_metrics_and_image_decision():
    rng = np.random.default_rng(11)
    masks = _blob_masks(rng, 20, 64, 64, 0.6)
    from scipy.ndimage import gaussian_filter
    maps = np.stack([gaussian_filter((rng.random((64, 64)) + 0.7 * (m != 0)).astype(np.float32), 2.0) for m in masks])
    t_px = float(np.quantile(maps[[i for i, m in enumerate(masks) if not m.any()]].astype(np.float64), 0.99, method="inverted_cdf"))
    thr = evaluate.above(t_px)
    for min_area in (1, 5):
        d = check_regions(maps, thr, min_area, masks)
        _, rows, n, gt_n, gt_det = R.defect_regions(list(maps), thr, min_area, masks)
        want = R.region_metrics(rows, n, gt_n, gt_det, len(maps))
        n_false = int((d.regions["gt_pixels"] == 0).sum())
        got = (d.gt_detected.sum() / d.gt_regions.sum(), (d.n_regions.sum() - n_false) / d.n_regions.sum(), n_false / len(maps))
        assert got == want, (got, want)
        if min_area == 1:                                     # the region decision is the map max against the same threshold
            assert np.array_equal(d.n_regions > 0, maps.reshape(len(maps), -1).max(1).astype(np.float64) >= thr)


def test_deterministic_and_batch_independent():
    rng = np.random.default_rng(12)
    masks = _blob_masks(rng, 24, 150, 170)
    maps = (rng.random((24, 150, 170)) * 0.8 + 0.5 * (np.stack(masks) != 0)).astype(np.float32)
    dm = torch.from_numpy(maps).cuda()
    a = metrics.defect_regions(dm, 0.6, 3, masks)
    b = metrics.defect_regions(dm, 0.6, 3, masks)
    assert torch.equal(a.labels, b.labels) and a.regions.tobytes() == b.regions.tobytes()
    for i in (0, 5, 23):
        one = metrics.defect_regions(dm[i:i + 1], 0.6, 3, masks[i:i + 1])
        assert torch.equal(one.labels[0], a.labels[i])
        rows = a.regions[a.regions["image"] == i].copy()
        rows["image"] = 0
        assert one.regions.tobytes() == rows.tobytes()
        assert (one.gt_regions[0], one.gt_detected[0]) == (a.gt_regions[i], a.gt_detected[i])


def test_rejections():
    x = torch.zeros(2, 8, 8, device="cuda")
    with pytest.raises(ValueError, match="NaN"):
        metrics.defect_regions(x, float("nan"))
    for bad in (0, -1, 1.5):
        with pytest.raises(ValueError, match="min_area"):
            metrics.defect_regions(x, 0.5, bad)
    with pytest.raises(ValueError, match="float32"):
        metrics.defect_regions(x.double(), 0.5)
    with pytest.raises(ValueError, match="masks"):
        metrics.defect_regions(x, 0.5, 1, np.zeros((2, 8, 7)))
    ws = torch.empty(ops.regions_workspace_bytes(2, 8, 8), dtype=torch.uint8, device="cuda")
    lab, cnt = torch.empty(2, 8, 8, dtype=torch.int32, device="cuda"), torch.empty(2, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="exactly one"):
        ops.label_regions(x, 0.5, x.to(torch.uint8), 1, ws, lab, cnt)
    with pytest.raises(RuntimeError, match="unsupported shape"):    # short workspace, checked by the C entry point
        ops.label_regions(x, 0.5, None, 1, ws[:64], lab, cnt)
    with pytest.raises(RuntimeError, match="unsupported shape"):
        ops.label_regions(x, float("nan"), None, 1, ws, lab, cnt)
    with pytest.raises(ValueError, match="unsupported batch shape"):
        ops.regions_workspace_bytes(1, 1 << 16, 1 << 15)
    with pytest.raises(ValueError, match="unsupported batch shape"):
        ops.regions_workspace_bytes(0, 8, 8)


# ------------------------------------------------------------------------------------------------------------- evaluator
def test_evaluate_cli_defect_regions(tmp_path, capsys, monkeypatch):
    n, q, min_area = 16, 0.99, 4
    root = str(tmp_path / "mvtec_128")
    _, _, labels, masks = _dataset_with_masks(root, "carpet", 3, n, seed=88)
    other = str(tmp_path / "other")
    _dataset_with_masks(other, "carpet", 3, 12, seed=89)
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
    out_dir = str(tmp_path / "out")
    mask_dir = os.path.join(root, "masks")
    argv = ["--model-type", "drct", "--classe", "carpet", "--scale", "4", "--resolution", "128", "--data-root", root,
            "--checkpoint", ckpt, "--batch-size", "8", "--output-dir", out_dir, "--mask-dir", mask_dir, "--calibration-dir", cal_dir,
            "--calibration-quantile", str(q), "--save-maps"]
    plain = evaluate.main(argv)
    plain_lines = capsys.readouterr().out.strip().splitlines()
    assert not os.path.exists(os.path.join(out_dir, "defects.csv"))
    res = evaluate.main(argv + ["--defect-regions", "--min-region-area", str(min_area)])
    lines = capsys.readouterr().out.strip().splitlines()

    reg_at = [i for i, l in enumerate(lines) if l.startswith("Map REG - ")]
    assert len(reg_at) == 1 and lines[reg_at[0] - 1].startswith("Map CAL - ")
    assert lines[:reg_at[0]] + lines[reg_at[0] + 1:] == plain_lines          # every other line as without the new flags
    reg_keys = {f"region_{k}_{m}" for k in ("count_good", "count_bad", "image_tpr", "image_fpr", "recall", "precision",
                                            "false_per_image") for m in ("ssim", "se")}
    assert {k for k in res if k.startswith("region_")} == reg_keys and not any(k.startswith("region_") for k in plain)
    same = lambda u, v: np.array_equal(u, v) if isinstance(v, np.ndarray) else (u == v or (u != u and v != v))
    assert all(same(res[k], plain[k]) for k in plain)

    order = np.argsort(labels, kind="stable")                  # evaluator order: good first, then bad
    split = lambda i: "good" if labels[i] == 0 else "bad"
    want_rows, parts = [], []
    y = labels[order]
    per_kind = {}
    for kind, label in (("ssim", "1-SSIM"), ("se", "SE")):
        thr = evaluate.above(res[f"calib_pixel_threshold_{kind}"])
        maps = [np.load(os.path.join(out_dir, "maps", split(i), f"{i:03d}_{kind}.npy")) for i in order]
        mk = [masks[i] != 0 for i in order]
        labs, rows, n_reg, gt_n, gt_det = R.defect_regions(maps, thr, min_area, mk)
        per_kind[kind] = rows
        flagged = n_reg > 0
        tpr, fpr = float(flagged[y == 1].mean()), float(flagged[y == 0].mean())
        good, bad = int(n_reg[y == 0].sum()), int(n_reg[y == 1].sum())
        recall, precision, fpi = R.region_metrics(rows, n_reg, gt_n, gt_det, n)
        assert (res[f"region_count_good_{kind}"], res[f"region_count_bad_{kind}"]) == (good, bad)
        assert (res[f"region_image_tpr_{kind}"], res[f"region_image_fpr_{kind}"]) == (tpr, fpr)
        got = (res[f"region_recall_{kind}"], res[f"region_precision_{kind}"], res[f"region_false_per_image_{kind}"])
        assert all((math.isnan(a) and math.isnan(b)) or a == b for a, b in zip(got, (recall, precision, fpi))), (kind, got)
        parts.append(f"{label} regions good {good}, bad {bad}, image TPR {tpr:.4f}, FPR {fpr:.4f}, region recall {recall:.4f}, "
                     f"precision {precision:.4f}, false regions per image {fpi:.4f}")
    assert lines[reg_at[0]] == f"Map REG - min area {min_area}: " + "; ".join(parts)
    for pos, i in enumerate(order):
        for kind in ("ssim", "se"):
            for r in per_kind[kind]:
                if r["image"] == pos:
                    want_rows.append([split(i), f"{i:03d}", kind, str(r["label"]), str(r["area"]), str(r["y0"]), str(r["x0"]),
                                      str(r["y1"]), str(r["x1"]), repr(r["sum_y"] / r["area"]), repr(r["sum_x"] / r["area"]),
                                      repr(r["peak"]), str(r["peak_y"]), str(r["peak_x"]), str(r["gt_pixels"])])
    with open(os.path.join(out_dir, "defects.csv"), newline="") as f:
        got_rows = list(csv.reader(f))
    assert got_rows[0] == ["split", "stem", "map", "region", "area", "y0", "x0", "y1", "x1", "centroid_y", "centroid_x", "peak", "peak_y",
                           "peak_x", "gt_pixels"]
    assert got_rows[1:] == want_rows
    assert len(want_rows) > 0

    # without masks: counts and image decisions only, the same values; min area 1 decides like the map max
    no_masks = [a for a in argv if a not in ("--mask-dir", mask_dir)]
    res2 = evaluate.main(no_masks + ["--defect-regions"])
    lines2 = capsys.readouterr().out.strip().splitlines()
    reg2 = [l for l in lines2 if l.startswith("Map REG - min area 1: ")]
    assert len(reg2) == 1 and "recall" not in reg2[0]
    for j, kind in enumerate(("ssim", "se")):
        flagged = res2["map_max"][:, j] >= evaluate.above(res2[f"calib_pixel_threshold_{kind}"])
        yy = np.asarray([0] * (n // 2) + [1] * (n - n // 2))
        assert res2[f"region_image_tpr_{kind}"] == float(flagged[yy == 1].mean())
        assert res2[f"region_image_fpr_{kind}"] == float(flagged[yy == 0].mean())
