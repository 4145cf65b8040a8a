"""CPU tests of the defect-region reference (oracle/region_oracle.py) on hand-made images -- 8-connectivity, renumbering after the
minimum-area filter, half-open boxes, the first-pixel peak tie rule, NaN and signed zeros at the threshold -- of the host table layout
of metrics.defect_regions, and of the `--defect-regions` / `--min-region-area` options."""
import importlib

import numpy as np
import pytest
import torch

from oracle import region_oracle as R

PKG = "anomaly-detection-super-resolution_b200"
metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")


def test_checkerboard_is_one_component():
    yy, xx = np.mgrid[:9, :12]
    lab, n = R.label_image((yy + xx) % 2 == 0)
    assert n == 1 and set(np.unique(lab)) == {0, 1}


def test_two_diagonal_pixels_form_one_region():
    fg = np.zeros((4, 4), bool)
    fg[1, 2] = fg[2, 1] = True                                # anti-diagonal: NE / SW neighbours
    lab, n = R.label_image(fg)
    assert n == 1 and lab[1, 2] == lab[2, 1] == 1
    rows = R.region_rows(lab, n)
    assert (rows[0]["y0"], rows[0]["x0"], rows[0]["y1"], rows[0]["x1"], rows[0]["area"]) == (1, 1, 3, 3, 2)


def test_min_area_drops_and_renumbers_in_raster_order():
    fg = np.zeros((6, 8), bool)
    fg[0, 6] = True                                           # first pixel in raster order, area 1
    fg[1, 0:3] = True                                         # area 3
    fg[4:6, 4:7] = True                                       # area 6
    lab, n = R.label_image(fg)
    assert n == 3 and lab[0, 6] == 1 and lab[1, 0] == 2 and lab[4, 4] == 3
    lab2, n2 = R.label_image(fg, min_area=2)
    assert n2 == 2 and lab2[0, 6] == 0 and lab2[1, 0] == 1 and lab2[4, 4] == 2
    lab3, n3 = R.label_image(fg, min_area=4)
    assert n3 == 1 and lab3[4, 4] == 1 and lab3.sum() == 6
    assert R.label_image(fg, min_area=7)[1] == 0


def test_half_open_boxes_and_integer_sums():
    fg = np.zeros((5, 7), bool)
    fg[1:4, 2] = True
    fg[3, 2:6] = True
    lab, n = R.label_image(fg)
    r, = R.region_rows(lab, n)
    assert (r["y0"], r["x0"], r["y1"], r["x1"]) == (1, 2, 4, 6)
    ys, xs = np.nonzero(fg)
    assert (r["area"], r["sum_y"], r["sum_x"]) == (len(ys), int(ys.sum()), int(xs.sum()))
    assert r["sum_y"] / r["area"] == ys.mean() and np.isnan(r["peak"]) and (r["peak_y"], r["peak_x"]) == (-1, -1)


def test_peak_tie_goes_to_the_first_raster_pixel():
    m = np.zeros((4, 5), np.float32)
    m[1, 3] = m[2, 1] = m[3, 4] = 0.75
    m[1:4, 1:5] = np.maximum(m[1:4, 1:5], 0.5)
    _, rows, n, _, _ = R.defect_regions([m], 0.5)
    assert n.tolist() == [1] and (rows[0]["peak"], rows[0]["peak_y"], rows[0]["peak_x"]) == (0.75, 1, 3)


def test_nan_is_never_foreground():
    m = np.full((3, 3), np.nan, np.float32)
    m[0, 0] = 1.0
    assert R.foreground(m, -np.inf).sum() == 1
    labs, rows, n, _, _ = R.defect_regions([m], -1e30)
    assert n.tolist() == [1] and rows[0]["area"] == 1


def test_negative_zero_is_at_least_zero():
    m = np.array([[-0.0, 0.0], [-1e-45, 0.0]], np.float32)
    assert R.foreground(m, 0.0).tolist() == [[True, True], [False, True]]
    _, rows, _, _, _ = R.defect_regions([m], 0.0)
    assert rows[0]["peak"] == 0.0 and not np.signbit(rows[0]["peak"]) and (rows[0]["peak_y"], rows[0]["peak_x"]) == (0, 0)
    assert R.foreground(m, float(np.nextafter(np.float32(0), np.float32(1)))).sum() == 0   # above(0.0): strictly positive


def test_ground_truth_regions_and_metrics():
    m = np.zeros((6, 6), np.float32)
    m[0, 0:2] = 1.0                                           # touches ground-truth region A
    m[4, 4] = 1.0                                             # false region
    gt = np.zeros((6, 6), bool)
    gt[0:2, 1] = True                                         # region A
    gt[3, 0] = True                                           # region B, missed
    _, rows, n, gt_n, gt_det = R.defect_regions([m], 0.5, 1, [gt])
    assert [r["gt_pixels"] for r in rows] == [1, 0] and gt_n.tolist() == [2] and gt_det.tolist() == [1]
    assert R.region_metrics(rows, n, gt_n, gt_det, 2) == (0.5, 0.5, 0.5)
    rec, prec, fpi = R.region_metrics([], [0], [0], [0], 1)
    assert np.isnan(rec) and np.isnan(prec) and fpi == 0.0


def test_table_layout():
    assert metrics.region_dtype(False).names == R.COLUMNS
    assert metrics.region_dtype(True).names == R.COLUMNS + ("gt_pixels",)
    assert metrics.region_dtype(True)["peak"] == np.float32 and metrics.region_dtype(True)["area"] == np.int64
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.defect_regions(torch.zeros(1, 4, 4), 0.5)


def test_cli_defect_region_flags():
    a = evaluate.parse_args([])
    assert a.defect_regions is False and a.min_region_area is None
    a = evaluate.parse_args(["--calibration-dir", "cal", "--defect-regions", "--min-region-area", "4"])
    assert a.defect_regions and a.min_region_area == 4
    assert evaluate.parse_args(["--calibration-dir", "cal", "--defect-regions"]).min_region_area is None
    for bad in (["--defect-regions"], ["--calibration-dir", "cal", "--min-region-area", "3"], ["--min-region-area", "2"],
                ["--calibration-dir", "cal", "--defect-regions", "--min-region-area", "0"],
                ["--calibration-dir", "cal", "--defect-regions", "--min-region-area", "1.5"]):
        with pytest.raises(SystemExit):
            evaluate.parse_args(bad)


def test_evaluate_on_test_checks_region_flags_first():
    with pytest.raises(ValueError, match="calibration_dir"):
        evaluate.evaluate_on_test(None, None, "", False, defect_regions=True)
    with pytest.raises(ValueError, match="min_region_area"):
        evaluate.evaluate_on_test(None, None, "", False, calibration_dir="cal", defect_regions=True, min_region_area=0)
