"""Reference (numpy / scipy) for the defect regions of csrc/regions.cu: 8-connected components of a thresholded map or a mask, a
minimum-area filter, per-region statistics and the region-level detection metrics.

Foreground is `map >= t` with the fp32 map compared against the exact double t (the rule of threshold_oracle.counts); a NaN score is
never foreground.  Regions are scipy.ndimage.label(fg, structure=ones((3, 3))); with min_area > 1 the components of fewer pixels are
removed and the kept foreground is labelled again, so the kept regions are numbered 1..n in raster order of their first pixel.  Boxes
come from scipy.ndimage.find_objects (half-open), sums from integer bincounts, the peak is the first raster argmax of the region's
scores (-0.0 reported as +0.0)."""
from __future__ import annotations

import numpy as np
from scipy.ndimage import find_objects, label

STRUCTURE = np.ones((3, 3), dtype=int)
COLUMNS = ("image", "label", "area", "y0", "x0", "y1", "x1", "sum_y", "sum_x", "peak", "peak_y", "peak_x")


def foreground(score_map, threshold):
    """bool `map >= threshold`: fp32 scores against the exact double threshold (float32 -> float64 is exact); NaN is never foreground."""
    return np.asarray(score_map, dtype=np.float32).astype(np.float64) >= float(threshold)


def label_image(fg, min_area=1):
    """(int32 labels, n) of one bool image: 8-connected components with at least min_area pixels, numbered in raster order."""
    lab, n = label(np.asarray(fg, dtype=bool), structure=STRUCTURE)
    if min_area > 1 and n:
        keep = np.bincount(lab.ravel(), minlength=n + 1) >= min_area
        keep[0] = False
        lab, n = label(keep[lab], structure=STRUCTURE)
    return lab.astype(np.int32), int(n)


def region_rows(lab, n, image=0, score_map=None, gt_mask=None):
    """The rows of one labelled image as a list of dicts (COLUMNS, plus gt_pixels with gt_mask); without scores the peak is NaN at
    (-1, -1)."""
    h, w = lab.shape
    flat = lab.ravel().astype(np.int64)
    yy, xx = np.divmod(np.arange(h * w, dtype=np.int64), w)
    area = np.bincount(flat, minlength=n + 1)
    sum_y = np.zeros(n + 1, np.int64)
    sum_x = np.zeros(n + 1, np.int64)
    np.add.at(sum_y, flat, yy)
    np.add.at(sum_x, flat, xx)
    first = {}
    if score_map is not None and n:
        s = np.asarray(score_map, dtype=np.float32).ravel()
        fg = np.flatnonzero(flat > 0)
        order = fg[np.lexsort((fg, -s[fg].astype(np.float64), flat[fg]))]   # by label, score descending, raster index
        lab_sorted = flat[order]
        starts = np.flatnonzero(np.r_[True, lab_sorted[1:] != lab_sorted[:-1]])
        first = {int(lab_sorted[k]): int(order[k]) for k in starts}
    gt = None if gt_mask is None else np.bincount(flat[np.asarray(gt_mask).ravel() != 0], minlength=n + 1)
    rows = []
    for l, sl in enumerate(find_objects(lab, max_label=n), start=1):
        r = dict(image=image, label=l, area=int(area[l]), y0=sl[0].start, x0=sl[1].start, y1=sl[0].stop, x1=sl[1].stop,
                 sum_y=int(sum_y[l]), sum_x=int(sum_x[l]), peak=float("nan"), peak_y=-1, peak_x=-1)
        if score_map is not None:
            i = first[l]
            r.update(peak=float(s[i]) + 0.0, peak_y=i // w, peak_x=i % w)
        if gt is not None:
            r["gt_pixels"] = int(gt[l])
        rows.append(r)
    return rows


def defect_regions(maps, threshold, min_area=1, masks=None):
    """(labels per image, rows, n_regions [B], gt_regions [B] or None, gt_detected [B] or None) of a batch of maps, as
    metrics.defect_regions defines them."""
    labels, rows, n_regions, gt_regions, gt_detected = [], [], [], [], []
    for i, m in enumerate(maps):
        lab, n = label_image(foreground(m, threshold), min_area)
        gt = None if masks is None else np.asarray(masks[i]) != 0
        labels.append(lab)
        rows += region_rows(lab, n, i, m, gt)
        n_regions.append(n)
        if gt is not None:
            gl, ng = label(gt, structure=STRUCTURE)
            gt_regions.append(ng)
            gt_detected.append(len(np.unique(gl[(lab > 0) & (gl > 0)])))
    as_arr = lambda v: np.asarray(v, dtype=np.int64)
    return labels, rows, as_arr(n_regions), (as_arr(gt_regions) if masks is not None else None), \
        (as_arr(gt_detected) if masks is not None else None)


def region_metrics(rows, n_regions, gt_regions, gt_detected, n_images):
    """Set-level numbers: (region recall = detected / ground-truth regions, region precision = true / predicted regions, false regions
    per image); recall NaN without ground-truth regions, precision NaN without predictions.  A region is true when gt_pixels > 0."""
    n_pred = int(np.sum(n_regions))
    n_true = sum(1 for r in rows if r["gt_pixels"] > 0)
    n_gt = int(np.sum(gt_regions))
    recall = int(np.sum(gt_detected)) / n_gt if n_gt else float("nan")
    precision = n_true / n_pred if n_pred else float("nan")
    return recall, precision, (n_pred - n_true) / n_images
