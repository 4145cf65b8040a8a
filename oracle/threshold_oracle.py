"""Reference (numpy / scipy) for the calibrated-threshold side of csrc/localisation.cu: the exact score quantile
(np.quantile(..., method="inverted_cdf"), an actual score) and the pixel counts and PRO of the prediction `score >= threshold`.

The quantile is taken over the scores converted to float64 (exact), so that numpy forms the rank from q n in float64: given fp32 input
numpy forms it in fp32, which misranks (n = 2880, q = 0.3 gives rank 865 instead of 864) and fails beyond 2^24 values.

Defect regions are the 8-connected components of the masks (scipy.ndimage.label, as for AU-PRO); PRO@t is the mean over the regions
of the share of the region's pixels whose score is >= t.  The fp32 scores are compared with the exact double threshold."""
from __future__ import annotations

import numpy as np

from .localisation_oracle import regions


def _scores(maps):
    s = np.concatenate([np.asarray(a, dtype=np.float32).ravel() for a in maps])
    if np.isnan(s).any():
        raise ValueError("NaN in a map")
    return s


def quantile(maps, q):
    """np.quantile of every pixel of the maps (as float64), method="inverted_cdf": an fp32 score, -0.0 reported as +0.0."""
    return float(np.quantile(_scores(maps).astype(np.float64), q, method="inverted_cdf") + 0.0)


def counts(maps, masks, threshold):
    """(TP, FP, FN, TN, PRO@threshold) of the prediction `score >= threshold`; PRO is NaN without a defect region."""
    s = _scores(maps).astype(np.float64)
    reg, sizes = regions(masks)
    r = np.concatenate([x.ravel() for x in reg])
    if len(r) != len(s):
        raise ValueError("every map needs a mask of its own shape")
    pred, defect = s >= float(threshold), r >= 0
    tp, fp = int((pred & defect).sum()), int((pred & ~defect).sum())
    fn, tn = int((~pred & defect).sum()), int((~pred & ~defect).sum())
    if len(sizes) == 0:
        return tp, fp, fn, tn, float("nan")
    hit = np.bincount(r[pred & defect], minlength=len(sizes))
    return tp, fp, fn, tn, float(np.mean(hit / sizes))
