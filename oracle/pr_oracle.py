"""Reference (numpy / sklearn) for the precision-recall metrics of csrc/localisation.cu over a whole test set: pixel AP
(sklearn.metrics.average_precision_score over every pixel) and F1-max with its threshold (numpy over the runs of equal scores).

Definition: the pixels of all images are sorted by score, descending (-0.0 = +0.0); a run is a maximal set of equal scores.  At the
end of run k, d_k defect and o_k defect-free pixels have been seen; N_def = all defect pixels.  F1_k = 2 d_k / (d_k + o_k + N_def) is
the F1 of the mask `score >= score of run k`; F1-max is the largest, a tie going to the earlier run (the higher threshold)."""
from __future__ import annotations

import numpy as np


def _flat(maps, masks):
    s = np.concatenate([np.asarray(a, dtype=np.float32).ravel() for a in maps]) + np.float32(0.0)   # -0.0 -> +0.0
    if np.isnan(s).any():
        raise ValueError("NaN in a map")
    y = np.concatenate([(np.asarray(m) != 0).ravel() for m in masks])
    if not y.any():
        raise ValueError("need at least one defect pixel")
    return s, y


def pixel_ap(maps, masks):
    from sklearn.metrics import average_precision_score

    s, y = _flat(maps, masks)
    return float(average_precision_score(y, s.astype(np.float64)))


def run_ends(maps, masks):
    """(fp32 score, d_k, o_k) at the end of every run, in descending score order, and N_def."""
    s, y = _flat(maps, masks)
    order = np.argsort(-s, kind="stable")
    s, y = s[order], y[order]
    last = np.append(s[1:] != s[:-1], True)                 # last pixel of each run of equal scores
    return s[last], np.cumsum(y, dtype=np.int64)[last], np.cumsum(~y, dtype=np.int64)[last], int(y.sum())


def f1_max(maps, masks):
    """(F1-max, threshold): the max over the runs taken exactly (integer cross products), the threshold is that run's fp32 score."""
    score, d, o, n_def = run_ends(maps, masks)
    den = d + o + n_def
    f = d / den
    cand = np.flatnonzero(f >= f.max() * (1.0 - 1e-12))     # every exact maximum is among these (the quotients are within 2^-53)
    best = int(cand[0])
    for k in cand[1:]:                                      # ascending runs: only a strictly larger fraction replaces an earlier run
        if int(d[k]) * int(den[best]) > int(d[best]) * int(den[k]):
            best = int(k)
    return 2 * int(d[best]) / int(den[best]), float(score[best])
