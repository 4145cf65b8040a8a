"""Reference (numpy / scipy) for the localisation metrics of csrc/localisation.cu: the (FPR, PRO) curve with one point per distinct
score, AU-PRO@alpha by the trapezoid rule with the crossing segment cut by linear interpolation, and pixel AUROC (sklearn).

Definition: every 8-connected component of a mask is one defect region r (R regions over all images); a defect pixel of region r
weighs 1 / (R |r|), each of the N_ok defect-free pixels 1 / N_ok.  Pixels of all images are sorted by score, descending (-0.0 = +0.0);
at every distinct score the cumulative defect-free weight is the FPR and the cumulative defect weight the PRO.  The curve is (0, 0)
followed by these points; tied pixels form one point (as the MVTec AD evaluation script treats ties)."""
from __future__ import annotations

import numpy as np
from scipy.ndimage import label


def regions(masks):
    """Per image: int region index per pixel (-1 = defect-free, numbered across the images) and the int64 region sizes."""
    out, sizes, base = [], [], 0
    for m in masks:
        lab, n = label(np.asarray(m) != 0, structure=np.ones((3, 3), dtype=int))
        out.append(np.where(lab > 0, lab + (base - 1), -1))
        sizes.append(np.bincount(lab.ravel(), minlength=n + 1)[1:])
        base += n
    return out, np.concatenate(sizes).astype(np.int64)


def curve(maps, masks):
    """(fpr, pro) at (0, 0) and every distinct score in descending order."""
    reg, sizes = regions(masks)
    s = np.concatenate([np.asarray(a, dtype=np.float32).ravel() for a in maps]) + np.float32(0.0)   # -0.0 -> +0.0
    if np.isnan(s).any():
        raise ValueError("NaN in a map")
    r = np.concatenate([x.ravel() for x in reg])
    n_reg, defect = len(sizes), r >= 0
    n_ok = int((~defect).sum())
    if n_reg == 0 or n_ok == 0:
        raise ValueError("need at least one defect region and one defect-free pixel")
    w = np.zeros(len(s))
    w[defect] = 1.0 / sizes[r[defect]]
    order = np.argsort(-s, kind="stable")
    s, w, defect = s[order], w[order], defect[order]
    fpr = np.cumsum(~defect) / n_ok
    pro = np.cumsum(w) / n_reg
    last = np.append(s[1:] != s[:-1], True)                 # last pixel of each run of equal scores
    return np.concatenate(([0.0], fpr[last])), np.concatenate(([0.0], pro[last]))


def area(fpr, pro, alpha):
    """(1 / alpha) * trapezoid area under the polyline (fpr, pro) from 0 to alpha; the segment crossing alpha is cut."""
    x0, x1, y0, y1 = fpr[:-1], fpr[1:].copy(), pro[:-1], pro[1:].copy()
    keep = x0 < alpha
    cut = keep & (x1 > alpha)
    y1[cut] = y0[cut] + (y1[cut] - y0[cut]) * (alpha - x0[cut]) / (x1[cut] - x0[cut])
    x1[cut] = alpha
    return float(np.sum(((x1 - x0) * (y0 + y1) * 0.5)[keep]) / alpha)


def au_pro(maps, masks, alpha=0.3):
    if not 0.0 < alpha <= 1.0:
        raise ValueError("alpha must be in (0, 1]")
    return area(*curve(maps, masks), alpha)


def pixel_auroc(maps, masks):
    from sklearn.metrics import roc_auc_score

    s = np.concatenate([np.asarray(a, dtype=np.float32).ravel() for a in maps]).astype(np.float64)
    y = np.concatenate([(np.asarray(m) != 0).ravel() for m in masks])
    return float(roc_auc_score(y, s))
