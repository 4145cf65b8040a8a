"""Drop-in for the reference's `src.metrics` (/root/reference/src/metrics.py): same four signatures, same
return types (Python floats), computed by the CUDA scoring kernel (csrc/scoring.cu) -- plus the batched
scorer the evaluator uses.  No CPU fallback: a CUDA device and libadsr_b200.so are required.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np
import torch

from . import ops


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("metrics need a CUDA device: this package has no CPU fallback")
    return torch.device("cuda")


def _as_hwc_batch(img: np.ndarray) -> torch.Tensor:
    a = np.asarray(img)
    t = torch.from_numpy(np.ascontiguousarray(a if a.dtype == np.uint8 else a.astype(np.float32)))
    if t.ndim == 2:
        t = t[:, :, None]
    return t[None].to(_device())


def _range_for(ref: np.ndarray, data_range: Optional[float]) -> float:
    if data_range is None:                                   # src/metrics.py:18-19, 30-31 (checked AFTER astype(float32))
        return 1.0
    return float(data_range)


def psnr_numpy(img_ref: np.ndarray, img: np.ndarray, data_range: Optional[float] = None) -> float:
    """src/metrics.py:15-23.  (The reference casts to float32 first, so `data_range=None` always means 1.0.)"""
    dr = _range_for(img_ref, data_range)
    ref, out = _as_hwc_batch(np.asarray(img_ref).astype(np.float32)), _as_hwc_batch(np.asarray(img).astype(np.float32))
    s = ops.score_images_strided(out, ref, "hwc", [], psnr_peak=dr)
    return float(s[0, 1].item())


def ssim_numpy(img_ref: np.ndarray, img: np.ndarray, win_size: int = 11, data_range: Optional[float] = None) -> float:
    """src/metrics.py:26-67: uniform win_size x win_size window, reflect padding, gray conversion for 3 channels."""
    dr = _range_for(img_ref, data_range)
    ref, out = _as_hwc_batch(np.asarray(img_ref).astype(np.float32)), _as_hwc_batch(np.asarray(img).astype(np.float32))
    if ref.shape[-1] == 2 or ref.shape[-1] > 3:
        raise ValueError("ssim_numpy supports HxW, HxWx1 and HxWx3 arrays")
    s = ops.score_images_strided(out, ref, "hwc", [int(win_size)], c1=(0.01 * dr) ** 2, c2=(0.03 * dr) ** 2, psnr_peak=dr)
    return float(s[0, 0].item())


def _shave(sr: torch.Tensor, hr: torch.Tensor, shave: int = 4):
    if sr.size(-1) > 2 * shave:                              # src/metrics.py:73-75, 88-91
        sr, hr = sr[..., shave:-shave, shave:-shave], hr[..., shave:-shave, shave:-shave]
    return sr, hr


def psnr_torch(sr: torch.Tensor, hr: torch.Tensor, rgb_range: float) -> float:
    """src/metrics.py:70-79: mean over the whole batch of ((sr-hr)/rgb_range)^2 on the 4-px shaved crop."""
    sr, hr = _shave(sr.float().to(_device()), hr.float().to(_device()))
    s = ops.score_images_strided(sr, hr, "chw", [], div=float(rgb_range))
    mse = float(s[:, 0].mean().item())
    if mse == 0:
        return float("inf")
    return 10.0 * float(np.log10(1.0 / mse))


def ssim_torch(sr: torch.Tensor, hr: torch.Tensor, rgb_range: float, win_size: int = 11) -> float:
    """src/metrics.py:82-108, including its quirks: zero-padded box filter and C1/C2 scaled by 255^2 on [0,1] data."""
    sr, hr = sr.float().to(_device()), hr.float().to(_device())
    if sr.size(-2) > hr.size(-2) or sr.size(-1) > hr.size(-1):
        sr = sr[..., :hr.size(-2), :hr.size(-1)]
    sr, hr = _shave(sr, hr)
    c1, c2 = (0.01 * 1.0) ** 2 * (255.0 ** 2), (0.03 * 1.0) ** 2 * (255.0 ** 2)
    s = ops.score_images_strided(sr, hr, "chw", [int(win_size)], div=float(rgb_range), clamp01=True, zero_pad=True, c1=c1,
                                 c2=c2)
    return float(s[:, 0].mean().item())


def window_sizes_for(min_dim: int) -> list[int]:
    """SSIM window sweep of src/evaluate.py:234-236."""
    max_w = max(3, min_dim - 3)
    return [w for w in range(3, max_w + 1, 10) if w % 2 == 1] or [3]


def score_batch(sr_u8: torch.Tensor, hr_u8: torch.Tensor, window_sizes: Sequence[int],
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 NHWC device tensors -> fp64 [B, n_ws + 2]: SSIM for every window size, MSE, PSNR (one launch)."""
    return ops.score_images(sr_u8, hr_u8, window_sizes, out)


def anomaly_maps(sr_u8: torch.Tensor, hr_u8: torch.Tensor, win_size: int = 11, sigma: float = 0.0):
    """Where an image is anomalous: uint8 NHWC device tensors -> (1 - SSIM map for one window size, squared-error map averaged over the
    channels, per-image max of both) as fp32 [B, H, W], fp32 [B, H, W], fp64 [B, 2].  sigma > 0 smooths both maps like
    scipy.ndimage.gaussian_filter(map, sigma, mode="reflect", truncate=4.0) before the max is taken."""
    return ops.anomaly_maps(sr_u8, hr_u8, win_size, sigma)


def pixel_auroc(maps, masks) -> float:
    """Pixel-level ROC AUC (the MVTec localisation number): every pixel of every map is one score, a non-zero mask pixel marks a defect.
    maps / masks: arrays (or sequences of per-image arrays) of matching shapes, on the host."""
    if isinstance(maps, (list, tuple)):
        if len(maps) != len(masks) or any(np.shape(a) != np.shape(k) for a, k in zip(maps, masks)):
            raise ValueError("pixel_auroc: every map needs a mask of its own shape")
        maps = np.concatenate([np.asarray(m).ravel() for m in maps]) if maps else np.empty(0)
        masks = np.concatenate([np.asarray(m).ravel() for m in masks]) if masks else np.empty(0)
    maps, masks = np.asarray(maps), np.asarray(masks)
    if maps.shape != masks.shape:
        raise ValueError(f"pixel_auroc: maps {maps.shape} and masks {masks.shape} differ in shape")
    return roc_auc((masks.ravel() != 0).astype(np.int64), maps.ravel())


def roc_auc(y_true, scores) -> float:
    """Image-level ROC AUC on the host (N_img scalars; stays on the CPU like the reference's sklearn call,
    src/evaluate.py:245,263-265).  Uses sklearn when available, else the equivalent rank statistic."""
    try:
        from sklearn.metrics import roc_auc_score

        return float(roc_auc_score(np.asarray(y_true), np.asarray(scores, dtype=np.float64)))
    except ImportError:                                      # pragma: no cover
        from scipy.stats import rankdata

        y, s = np.asarray(y_true), np.asarray(scores, dtype=np.float64)
        r = rankdata(s)
        n1, n0 = int((y == 1).sum()), int((y == 0).sum())
        return float((r[y == 1].sum() - n1 * (n1 + 1) / 2.0) / (n1 * n0))


def aucs_from_scores(y_true, scores: np.ndarray, window_sizes: Sequence[int]):
    """Best-window selection and the three AUCs exactly as src/evaluate.py:238-265 (strict '>' keeps the first
    window size on ties).  scores: [n_img, n_ws + 2] as returned by score_batch."""
    n_ws = len(window_sizes)
    best_ws, best_auc, best_j = window_sizes[0], -1.0, 0
    for j, ws in enumerate(window_sizes):
        a = roc_auc(y_true, 1.0 - scores[:, j])
        if a > best_auc:
            best_auc, best_ws, best_j = a, ws, j
    return (best_ws, roc_auc(y_true, 1.0 - scores[:, best_j]), roc_auc(y_true, scores[:, n_ws]),
            roc_auc(y_true, -scores[:, n_ws + 1]))
