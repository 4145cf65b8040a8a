"""Drop-in for the reference's `src.metrics` (/root/reference/src/metrics.py): same four signatures, same
return types (Python floats), computed by the CUDA scoring kernel (csrc/scoring.cu) -- plus the batched
scorer the evaluator uses.  No CPU fallback: a CUDA device and libadsr_b200.so are required.
"""
from __future__ import annotations

from typing import NamedTuple, Optional, Sequence

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


def gms_map(sr_u8: torch.Tensor, hr_u8: torch.Tensor, sigma: float = 0.0):
    """Where edge structure was not reconstructed: uint8 NHWC device tensors -> (multi-scale gradient-magnitude-similarity map, per-image
    max) as fp32 [B, H, W], fp64 [B].  RIAD's MSGMS on the gray plane of anomaly_maps: 4 pyramid levels of 2 x 2 means, Prewitt gradient
    magnitudes, 1 - GMS with c = 0.0026 per level, bilinear upsampling, mean over the levels.  sigma > 0 smooths it like anomaly_maps
    before the max is taken."""
    return ops.gms_map(sr_u8, hr_u8, sigma)


def _map_pieces(maps):
    """A CUDA map set -> (list of fp32 tensors to append in order, list of per-image (H, W) shapes)."""
    if isinstance(maps, torch.Tensor):
        if maps.dim() != 3:
            raise ValueError(f"maps: expected a [N, H, W] tensor, got shape {tuple(maps.shape)}")
        pieces, shapes = [maps], [tuple(maps.shape[1:])] * maps.shape[0]
    else:
        pieces = list(maps)
        if any(not isinstance(m, torch.Tensor) or m.dim() != 2 for m in pieces):
            raise ValueError("maps: expected a [N, H, W] tensor or a sequence of [H, W] tensors")
        shapes = [tuple(m.shape) for m in pieces]
    for m in pieces:
        ops._cuda(m, "maps")
        if m.dtype != torch.float32:
            raise TypeError(f"maps must be float32, got {m.dtype}")
    return pieces, shapes


class LocalisationMetrics(NamedTuple):
    """The localisation numbers of one anomaly map over a whole test set (LocalisationAccumulator.results).  f1_threshold is an oracle
    threshold: it is chosen with the ground truth of the very pixels it is scored on (anomalib's adaptive threshold is also picked from
    labelled data, but from a validation set)."""
    pixel_auroc: float
    au_pro: float
    pixel_ap: float         # area under the pixel precision-recall curve (sklearn's average_precision_score)
    f1_max: float           # the best pixel F1 over all thresholds
    f1_threshold: float     # the fp32 score that attains it: `map >= f1_threshold` is the F1-max defect mask


class ThresholdMetrics(NamedTuple):
    """The pixel metrics of the prediction `map >= threshold` over a whole test set (LocalisationAccumulator.at_threshold).  Precision
    is 0 when nothing is predicted; recall, fpr, f1 and iou are NaN when their denominator is 0, pro when there is no defect region."""
    threshold: float
    tp: int                 # predicted defect pixels that are defects
    fp: int                 # predicted defect pixels that are defect-free
    fn: int                 # defect pixels not predicted
    tn: int                 # defect-free pixels not predicted
    precision: float        # tp / (tp + fp)
    recall: float           # tp / (tp + fn)
    fpr: float              # fp / (fp + tn)
    f1: float               # 2 tp / (2 tp + fp + fn)
    iou: float              # tp / (tp + fp + fn)
    pro: float              # mean over the defect regions of the share of the region's pixels predicted


def inverted_cdf_rank(n: int, q: float) -> int:
    """The 1-based rank k of np.quantile(x, q, method="inverted_cdf") among n sorted float64 values: max(1, ceil(q n)), with q n
    formed in float64 exactly as numpy forms it (so q = 0.28, n = 25 gives k = 8: 0.28 * 25 rounds to 7.000000000000001).  (Given an
    fp32 array numpy forms q n in fp32 instead, which misranks and fails beyond 2^24 values; the scores convert to float64 exactly.)"""
    index = np.float64(n) * np.float64(q) - 1.0
    prev = np.floor(index)
    k0 = int(prev) if index == prev else int(prev) + 1
    return max(k0, 0) + 1


def fp32_at_least(threshold: float) -> np.float32:
    """The smallest fp32 >= threshold: for every fp32 x, x >= result <=> x >= threshold (the exact double)."""
    t = np.float32(threshold)
    if float(t) < threshold:                          # a Python float against np.float32 would be compared in fp32
        t = np.nextafter(t, np.float32(np.inf))
    return t


class LocalisationAccumulator:
    """Pixel AUROC, AU-PRO, pixel AP and F1-max of `n_maps` anomaly maps over a whole test set, fed one batch at a time.

    append(maps, masks=None): maps = one entry per map, each a CUDA fp32 [B, H, W] tensor or a sequence of [H, W] tensors (any sizes);
    masks = the host masks of the same B images (non-zero = defect), or None: every pixel is defect-free (calibration images).  The maps are copied on the device into one growing buffer per map
    (no device -> host copy); each mask is labelled once on the host (scipy.ndimage.label, 8-connectivity) and its per-pixel region
    indices are shared by all maps.  results(fpr_limit) runs adsr_localisation_metrics once per map and returns one LocalisationMetrics
    per map, finish(fpr_limit) the [(pixel_auroc, au_pro), ...] part of it: the same numbers for the same image sequence however it was
    split into batches.  segmentation(map_index, threshold) thresholds the accumulated maps into per-image defect masks,
    at_threshold(map_index, threshold) scores that prediction against the masks, quantile(map_index, q) is an exact score quantile."""

    def __init__(self, n_maps: int = 1):
        self.n_maps = int(n_maps)
        self._maps = [None] * self.n_maps             # device fp32 buffers, capacity >= self.n
        self._regions = None                          # device int32 buffer: -1 = defect-free, else the global region index
        self.n = 0
        self.n_ok = 0
        self._sizes = []                              # host int64 region sizes, one array per image with defects
        self._shapes = []                             # (H, W) of every appended image, in append order

    @property
    def n_regions(self) -> int:
        return sum(len(s) for s in self._sizes)

    def _reserve(self, n_new: int, device) -> None:
        need = self.n + n_new
        cap = 0 if self._regions is None else self._regions.numel()
        if need <= cap:
            return
        cap = max(need, 2 * cap)
        grow = lambda old, dt: (torch.empty(cap, dtype=dt, device=device) if old is None else
                                torch.cat([old[:self.n], torch.empty(cap - self.n, dtype=dt, device=device)]))
        self._maps = [grow(m, torch.float32) for m in self._maps]
        self._regions = grow(self._regions, torch.int32)

    def append(self, maps, masks=None) -> None:
        from scipy.ndimage import label

        if len(maps) != self.n_maps:
            raise ValueError(f"append: {len(maps)} maps given, the accumulator holds {self.n_maps}")
        parts = [_map_pieces(m) for m in maps]
        shapes = parts[0][1]
        if masks is None:                             # defect-free images: no labelling, every region index is -1
            if any(p[1] != shapes for p in parts):
                raise ValueError("append: all maps must hold the same images")
            n_new = sum(h * w for h, w in shapes)
            self._reserve(n_new, parts[0][0][0].device)
            self._copy_maps(parts)
            self._regions[self.n:self.n + n_new].fill_(-1)
            self._shapes += shapes
            self.n += n_new
            self.n_ok += n_new
            return
        masks = [np.asarray(k) for k in masks]
        if any(p[1] != shapes for p in parts) or len(masks) != len(shapes) or any(k.shape != s for k, s in zip(masks, shapes)):
            raise ValueError("append: every map needs a mask of its own shape, and all maps the same images")
        regions, sizes, n_ok, n_reg = [], [], 0, self.n_regions
        for k in masks:
            lab, nr = label(k != 0, structure=np.ones((3, 3), dtype=int))
            lab = lab.ravel()
            regions.append(np.where(lab > 0, lab + (n_reg - 1), -1).astype(np.int32))
            if nr:
                sizes.append(np.bincount(lab, minlength=nr + 1)[1:].astype(np.int64))
            n_ok += int((lab == 0).sum())
            n_reg += nr
        if n_reg > np.iinfo(np.int32).max:
            raise ValueError("append: more than 2^31 - 1 defect regions")
        n_new = sum(k.size for k in masks)
        device = parts[0][0][0].device
        self._reserve(n_new, device)
        self._copy_maps(parts)
        if n_new:
            self._regions[self.n:self.n + n_new].copy_(torch.from_numpy(np.concatenate(regions)))
        self._sizes += sizes
        self._shapes += shapes
        self.n += n_new
        self.n_ok += n_ok

    def _copy_maps(self, parts) -> None:
        for buf, (pieces, _) in zip(self._maps, parts):
            off = self.n
            for m in pieces:
                buf[off:off + m.numel()].copy_(m.reshape(-1))
                off += m.numel()

    def results(self, fpr_limit: float = 0.3) -> list[LocalisationMetrics]:
        """One LocalisationMetrics per map (AU-PRO up to FPR = fpr_limit).  ValueError: fpr_limit outside (0, 1], no defect region
        (R == 0), no defect-free pixel, or a NaN in a map."""
        fpr_limit = float(fpr_limit)
        if not 0.0 < fpr_limit <= 1.0:
            raise ValueError(f"fpr_limit must be in (0, 1], got {fpr_limit}")
        if self.n_regions == 0:
            raise ValueError("localisation metrics need at least one defect region (all masks are empty)")
        if self.n_ok == 0:
            raise ValueError("localisation metrics need at least one defect-free pixel")
        device = self._regions.device
        sizes = torch.from_numpy(np.concatenate(self._sizes)).to(device)
        ws = torch.empty(ops.localisation_workspace_bytes(self.n), dtype=torch.uint8, device=device)
        out = torch.empty(self.n_maps, 8, dtype=torch.float64, device=device)
        for j, buf in enumerate(self._maps):
            ops.localisation_metrics(buf[:self.n], self._regions[:self.n], sizes, self.n_ok, fpr_limit, ws, out[j])
        res = out.cpu().numpy()
        for j in range(self.n_maps):
            if res[j, 2]:
                raise ValueError(f"map {j} holds {int(res[j, 2])} NaN scores")
            if res[j, 3] != self.n_ok or res[j, 4]:
                raise RuntimeError(f"localisation metrics: inconsistent region indices on the device (map {j}: {res[j, 2:]})")
        return [LocalisationMetrics(*(float(r[k]) for k in (0, 1, 5, 6, 7))) for r in res]

    def finish(self, fpr_limit: float = 0.3):
        """[(pixel AUROC, AU-PRO@fpr_limit)] per map, from results() (same checks and errors)."""
        return [(r.pixel_auroc, r.au_pro) for r in self.results(fpr_limit)]

    def segmentation(self, map_index: int, threshold: float) -> list[np.ndarray]:
        """Predicted defect masks: bool [H, W] host arrays `map >= threshold` of map `map_index`, one per appended image in append order
        (one comparison on the device over the accumulated map, one device -> host copy).  With the f1_threshold of results() they are
        the masks that attain F1-max.  The comparison is that of the fp32 map with the exact double `threshold`."""
        j = self._map_index(map_index, "segmentation")
        t = fp32_at_least(threshold)
        if self.n == 0:
            return []
        flat = (self._maps[j][:self.n] >= float(t)).cpu().numpy()
        out, off = [], 0
        for h, w in self._shapes:
            out.append(flat[off:off + h * w].reshape(h, w))
            off += h * w
        return out

    def _map_index(self, map_index: int, what: str) -> int:
        j = int(map_index)
        if not 0 <= j < self.n_maps:
            raise IndexError(f"{what}: map {map_index} of {self.n_maps}")
        return j

    def quantile(self, map_index: int, q: float) -> float:
        """The exact q-quantile of all accumulated scores of map `map_index`: np.quantile(scores.astype(float64), q,
        method="inverted_cdf"), the fp32 score of rank k = inverted_cdf_rank(n, q) (no interpolation; -0.0 reported as +0.0), found on the device by a radix select.
        ValueError: q outside [0, 1], nothing appended, or a NaN in the map."""
        j = self._map_index(map_index, "quantile")
        q = float(q)
        if not 0.0 <= q <= 1.0:
            raise ValueError(f"quantile: q must be in [0, 1], got {q}")
        if self.n == 0:
            raise ValueError("quantile: no scores appended")
        device = self._regions.device
        ws = torch.empty(ops.localisation_workspace_bytes(self.n), dtype=torch.uint8, device=device)
        out = torch.empty(2, dtype=torch.float64, device=device)
        ops.score_quantile(self._maps[j][:self.n], inverted_cdf_rank(self.n, q), ws, out)
        score, nan = out.tolist()
        if nan:
            raise ValueError(f"map {j} holds {int(nan)} NaN scores")
        return score

    def at_threshold(self, map_index: int, threshold: float) -> ThresholdMetrics:
        """The pixel metrics of the prediction `map >= threshold` of map `map_index` against the appended masks: the comparison of
        segmentation() (the fp32 map against the exact double threshold), counted on the device in one pass.  ValueError: a NaN
        threshold, nothing appended, or a NaN in the map."""
        j = self._map_index(map_index, "at_threshold")
        threshold = float(threshold)
        if threshold != threshold:
            raise ValueError("at_threshold: the threshold is NaN")
        if self.n == 0:
            raise ValueError("at_threshold: no scores appended")
        device = self._regions.device
        sizes = torch.from_numpy(np.concatenate(self._sizes)).to(device) if self._sizes else None
        ws = torch.empty(ops.localisation_workspace_bytes(self.n), dtype=torch.uint8, device=device)
        out = torch.empty(7, dtype=torch.float64, device=device)
        ops.threshold_metrics(self._maps[j][:self.n], self._regions[:self.n], sizes, float(fp32_at_least(threshold)), ws, out)
        r = out.tolist()
        if r[5]:
            raise ValueError(f"map {j} holds {int(r[5])} NaN scores")
        tp, fp, fn, tn = (int(v) for v in r[:4])
        if r[6] or fp + tn != self.n_ok:
            raise RuntimeError(f"threshold metrics: inconsistent region indices on the device (map {j}: {r})")
        ratio = lambda a, b: a / b if b else float("nan")
        return ThresholdMetrics(threshold, tp, fp, fn, tn, tp / (tp + fp) if tp + fp else 0.0, ratio(tp, tp + fn), ratio(fp, fp + tn),
                                ratio(2 * tp, 2 * tp + fp + fn), ratio(tp, tp + fp + fn), r[4])


REGION_COLUMNS = ("image", "label", "area", "y0", "x0", "y1", "x1", "sum_y", "sum_x", "peak", "peak_y", "peak_x")


def region_dtype(with_gt: bool) -> np.dtype:
    """Row type of DefectRegions.regions: int64 columns, peak float32, gt_pixels only with ground truth."""
    cols = REGION_COLUMNS + (("gt_pixels",) if with_gt else ())
    return np.dtype([(c, np.float32 if c == "peak" else np.int64) for c in cols])


class DefectRegions(NamedTuple):
    """The defects of a batch of anomaly maps (defect_regions).  regions has one row per region, sorted by (image, label): area,
    the half-open box y0 <= y < y1, x0 <= x < x1 (scipy.ndimage.find_objects), the integer sums of y and x (centroid = sum / area),
    the largest fp32 score and the first raster pixel that attains it, and with masks the region's ground-truth pixels."""
    labels: torch.Tensor                  # CUDA int32 [B, H, W]: 0 = background, 1..n_regions[b] = the regions of image b
    regions: np.ndarray                   # host table, dtype region_dtype(masks given)
    n_regions: np.ndarray                 # int64 [B] regions per image
    gt_regions: Optional[np.ndarray]      # int64 [B] ground-truth regions (8-connected components of the mask) per image, with masks
    gt_detected: Optional[np.ndarray]     # int64 [B] of those, the ones holding a pixel of a region, with masks


def _region_counts(counts: torch.Tensor, workspace: torch.Tensor, what: str) -> np.ndarray:
    host = torch.cat([counts, workspace[:4].view(torch.int32)]).cpu().numpy().astype(np.int64)
    if host[-1]:
        raise RuntimeError(f"{what}: {int(host[-1])} union-find loops or labels out of range on the device")
    return host[:-1]


def defect_regions(maps: torch.Tensor, threshold: float, min_area: int = 1, masks=None) -> DefectRegions:
    """Every 8-connected blob of `maps >= threshold` as one defect: maps = CUDA fp32 [B, H, W], compared with the exact double
    threshold like LocalisationAccumulator.segmentation (a NaN score is never foreground; pass evaluate.above(t) for the strict
    `map > t`).  Blobs of fewer than min_area pixels are dropped, the rest numbered 1..n per image in raster order of their first pixel
    (scipy.ndimage.label of the kept foreground with structure ones((3, 3))).  masks (bool / uint8 [B, H, W], host or device, non-zero
    = defect) add gt_pixels per region and the ground-truth regions and detections per image.  Labels and statistics are computed on
    the device with integer atomics (csrc/regions.cu): the same bits on every run and for an image whatever batch it is in."""
    ops._cuda(maps, "maps")
    if maps.dtype != torch.float32 or maps.dim() != 3:
        raise ValueError(f"defect_regions: maps must be a float32 [B, H, W] tensor, got {maps.dtype} {tuple(maps.shape)}")
    threshold = float(threshold)
    if threshold != threshold:
        raise ValueError("defect_regions: the threshold is NaN")
    if int(min_area) != min_area or int(min_area) < 1:
        raise ValueError(f"defect_regions: min_area must be an integer >= 1, got {min_area}")
    maps = maps.contiguous()
    b, h, w = maps.shape
    dev = maps.device
    ws = torch.empty(ops.regions_workspace_bytes(b, h, w), dtype=torch.uint8, device=dev)
    labels = torch.empty(b, h, w, dtype=torch.int32, device=dev)
    counts = torch.empty(b, dtype=torch.int32, device=dev)
    ops.label_regions(maps, float(fp32_at_least(threshold)), None, int(min_area), ws, labels, counts)
    n_regions = _region_counts(counts, ws, "label_regions")
    gt_labels = gt_off = gt_hit = gt_regions = None
    if masks is not None:
        m = masks if isinstance(masks, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(masks)))
        if tuple(m.shape) != (b, h, w):
            raise ValueError(f"defect_regions: masks {tuple(m.shape)} for maps {(b, h, w)}")
        m = (m.to(dev) != 0).to(torch.uint8).contiguous()
        gt_ws = torch.empty_like(ws)
        gt_labels = torch.empty_like(labels)
        gt_counts = torch.empty_like(counts)
        ops.label_regions(None, 0.0, m, 1, gt_ws, gt_labels, gt_counts)
        gt_regions = _region_counts(gt_counts, gt_ws, "label_regions (masks)")
        gt_off = torch.from_numpy(np.concatenate([[0], np.cumsum(gt_regions)]).astype(np.int64)).to(dev)
        gt_hit = torch.empty(int(gt_regions.sum()), dtype=torch.int32, device=dev)
    offsets = np.concatenate([[0], np.cumsum(n_regions)]).astype(np.int64)
    n_rows = int(offsets[-1])
    table = torch.empty(n_rows, 9, dtype=torch.int64, device=dev)
    ops.region_stats(labels, maps, gt_labels, torch.from_numpy(offsets).to(dev), gt_off, ws, table, gt_hit)
    tab = table.cpu().numpy()
    _region_counts(counts[:0], ws, "region_stats")            # no counts: only the error counter (labels out of range)
    out = np.zeros(n_rows, dtype=region_dtype(masks is not None))
    out["image"] = np.repeat(np.arange(b), n_regions)
    out["label"] = np.arange(n_rows) - np.repeat(offsets[:-1], n_regions) + 1
    for name, col in (("area", 0), ("y0", 1), ("x0", 2), ("sum_y", 5), ("sum_x", 6)):
        out[name] = tab[:, col]
    out["y1"], out["x1"] = tab[:, 3] + 1, tab[:, 4] + 1
    key = tab[:, 7].view(np.uint64)
    k = (key >> np.uint64(32)).astype(np.uint32)             # order-preserving key: sign bit set for scores >= 0, all bits flipped below
    out["peak"] = np.where(k & np.uint32(0x80000000), k & np.uint32(0x7fffffff), ~k).astype(np.uint32).view(np.float32)
    idx = (~(key & np.uint64(0xffffffff))).astype(np.uint32).astype(np.int64)   # the low word holds ~(y W + x)
    out["peak_y"], out["peak_x"] = idx // w, idx % w
    gt_detected = None
    if masks is not None:
        out["gt_pixels"] = tab[:, 8]
        hit = gt_hit.cpu().numpy().astype(np.int64)
        gt_detected = np.bincount(np.repeat(np.arange(b), gt_regions), weights=hit, minlength=b).astype(np.int64)
    return DefectRegions(labels, out, n_regions, gt_regions, gt_detected)


def _on_device(maps) -> bool:
    if isinstance(maps, torch.Tensor):
        return maps.is_cuda
    return isinstance(maps, (list, tuple)) and len(maps) > 0 and isinstance(maps[0], torch.Tensor) and maps[0].is_cuda


def au_pro(maps, masks, fpr_limit: float = 0.3) -> float:
    """AU-PRO@fpr_limit (the MVTec AD per-region-overlap localisation number): maps = CUDA fp32 [N, H, W] tensor or a sequence of
    [H, W] tensors of any sizes, masks = host arrays of the same shapes (non-zero = defect).  Defect regions are the 8-connected
    components of each mask, every region weighs the same; the (FPR, PRO) curve has one point per distinct score and its trapezoid
    area up to FPR = fpr_limit is divided by fpr_limit.  Computed on the device (adsr_localisation_metrics)."""
    acc = LocalisationAccumulator(1)
    acc.append([maps], masks)
    return acc.finish(fpr_limit)[0][1]


def pixel_ap(maps, masks) -> float:
    """Pixel-level average precision (area under the precision-recall curve; sklearn.metrics.average_precision_score over every pixel,
    ties included): maps = CUDA fp32 [N, H, W] tensor or a sequence of [H, W] tensors, masks = host arrays of the same shapes (non-zero
    = defect).  Computed on the device (adsr_localisation_metrics)."""
    acc = LocalisationAccumulator(1)
    acc.append([maps], masks)
    return acc.results()[0].pixel_ap


def f1_max(maps, masks) -> tuple[float, float]:
    """(best pixel F1 over all thresholds, the fp32 score that attains it; on a tie the higher one) of CUDA maps against host masks,
    inputs as pixel_ap.  `map >= threshold` reproduces the F1.  An oracle threshold: chosen on the ground truth it is scored on."""
    acc = LocalisationAccumulator(1)
    acc.append([maps], masks)
    r = acc.results()[0]
    return r.f1_max, r.f1_threshold


def score_quantile(maps, q: float) -> float:
    """np.quantile(scores.astype(float64), q, method="inverted_cdf") of every pixel of CUDA fp32 maps (an [N, H, W] tensor or a sequence of [H, W]
    tensors): an actual score, exact, found on the device (adsr_score_quantile); also beyond the 2^24 elements torch.quantile takes."""
    acc = LocalisationAccumulator(1)
    acc.append([maps])
    return acc.quantile(0, q)


def pixel_auroc(maps, masks) -> float:
    """Pixel-level ROC AUC (the MVTec localisation number): every pixel of every map is one score, a non-zero mask pixel marks a defect.
    maps / masks: arrays (or sequences of per-image arrays) of matching shapes, on the host.  CUDA maps (an fp32 [N, H, W] tensor or a
    sequence of [H, W] tensors) with host masks are ranked on the device instead, as au_pro does (the same value)."""
    if _on_device(maps):
        acc = LocalisationAccumulator(1)
        acc.append([maps], masks)
        return acc.finish()[0][0]
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
