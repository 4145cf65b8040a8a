"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's anomaly scoring.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline / `--impl reference` legs may
import this file.

What is restated (citations into /root/reference):
  * uint8 quantisation of SR / HR ........ src/evaluate.py:212-215  (mul, clamp, .byte() = TRUNCATION)
  * ssim_numpy ........................... src/metrics.py:26-67  (gray conversion :37-39, reflect pad
                                            + uniform ws x ws mean :45-56, C1/C2 :30-33, SSIM map :58-67)
  * MSE / psnr_numpy ..................... src/evaluate.py:259-260, src/metrics.py:15-23
  * window-size sweep + best-ws + AUCs ... src/evaluate.py:233-265
  * roc_auc_score ........................ sklearn (third party, scikit-learn==1.7.1 in
                                            requirements.lock.txt:52): rank statistic with tie handling;
                                            restated here as the Mann-Whitney U form.

Two SSIM restatements are kept:
  * `ssim_loops`  -- literal per-pixel fp32 loop (O(H*W*ws^2)); only for tiny cases in tests.
  * `ssim_box`    -- vectorised: fp64 prefix sums over the reflect-padded image.  Differs from the
                     reference's fp32 `np.sum(region*kernel)` only by summation rounding (<= 1e-6 on
                     the SSIM value, measured in tests/test_oracle_pinning.py against the reference).
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np

GRAY_COEFFS = np.array([65.738, 129.057, 25.064], dtype=np.float32) / np.float32(256.0)  # src/metrics.py:37


def quantize_u8(x: np.ndarray, rgb_range: float) -> np.ndarray:
    """[.., C, H, W] float in [0, rgb_range] -> uint8 [.., H, W, C] (src/evaluate.py:214-215).
    torch: x.mul(255 / rgb_range).clamp(0, 255).byte()  -- fp32 multiply, truncation toward zero."""
    y = x.astype(np.float32) * np.float32(255.0 / rgb_range)
    y = np.clip(y, np.float32(0), np.float32(255)).astype(np.uint8)
    return np.moveaxis(y, -3, -1)


def to_gray01(img_u8: np.ndarray) -> np.ndarray:
    """uint8 [H, W, C] -> float32 [H, W] in [0,1] exactly as evaluate.py:241 + metrics.py:35-43 do."""
    f = img_u8.astype(np.float32) / np.float32(255.0)
    if f.ndim == 3:
        if f.shape[2] > 1:
            f = np.tensordot(f, GRAY_COEFFS, axes=([2], [0]))
        else:
            f = f[:, :, 0]
    return f.astype(np.float32)


def ssim_loops(ref01: np.ndarray, out01: np.ndarray, ws: int) -> float:
    """Literal restatement of metrics.py:45-67 (fp32, per-pixel window sums). Gray [H, W] inputs in [0,1]."""
    C1, C2 = (0.01 * 1.0) ** 2, (0.03 * 1.0) ** 2
    pad = ws // 2
    inv = np.float32(1.0) / np.float32(ws * ws)

    def box(x):
        xp = np.pad(x, ((pad, pad), (pad, pad)), mode="reflect")
        o = np.empty_like(x, dtype=np.float32)
        for i in range(x.shape[0]):
            for j in range(x.shape[1]):
                o[i, j] = np.float32(np.sum(xp[i:i + ws, j:j + ws] * inv))
        return o

    ref, out = ref01.astype(np.float32), out01.astype(np.float32)
    mu1, mu2 = box(ref), box(out)
    s1 = box(ref * ref) - mu1 * mu1
    s2 = box(out * out) - mu2 * mu2
    s12 = box(ref * out) - mu1 * mu2
    m = ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 * mu1 + mu2 * mu2 + C1) * (s1 + s2 + C2))
    return float(np.mean(m))


def _box_mean_f64(x: np.ndarray, ws: int) -> np.ndarray:
    pad = ws // 2
    xp = np.pad(x.astype(np.float64), ((pad, pad), (pad, pad)), mode="reflect")
    c = np.zeros((xp.shape[0] + 1, xp.shape[1] + 1), dtype=np.float64)
    c[1:, 1:] = xp.cumsum(0).cumsum(1)
    H, W = x.shape
    s = c[ws:ws + H, ws:ws + W] - c[:H, ws:ws + W] - c[ws:ws + H, :W] + c[:H, :W]
    return s / float(ws * ws)


def ssim_box(ref01: np.ndarray, out01: np.ndarray, ws: int) -> float:
    """Vectorised metrics.py:26-67 for gray [H, W] float32 inputs in [0,1] (data_range 1.0)."""
    C1, C2 = (0.01 * 1.0) ** 2, (0.03 * 1.0) ** 2
    ref, out = ref01.astype(np.float32), out01.astype(np.float32)
    mu1, mu2 = _box_mean_f64(ref, ws), _box_mean_f64(out, ws)
    # the reference squares in fp32 before filtering (ref * ref on float32 arrays)
    s1 = _box_mean_f64(ref * ref, ws) - mu1 * mu1
    s2 = _box_mean_f64(out * out, ws) - mu2 * mu2
    s12 = _box_mean_f64(ref * out, ws) - mu1 * mu2
    m = ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 * mu1 + mu2 * mu2 + C1) * (s1 + s2 + C2))
    return float(np.mean(m))


# ---------------------------------------------------------------------------------------------------------------------
# kernel-faithful restatement: what csrc/scoring.cu and csrc/anomaly_maps.cu compute, to the last bits, for tests that hold the
# kernels to ~1e-10 instead of the reference's fp32 tolerance
# ---------------------------------------------------------------------------------------------------------------------
def gray01_like_kernel(img: np.ndarray) -> np.ndarray:
    """[H, W, C] (C = 1 or 3) -> fp32 [H, W] gray plane as the kernels build it.  uint8 input is divided by 255 in fp32 first; float
    input is taken as is.  One channel: as is.  Three channels: the kernels' fmaf chain fmaf(b, c2, fmaf(g, c1, r * c0)) -- r * c0
    rounded to fp32, then each fmaf formed exactly and rounded once to fp32 (np.longdouble holds the exact sum of an fp32 product and
    an fp32 value of these magnitudes).  This is NOT the reference's formula: `to_gray01` uses np.tensordot, which can differ from the
    kernels in the last bit of a pixel."""
    f = img.astype(np.float32) / np.float32(255.0) if img.dtype == np.uint8 else img.astype(np.float32)
    if f.ndim == 2:
        return f
    if f.shape[2] == 1:
        return f[:, :, 0]
    c0, c1, c2 = (np.longdouble(c) for c in GRAY_COEFFS)
    r, g, b = (f[:, :, k].astype(np.longdouble) for k in range(3))
    p0 = (r * c0).astype(np.float32)
    t1 = (g * c1 + p0.astype(np.longdouble)).astype(np.float32)
    return (b * c2 + t1.astype(np.longdouble)).astype(np.float32)


def _prefix2d(x: np.ndarray, pad: int, mode: str) -> np.ndarray:
    xp = np.pad(x, pad, mode=mode)
    c = np.zeros((xp.shape[0] + 1, xp.shape[1] + 1), dtype=np.float64)
    c[1:, 1:] = xp.cumsum(0).cumsum(1)
    return c


def ssim_maps_like_kernel(ref: np.ndarray, out: np.ndarray, window_sizes: Sequence[int], c1: float = 0.01 * 0.01,
                          c2: float = 0.03 * 0.03, zero_pad: bool = False):
    """Per-pixel SSIM maps (fp64 [H, W], one per odd window size, yielded in order) of two fp32 gray planes [H, W] as the kernels form
    them: window sums of the values and of their fp32 products (x * x, y * y, x * y) with np.pad(mode="reflect") borders (zero_pad:
    zeros, as ssim_torch), then the fp64 term of ssim_term in csrc/adsr_kernels.h (every operation rounded on its own, means =
    sums * (1 / ws^2)).  The window sums come from a 2-D prefix of each plane split as hi + lo, hi a multiple of 2^-20: the hi sums
    are exact and the lo sums tiny, so each window sum is the exact one to ~1e-16 relative, well inside the kernels' own rounding.
    (A plain fp64 prefix reaches H * W in magnitude and loses ~1e-13 on one window, which 1 / C2 turns into ~1e-10 of SSIM.)"""
    planes = [ref.astype(np.float32), out.astype(np.float32)]
    planes += [planes[0] * planes[0], planes[1] * planes[1], planes[0] * planes[1]]
    H, W = ref.shape
    P = max(window_sizes) // 2
    mode = "constant" if zero_pad else "reflect"
    prefixes = []
    for x in planes:
        x = x.astype(np.float64)
        hi = np.round(x * 2.0 ** 20) / 2.0 ** 20
        prefixes.append((_prefix2d(hi, P, mode), _prefix2d(x - hi, P, mode)))
    for ws in window_sizes:
        a, e = P - ws // 2, P + ws // 2 + 1           # prefix rows / columns bounding the window of pixel 0

        def box(c):
            return c[e:e + H, e:e + W] - c[a:a + H, e:e + W] - c[e:e + H, a:a + W] + c[a:a + H, a:a + W]

        inv_n = 1.0 / (float(ws) * ws)
        mu1, mu2, e11, e22, e12 = ((box(ch) + box(cl)) * inv_n for ch, cl in prefixes)
        m11, m22, m12 = mu1 * mu1, mu2 * mu2, mu1 * mu2
        s1, s2, s12 = e11 - m11, e22 - m22, e12 - m12
        yield ((2.0 * m12 + c1) * (2.0 * s12 + c2)) / ((m11 + m22 + c1) * (s1 + s2 + c2))


def ssim_sweep_like_kernel(ref: np.ndarray, out: np.ndarray, window_sizes: Sequence[int], c1: float = 0.01 * 0.01,
                           c2: float = 0.03 * 0.03, zero_pad: bool = False) -> np.ndarray:
    """The scorer's SSIM for each window size: the mean of each of ssim_maps_like_kernel's maps."""
    return np.array([np.mean(m) for m in ssim_maps_like_kernel(ref, out, window_sizes, c1, c2, zero_pad)], dtype=np.float64)


def mse_like_kernel(sr01: np.ndarray, hr01: np.ndarray) -> float:
    """Mean over every element of (sr - hr)^2 with the difference and its square in fp32, summed in fp64 (the kernels' MSE term)."""
    d = sr01.astype(np.float32) - hr01.astype(np.float32)
    return float(np.sum((d * d).astype(np.float64)) / d.size)


def mse01(sr_u8: np.ndarray, hr_u8: np.ndarray) -> float:
    """src/evaluate.py:255-260."""
    d = sr_u8.astype(np.float32) / np.float32(255.0) - hr_u8.astype(np.float32) / np.float32(255.0)
    return float(np.mean(d * d))


def psnr01(hr_u8: np.ndarray, sr_u8: np.ndarray) -> float:
    """psnr_numpy(hr_f, sr_f) with float inputs => data_range 1.0 (src/metrics.py:15-23)."""
    m = mse01(sr_u8, hr_u8)
    if m == 0:
        return float("inf")
    return 10.0 * float(np.log10(1.0 / m))


def window_sizes_for(min_dim: int) -> List[int]:
    """src/evaluate.py:234-236."""
    max_w = max(3, min_dim - 3)
    return [w for w in range(3, max_w + 1, 10) if w % 2 == 1] or [3]


def roc_auc(y_true: Sequence[int], scores: Sequence[float]) -> float:
    """Area under the ROC curve == P(score_pos > score_neg) + 0.5 P(tie)  (what sklearn computes)."""
    y = np.asarray(y_true)
    s = np.asarray(scores, dtype=np.float64)
    pos, neg = s[y == 1], s[y == 0]
    if len(pos) == 0 or len(neg) == 0:
        raise ValueError("AUC needs both classes")
    order = np.argsort(s, kind="mergesort")
    ranks = np.empty(len(s), dtype=np.float64)
    sorted_s = s[order]
    i = 0
    while i < len(s):
        j = i
        while j + 1 < len(s) and sorted_s[j + 1] == sorted_s[i]:
            j += 1
        ranks[order[i:j + 1]] = 0.5 * (i + j) + 1.0
        i = j + 1
    u = ranks[y == 1].sum() - len(pos) * (len(pos) + 1) / 2.0
    return float(u / (len(pos) * len(neg)))


def score_images(sr_u8: Sequence[np.ndarray], hr_u8: Sequence[np.ndarray], window_sizes: Sequence[int]):
    """Per-image score table: ssim[n_img, n_ws], mse[n_img], psnr[n_img]."""
    n = len(sr_u8)
    ssim = np.zeros((n, len(window_sizes)), dtype=np.float64)
    mse = np.zeros(n, dtype=np.float64)
    psnr = np.zeros(n, dtype=np.float64)
    for i, (s, h) in enumerate(zip(sr_u8, hr_u8)):
        gs, gh = to_gray01(s), to_gray01(h)
        for j, ws in enumerate(window_sizes):
            ssim[i, j] = ssim_box(gh, gs, ws)
        mse[i] = mse01(s, h)
        psnr[i] = psnr01(h, s)
    return ssim, mse, psnr


def aucs_from_scores(y_true, ssim, mse, psnr, window_sizes) -> Tuple[int, float, float, float]:
    """Best-ws selection and the three AUCs exactly as src/evaluate.py:238-265 (strict '>' keeps the
    first window size on ties)."""
    best_ws, best_auc, best_j = window_sizes[0], -1.0, 0
    for j, ws in enumerate(window_sizes):
        a = roc_auc(y_true, 1.0 - ssim[:, j])
        if a > best_auc:
            best_auc, best_ws, best_j = a, ws, j
    auc_ssim = roc_auc(y_true, 1.0 - ssim[:, best_j])
    auc_mse = roc_auc(y_true, mse)
    auc_psnr = roc_auc(y_true, -psnr)
    return best_ws, auc_ssim, auc_mse, auc_psnr


def synthetic_dataset(n_images: int, hr: int = 128, nc: int = 3, scale: int = 4, seed: int = 1234):
    """MVTec-shaped synthetic pairs (SURVEY.md section 8d): low-pass texture; the 'bad' half gets a 16-32 px
    constant square.  Returns HR uint8 [n, hr, hr, nc], LR uint8 [n, hr/s, hr/s, nc] (PIL LANCZOS as
    scripts/prepare_mvtec_data.py:30-33) and labels (good=0 first, then bad=1)."""
    from PIL import Image

    rng = np.random.default_rng(seed)
    n_good = n_images // 2
    hrs, lrs, labels = [], [], []
    for i in range(n_images):
        noise = rng.random((hr + 4, hr + 4, nc))
        c = np.zeros((hr + 5, hr + 5, nc))
        c[1:, 1:] = noise.cumsum(0).cumsum(1)
        blur = (c[5:, 5:] - c[:-5, 5:] - c[5:, :-5] + c[:-5, :-5]) / 25.0
        blur = (blur - blur.min()) / max(blur.max() - blur.min(), 1e-9)
        img = (blur * 255.0).astype(np.uint8)
        label = 0 if i < n_good else 1
        if label:
            sz = int(rng.integers(16, 33))
            y0, x0 = int(rng.integers(0, hr - sz)), int(rng.integers(0, hr - sz))
            img[y0:y0 + sz, x0:x0 + sz] = 255 if rng.random() < 0.5 else 0
        pil = Image.fromarray(img if nc == 3 else img[:, :, 0])
        lr = np.asarray(pil.resize((hr // scale, hr // scale), Image.LANCZOS))
        if nc == 1:
            lr = lr[:, :, None]
        hrs.append(img)
        lrs.append(lr)
        labels.append(label)
    return np.stack(hrs), np.stack(lrs), np.asarray(labels)


# ---------------------------------------------------------------------------------------------------------------------
# validation loop of the training script: Trainer.test (src/trainer.py:242-304)
# ---------------------------------------------------------------------------------------------------------------------
def quantize_round(img: np.ndarray, rgb_range: float) -> np.ndarray:
    """`quantize` (src/trainer.py:45-47): img.mul(255 / rgb_range).clamp(0, 255).round().div(255 / rgb_range), fp32, round half to even."""
    pr = np.float32(255.0 / rgb_range)
    return (np.rint(np.clip(img.astype(np.float32) * pr, 0, 255)).astype(np.float32) / pr).astype(np.float32)


def psnr_torch_np(sr: np.ndarray, hr: np.ndarray, rgb_range: float) -> float:
    """`psnr_torch` (src/metrics.py:70-79) on [1, C, H, W] arrays: shave 4, no clamp."""
    diff = (sr.astype(np.float32) - hr.astype(np.float32)) / np.float32(rgb_range)
    if sr.shape[-1] > 8:
        diff = diff[..., 4:-4, 4:-4]
    mse = float(np.mean(diff.astype(np.float64) ** 2))
    return float("inf") if mse == 0 else 10.0 * float(np.log10(1.0 / mse))


def ssim_torch_np(sr: np.ndarray, hr: np.ndarray, rgb_range: float, win_size: int = 11) -> float:
    """`ssim_torch` (src/metrics.py:82-108) on [1, C, H, W] arrays: / rgb_range, clamp [0, 1], shave 4, gray for 3 channels, ZERO-padded
    win_size box filter (F.conv2d padding), C1 / C2 scaled by 255^2 (the reference's quirk), mean of the map."""
    a = np.clip(sr.astype(np.float32) / np.float32(rgb_range), 0, 1)
    b = np.clip(hr.astype(np.float32) / np.float32(rgb_range), 0, 1)
    if a.shape[-1] > 8:
        a, b = a[..., 4:-4, 4:-4], b[..., 4:-4, 4:-4]
    if a.shape[1] > 1:
        cv = (np.array([65.738, 129.057, 25.064], dtype=np.float32) / np.float32(256)).reshape(1, 3, 1, 1)
        a, b = (a * cv).sum(1, keepdims=True), (b * cv).sum(1, keepdims=True)
    a, b = a[0, 0].astype(np.float64), b[0, 0].astype(np.float64)
    c1, c2 = 0.01 ** 2 * 255.0 ** 2, 0.03 ** 2 * 255.0 ** 2
    h = win_size // 2

    def box(x):
        xp = np.pad(x, h, mode="constant")
        c = np.zeros((xp.shape[0] + 1, xp.shape[1] + 1))
        c[1:, 1:] = xp.cumsum(0).cumsum(1)
        n0, n1 = x.shape
        return (c[win_size:win_size + n0, win_size:win_size + n1] - c[:n0, win_size:win_size + n1] - c[win_size:win_size + n0, :n1] +
                c[:n0, :n1]) / (win_size * win_size)

    mu1, mu2 = box(a), box(b)
    s1, s2, s12 = box(a * a) - mu1 * mu1, box(b * b) - mu2 * mu2, box(a * b) - mu1 * mu2
    m = ((2 * mu1 * mu2 + c1) * (2 * s12 + c2)) / ((mu1 * mu1 + mu2 * mu2 + c1) * (s1 + s2 + c2))
    return float(m.mean())


def validate_pairs(sr: np.ndarray, hr: np.ndarray, rgb_range: float):
    """Body of Trainer.test over a set of [n, C, H, W] pairs, one image at a time (the loader's batch size is 1):
    -> (per-image psnr, per-image ssim, eval_psnr, eval_ssim) with eval_* = sum / len(loader_test)."""
    ps, ss = [], []
    for i in range(sr.shape[0]):
        q = quantize_round(sr[i:i + 1], rgb_range)
        ps.append(psnr_torch_np(q, hr[i:i + 1], rgb_range))
        ss.append(ssim_torch_np(q, hr[i:i + 1], rgb_range))
    return np.asarray(ps), np.asarray(ss), float(sum(ps) / len(ps)), float(sum(ss) / len(ss))

