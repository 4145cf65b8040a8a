"""numpy fp64 reference of the multi-scale gradient-magnitude-similarity (MSGMS) anomaly map (csrc/anomaly_maps.cu adsr_gms_map).

RIAD (Zavrtanik, Kristan, Skocaj, "Reconstruction by inpainting for visual anomaly detection", Pattern Recognition 2021) scores a
reconstruction with the MSGMS of GMSD (Xue et al., IEEE TIP 2014).  Per uint8 HWC SR / HR pair:
  1. gray planes x (HR) and y (SR) in [0, 1] as the 1 - SSIM map builds them (scoring_oracle.to_gray01; RIAD averages the channels);
  2. 4 pyramid levels, level k + 1 = the 2 x 2 means of level k with odd sizes floored (avg_pool2d(2, 2));
  3. Prewitt correlation at each level with zero padding, g = sqrt(gx^2 + gy^2 + 1e-12);
  4. gms = (2 g_x g_y + c) / (g_x^2 + g_y^2 + c), c = 0.0026 (GMSD's T = 170 on the 0-255 scale);
  5. map = (1/4) sum_k up_k(1 - gms_k), up_k the bilinear resize to H x W with align_corners=False, summed in level order;
  6. sigma > 0: scipy.ndimage.gaussian_filter(map, sigma, mode="reflect", truncate=4.0) (RIAD uses a 21 x 21 mean filter).
Written without torch: explicit zero-padded correlation, floor pooling and align_corners=False weights."""
from __future__ import annotations

import numpy as np

from . import scoring_oracle as S

LEVELS = 4
C = 0.0026
PREWITT_X = np.array([[1.0, 0.0, -1.0]] * 3) / 3.0      # correlation kernel of gx; gy uses its transpose


def pool2(p: np.ndarray) -> np.ndarray:
    """2 x 2 means with stride 2 of an [h, w] plane; an odd last row / column is dropped."""
    h, w = p.shape[0] // 2, p.shape[1] // 2
    q = p[:2 * h, :2 * w]
    return (q[0::2, 0::2] + q[0::2, 1::2] + q[1::2, 0::2] + q[1::2, 1::2]) / 4.0


def correlate3_zero(p: np.ndarray, k: np.ndarray) -> np.ndarray:
    """out[i, j] = sum_{a, b} k[a, b] p[i + a - 1, j + b - 1], zero outside the plane (F.conv2d(..., padding=1))."""
    h, w = p.shape
    q = np.zeros((h + 2, w + 2))
    q[1:-1, 1:-1] = p
    out = np.zeros((h, w))
    for a in range(3):
        for b in range(3):
            out += k[a, b] * q[a:a + h, b:b + w]
    return out


def gradient_magnitude(p: np.ndarray) -> np.ndarray:
    gx = correlate3_zero(p, PREWITT_X)
    gy = correlate3_zero(p, PREWITT_X.T)
    return np.sqrt(gx * gx + gy * gy + 1e-12)


def bilinear_weights(n_in: int, n_out: int):
    """align_corners=False source indices and weights of one axis: out[o] = l0[o] in[i0[o]] + l1[o] in[i1[o]]."""
    src = np.maximum((np.arange(n_out) + 0.5) * (n_in / n_out) - 0.5, 0.0)
    i0 = np.floor(src).astype(np.int64)
    i1 = np.where(i0 < n_in - 1, i0 + 1, i0)
    l1 = src - i0
    return i0, i1, 1.0 - l1, l1


def upsample_bilinear(p: np.ndarray, h: int, w: int) -> np.ndarray:
    r0, r1, a0, a1 = bilinear_weights(p.shape[0], h)
    c0, c1, b0, b1 = bilinear_weights(p.shape[1], w)
    top = p[r0][:, c0] * b0 + p[r0][:, c1] * b1
    bot = p[r1][:, c0] * b0 + p[r1][:, c1] * b1
    return a0[:, None] * top + a1[:, None] * bot


def level_maps(sr_u8: np.ndarray, hr_u8: np.ndarray) -> list:
    """The 1 - GMS plane of every pyramid level (level k is (H >> k) x (W >> k)), fp64."""
    x = S.to_gray01(hr_u8).astype(np.float64)
    y = S.to_gray01(sr_u8).astype(np.float64)
    out = []
    for k in range(LEVELS):
        if k:
            x, y = pool2(x), pool2(y)
        gx, gy = gradient_magnitude(x), gradient_magnitude(y)
        out.append(1.0 - (2.0 * gx * gy + C) / (gx * gx + gy * gy + C))
    return out


def gms_map(sr_u8: np.ndarray, hr_u8: np.ndarray, sigma: float = 0.0) -> np.ndarray:
    """One uint8 HWC pair (H, W >= 8; C = 1 or 3) -> the MSGMS map, fp64 [H, W]."""
    h, w = hr_u8.shape[:2]
    acc = np.zeros((h, w))
    for d in level_maps(sr_u8, hr_u8):
        acc = acc + upsample_bilinear(d, h, w)
    m = acc / LEVELS
    if sigma > 0:
        from scipy.ndimage import gaussian_filter

        m = gaussian_filter(m, sigma, mode="reflect", truncate=4.0)
    return m
