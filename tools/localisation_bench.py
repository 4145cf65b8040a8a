"""Device time of the localisation metrics (pixel AUROC, AU-PRO, pixel AP and F1-max of one anomaly map over a whole test set,
csrc/localisation.cu) on synthetic maps and masks: random rectangles and round blobs as defects, smoothed noise with raised scores on the defects as the map.

Per repetition (CUDA events): the append of one map (device copy of every batch into the accumulator's buffer) and the finish (the
sixteen kernels of adsr_localisation_metrics).  The default 1024 images of 256 x 256 are 67 M pixels per map: the sort's 16 bytes of
pairs per pixel are far above the 126 MB of L2.  --host also times the host path of the same inputs (sklearn's roc_auc_score behind
metrics.pixel_auroc on host arrays, the oracle's AU-PRO, sklearn's average_precision_score, the oracle's F1-max) and reports the
agreement.  One JSON line, with the card and its power limit.

It also times, on the same map, the two passes that need no sort: the exact score quantile (adsr_score_quantile, a radix select
reading ~16 B per pixel) at --quantile, and the pixel counts + PRO at that score (adsr_threshold_metrics, one pass over the 8 B of
score and region index per pixel).  --host adds np.quantile(method="inverted_cdf") and the oracle's counts, and their agreement.

    python tools/localisation_bench.py [--images 1024] [--side 256] [--reps 20] [--quantile 0.999] [--host]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "anomaly-detection-super-resolution_b200"


def synthetic(n, side, seed):
    """uint8 masks [n, side, side] (a third of the images defect-free) and fp32 maps, generated on the device from a seed."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    rng = np.random.default_rng(seed)
    masks = np.zeros((n, side, side), np.uint8)
    yy, xx = np.mgrid[:side, :side]
    for i in range(n):
        if i % 3 == 0:
            continue
        for _ in range(rng.integers(1, 4)):
            y, x = rng.integers(0, side, 2)
            masks[i, y:y + rng.integers(2, side // 6), x:x + rng.integers(2, side // 6)] = 1
        cy, cx, r = rng.integers(0, side), rng.integers(0, side), rng.integers(3, side // 10)
        masks[i][(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = 1
    noise = torch.rand(n, 1, side, side, generator=g, device="cuda")
    k = torch.ones(1, 1, 5, 5, device="cuda") / 25.0
    smooth = torch.nn.functional.conv2d(noise, k, padding=2)[:, 0]
    maps = (smooth + 0.15 * torch.from_numpy(masks).cuda().float()).contiguous()
    return maps, masks


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = float(q.stdout.strip().splitlines()[0])
    except Exception:                                       # nvidia-smi missing or unreadable: the number stays unreported
        power = None
    return name, power


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--side", type=int, default=256)
    ap.add_argument("--batch", type=int, default=64, help="images per append")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--fpr-limit", type=float, default=0.3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--quantile", type=float, default=0.999, help="q of the timed quantile; its score is the timed threshold")
    ap.add_argument("--host", action="store_true", help="also time the host path on the same inputs and report the agreement")
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("localisation_bench needs a CUDA device")
    metrics = importlib.import_module(PKG + ".metrics")
    ops = importlib.import_module(PKG + ".ops")

    maps, masks = synthetic(a.images, a.side, a.seed)
    acc = metrics.LocalisationAccumulator(1)
    for s in range(0, a.images, a.batch):                   # host labelling + region upload happen here, once
        acc.append([maps[s:s + a.batch]], masks[s:s + a.batch])
    r, = acc.results(a.fpr_limit)
    auroc, aupro = r.pixel_auroc, r.au_pro
    n = acc.n
    buf, regions = acc._maps[0], acc._regions[:n]
    sizes = torch.from_numpy(np.concatenate(acc._sizes)).cuda()
    ws = torch.empty(ops.localisation_workspace_bytes(n), dtype=torch.uint8, device="cuda")
    out = torch.empty(8, dtype=torch.float64, device="cuda")

    def one():                                              # the device work of append (per-batch copies) + finish, one map
        off = 0
        for s in range(0, a.images, a.batch):
            m = maps[s:s + a.batch]
            buf[off:off + m.numel()].copy_(m.reshape(-1))
            off += m.numel()
        ops.localisation_metrics(buf[:n], regions, sizes, acc.n_ok, a.fpr_limit, ws, out)

    for _ in range(a.warmup):
        one()
    times = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        one()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    again = out.cpu().numpy()

    def timed(fn):                                          # median device ms of fn over the repetitions, after the warm-ups
        for _ in range(a.warmup):
            fn()
        ts = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts)

    k = metrics.inverted_cdf_rank(n, a.quantile)
    q_out, t_out = torch.empty(2, dtype=torch.float64, device="cuda"), torch.empty(7, dtype=torch.float64, device="cuda")
    q_ms = timed(lambda: ops.score_quantile(buf[:n], k, ws, q_out))
    t_q = float(q_out[0])
    thr_ms = timed(lambda: ops.threshold_metrics(buf[:n], regions, sizes, t_q, ws, t_out))
    th = acc.at_threshold(0, t_q)
    name, power = card()
    res = dict(tool="localisation_bench", gpu=name, power_limit_w=power, images=a.images, side=a.side, pixels_per_map=n,
               regions=acc.n_regions, fpr_limit=a.fpr_limit, reps=a.reps, device_ms_per_map_median=statistics.median(times),
               device_ms_per_map_min=min(times), device_ms_per_map_max=max(times), pixel_auroc=auroc, au_pro=aupro,
               pixel_ap=r.pixel_ap, f1_max=r.f1_max, f1_threshold=r.f1_threshold,
               repeat_bitwise_equal=bool(tuple(float(again[k]) for k in (0, 1, 5, 6, 7)) == tuple(r)),
               bytes_per_pixel_floor=80, floor_ms_at_7_7_tbps=n * 80 / 7.7e12 * 1e3,
               quantile=a.quantile, quantile_score=t_q, quantile_device_ms_median=q_ms, quantile_floor_ms_at_7_7_tbps=n * 16 / 7.7e12 * 1e3,
               quantile_equals_accumulator=t_q == acc.quantile(0, a.quantile),
               threshold_device_ms_median=thr_ms, threshold_floor_ms_at_7_7_tbps=n * 8 / 7.7e12 * 1e3,
               threshold_counts=[th.tp, th.fp, th.fn, th.tn], threshold_pro=th.pro)
    if a.host:
        from oracle import localisation_oracle as L
        from oracle import pr_oracle as P

        h_maps = maps.cpu().numpy()
        t0 = time.perf_counter()
        h_auc = metrics.pixel_auroc(h_maps, masks)
        res["host_pixel_auroc_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        h_pro = L.au_pro(list(h_maps), list(masks), a.fpr_limit)
        res["host_au_pro_oracle_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        h_ap = P.pixel_ap(list(h_maps), list(masks))
        res["host_pixel_ap_sklearn_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        h_f1, h_thr = P.f1_max(list(h_maps), list(masks))
        res["host_f1_max_oracle_s"] = time.perf_counter() - t0
        res["abs_diff_pixel_auroc"] = abs(h_auc - auroc)
        res["abs_diff_au_pro"] = abs(h_pro - aupro)
        res["abs_diff_pixel_ap"] = abs(h_ap - r.pixel_ap)
        res["abs_diff_f1_max"] = abs(h_f1 - r.f1_max)
        res["f1_threshold_equal"] = h_thr == r.f1_threshold
        from oracle import threshold_oracle as T

        t0 = time.perf_counter()
        h_q = T.quantile(list(h_maps), a.quantile)
        res["host_quantile_numpy_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        h_counts = T.counts(list(h_maps), list(masks), t_q)
        res["host_threshold_oracle_s"] = time.perf_counter() - t0
        res["quantile_equal"] = h_q == t_q
        res["threshold_counts_equal"] = list(h_counts[:4]) == [th.tp, th.fp, th.fn, th.tn]
        res["abs_diff_threshold_pro"] = abs(h_counts[4] - th.pro)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
