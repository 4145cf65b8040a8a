"""Timing of the anomaly maps (ops.anomaly_maps: 1 - SSIM map of one window size + squared-error map, optional Gaussian smoothing,
per-image max) and of the MSGMS map (ops.gms_map) next to the scorer's full window sweep (ops.score_images) on the same uint8 SR / HR
batches, with CUDA events.

    python tools/anomaly_map_bench.py [--launches 50] [--warmup 5]

Shapes are the evaluator's: B = 256 at 128 x 128 x 3 and B = 128 at 256 x 256 x 3 (the 64 px LR configuration), window size 11,
sigma 0 and 4.  Each figure is the mean time per call over `--launches` back-to-back calls after `--warmup` calls.  The inputs stay
resident in L2 between calls, as they are in the evaluator, which scores the SR batch its last kernel just wrote.  For the MSGMS map
`gms_bytes` counts the bytes its kernels read and write per call (gms_bytes_moved) and `gms_tb_s` / `gms_of_7_7_tb_s` the resulting
rate against the B200's 7.7 TB/s HBM bandwidth; much of that traffic is served by the 126 MB L2, so the fraction is an effective
rate, not an HBM measurement.  Prints one JSON line that includes the device name and its power limit."""
import argparse
import importlib
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PKG = "anomaly-detection-super-resolution_b200"


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


HBM_BYTES_PER_S = 7.7e12


def gms_bytes_moved(b, h, w, c, sigma):
    """Bytes the MSGMS kernels read and write per call, each plane access counted once: the uint8 pair in, both gray pyramids out
    (level 0 plus the 2 x 2-mean levels), the coarse levels read back and their 1 - GMS planes written, the level-0 gray planes and the
    1 - GMS planes read by the combine pass and the map written, the Gaussian's two passes over map and scratch, the max pass."""
    px = h * w
    coarse = sum((h >> k) * (w >> k) for k in range(1, 4))
    per_image = (2 * c * px + 4 * 2 * (px + coarse)          # pyramid
                 + 4 * 2 * coarse + 4 * coarse                 # levels 1-3
                 + 4 * 2 * px + 4 * coarse + 4 * px            # combine
                 + (4 * 4 * px if sigma > 0 else 0)            # Gaussian rows + columns
                 + 4 * px + 8)                                 # max
    return b * per_image


def time_ms(fn, launches, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches


def main():
    p = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    p.add_argument("--launches", type=int, default=50)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--window-size", type=int, default=11)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("anomaly_map_bench needs a CUDA device")
    ops = importlib.import_module(PKG + ".ops")
    metrics = importlib.import_module(PKG + ".metrics")
    g = torch.Generator(device="cuda").manual_seed(0)
    cases = []
    for b, side in ((256, 128), (128, 256)):
        hr = torch.randint(0, 256, (b, side, side, 3), generator=g, device="cuda", dtype=torch.uint8)
        noise = torch.randint(-8, 9, hr.shape, generator=g, device="cuda", dtype=torch.int16)
        sr = (hr.to(torch.int16) + noise).clamp(0, 255).to(torch.uint8)
        wss = metrics.window_sizes_for(side)
        f32 = dict(dtype=torch.float32, device="cuda")
        out = (torch.empty(b, side, side, **f32), torch.empty(b, side, side, **f32), torch.empty(b, 2, dtype=torch.float64, device="cuda"),
               torch.empty(b, side, side, **f32))
        scores = torch.empty(b, len(wss) + 2, dtype=torch.float64, device="cuda")
        score_ms = time_ms(lambda: ops.score_images(sr, hr, wss, scores), args.launches, args.warmup)
        gms_out = (torch.empty(b, side, side, **f32), torch.empty(b, dtype=torch.float64, device="cuda"),
                   torch.empty(ops.gms_workspace_bytes(b, side, side), dtype=torch.uint8, device="cuda"))
        for sigma in (0.0, 4.0):
            ms = time_ms(lambda: ops.anomaly_maps(sr, hr, args.window_size, sigma, out=out), args.launches, args.warmup)
            gms_ms = time_ms(lambda: ops.gms_map(sr, hr, sigma, out=gms_out), args.launches, args.warmup)
            nbytes = gms_bytes_moved(b, side, side, 3, sigma)
            cases.append(dict(batch=b, shape=[side, side, 3], window_size=args.window_size, sigma=sigma, maps_ms=round(ms, 4),
                              gms_ms=round(gms_ms, 4), score_images_ms=round(score_ms, 4), score_images_windows=len(wss),
                              maps_over_score=round(ms / score_ms, 3), maps_faster=ms < score_ms, gms_over_maps=round(gms_ms / ms, 3),
                              gms_bytes=nbytes, gms_tb_s=round(nbytes / (gms_ms * 1e-3) / 1e12, 3),
                              gms_of_7_7_tb_s=round(nbytes / (gms_ms * 1e-3) / HBM_BYTES_PER_S, 3)))
    print(json.dumps(dict(tool="anomaly_map_bench", device=torch.cuda.get_device_name(), power_limit_w=power_limit_w(),
                          launches=args.launches, warmup=args.warmup, inputs="L2-resident between calls", cases=cases)))


if __name__ == "__main__":
    main()
