"""Timing of the anomaly maps (ops.anomaly_maps: 1 - SSIM map of one window size + squared-error map, optional Gaussian smoothing,
per-image max) next to the scorer's full window sweep (ops.score_images) on the same uint8 SR / HR batches, with CUDA events.

    python tools/anomaly_map_bench.py [--launches 50] [--warmup 5]

Shapes are the evaluator's: B = 256 at 128 x 128 x 3 and B = 128 at 256 x 256 x 3 (the 64 px LR configuration), window size 11,
sigma 0 and 4.  Each figure is the mean time per call over `--launches` back-to-back calls after `--warmup` calls.  The inputs stay
resident in L2 between calls, as they are in the evaluator, which scores the SR batch its last kernel just wrote.  Prints one JSON
line that includes the device name and its power limit."""
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
        for sigma in (0.0, 4.0):
            ms = time_ms(lambda: ops.anomaly_maps(sr, hr, args.window_size, sigma, out=out), args.launches, args.warmup)
            cases.append(dict(batch=b, shape=[side, side, 3], window_size=args.window_size, sigma=sigma, maps_ms=round(ms, 4),
                              score_images_ms=round(score_ms, 4), score_images_windows=len(wss),
                              maps_over_score=round(ms / score_ms, 3), maps_faster=ms < score_ms))
    print(json.dumps(dict(tool="anomaly_map_bench", device=torch.cuda.get_device_name(), power_limit_w=power_limit_w(),
                          launches=args.launches, warmup=args.warmup, inputs="L2-resident between calls", cases=cases)))


if __name__ == "__main__":
    main()
