"""Timing of the defect-region kernels (ops.label_regions, ops.region_stats: csrc/regions.cu) with CUDA events, next to the host
reference (scipy.ndimage.label + find_objects + the numpy statistics of oracle/region_oracle.py) on the same maps.

    python tools/region_bench.py [--cases 1024x256,256x128] [--calls 20] [--warmup 3] [--host-images 64]

A case BxS is B uniform random fp32 maps of S x S, thresholded at three foreground densities: sparse (0.1 % of the pixels), dense (70 %)
and 0.41, near the site-percolation point of 8-connectivity (0.407), where one component spans most 32 x 32 tiles of an image.  Each
GPU figure is the median over `--calls` calls after `--warmup` calls, each call timed alone with a pair of CUDA events: label = the
seven labelling kernels (and the two memsets), stats = table initialisation and the statistics pass (the region counts are read once,
outside the timing, to size the table).  The maps (1 GiB at 1024 x 256^2) do not fit the 126 MB L2.  The host figure times the
reference on the first `--host-images` images of the case (single thread) and is scaled to B.  Prints one JSON line with the device name
and its power limit."""
import argparse
import importlib
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from anomaly_map_bench import PKG, power_limit_w  # noqa: E402
from oracle import region_oracle as R  # noqa: E402

DENSITIES = (("sparse", 0.001), ("percolation", 0.41), ("dense", 0.7))


def median_ms(fn, calls, warmup):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return statistics.median(times)


def main():
    p = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    p.add_argument("--cases", default="1024x256,256x128")
    p.add_argument("--calls", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--host-images", type=int, default=64)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("region_bench needs a CUDA device")
    ops = importlib.import_module(PKG + ".ops")
    g = torch.Generator(device="cuda").manual_seed(0)
    cases = []
    for spec in args.cases.split(","):
        b, side = (int(v) for v in spec.split("x"))
        maps = torch.rand(b, side, side, generator=g, device="cuda")
        ws = torch.empty(ops.regions_workspace_bytes(b, side, side), dtype=torch.uint8, device="cuda")
        labels = torch.empty(b, side, side, dtype=torch.int32, device="cuda")
        counts = torch.empty(b, dtype=torch.int32, device="cuda")
        host_n = min(b, args.host_images)
        host_maps = maps[:host_n].cpu().numpy()
        for name, density in DENSITIES:
            t = float(np.float32(1.0 - density))
            label = lambda: ops.label_regions(maps, t, None, 1, ws, labels, counts)
            label_ms = median_ms(label, args.calls, args.warmup)
            label()
            n = counts.cpu().numpy().astype(np.int64)
            assert int(ws[:4].view(torch.int32).item()) == 0
            offsets = torch.from_numpy(np.concatenate([[0], np.cumsum(n)])).cuda()
            table = torch.empty(int(n.sum()), 9, dtype=torch.int64, device="cuda")
            stats_ms = median_ms(lambda: ops.region_stats(labels, maps, None, offsets, None, ws, table), args.calls, args.warmup)
            t0 = time.perf_counter()
            for i in range(host_n):
                lab, k = R.label_image(R.foreground(host_maps[i], t))
                R.region_rows(lab, k, i, host_maps[i])
            host_ms = (time.perf_counter() - t0) * 1e3 * b / host_n
            cases.append(dict(batch=b, side=side, density=name, foreground=round(density, 4), regions=int(n.sum()),
                              largest_region=int(torch.bincount(labels[0].reshape(-1))[1:].max().item()) if n[0] else 0,
                              label_ms=round(label_ms, 3), stats_ms=round(stats_ms, 3), gpu_ms=round(label_ms + stats_ms, 3),
                              host_ms_scaled=round(host_ms, 1), host_images_timed=host_n,
                              speedup=round(host_ms / (label_ms + stats_ms), 1)))
    print(json.dumps(dict(tool="region_bench", device=torch.cuda.get_device_name(), power_limit_w=power_limit_w(), calls=args.calls,
                          warmup=args.warmup, statistic="median per call", cases=cases)))


if __name__ == "__main__":
    main()
