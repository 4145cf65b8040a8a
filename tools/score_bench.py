"""Timing of the scorer (ops.score_images: the evaluator's full SSIM window sweep, MSE and PSNR of uint8 SR / HR batches) with CUDA
events, at the batch sizes that pick its different kernels.

    python tools/score_bench.py [--cases 64x128,256x128,128x256] [--launches 50] [--warmup 5]
    python tools/score_bench.py --libs build/libadsr_base.so,in-tree [--rounds 3]     # A/B of two builds

A case BxS is B images of S x S x 3 with metrics.window_sizes_for(S) (13 window sizes at 128 px, 26 at 256 px).  On a 148-SM B200,
64 images at 128 px run score_images_fast4_kernel, 256 run score_images_fast_kernel and 256 px images run score_images_kernel.  Each
figure is the mean time per call over `--launches` back-to-back calls after `--warmup` calls, with the inputs resident in L2 as they
are in the evaluator.  ADSR_LIB=<path> times another build of the library (tools/build_variant.sh).  --libs times several builds
(`in-tree` = this tree's library) in alternation, one process per build and round, so that drift of the shared machine falls on
all of them alike, and reports each build's median per case over the rounds.  Prints one JSON line that includes the device name
and its power limit."""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from anomaly_map_bench import PKG, power_limit_w, time_ms  # noqa: E402


def main():
    p = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    p.add_argument("--cases", default="64x128,256x128,128x256")
    p.add_argument("--launches", type=int, default=50)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--libs", default=None, help="comma-separated library paths (or in-tree) to time in alternation")
    p.add_argument("--rounds", type=int, default=3, help="with --libs: rounds of one run per build")
    args = p.parse_args()
    if args.libs:
        return alternate(args)
    if not torch.cuda.is_available():
        raise SystemExit("score_bench needs a CUDA device")
    ops = importlib.import_module(PKG + ".ops")
    metrics = importlib.import_module(PKG + ".metrics")
    g = torch.Generator(device="cuda").manual_seed(0)
    cases = []
    for spec in args.cases.split(","):
        b, side = (int(v) for v in spec.split("x"))
        hr = torch.randint(0, 256, (b, side, side, 3), generator=g, device="cuda", dtype=torch.uint8)
        noise = torch.randint(-8, 9, hr.shape, generator=g, device="cuda", dtype=torch.int16)
        sr = (hr.to(torch.int16) + noise).clamp(0, 255).to(torch.uint8)
        wss = metrics.window_sizes_for(side)
        scores = torch.empty(b, len(wss) + 2, dtype=torch.float64, device="cuda")
        ms = time_ms(lambda: ops.score_images(sr, hr, wss, scores), args.launches, args.warmup)
        cases.append(dict(batch=b, shape=[side, side, 3], windows=len(wss), score_images_ms=round(ms, 4),
                          us_per_image=round(ms * 1e3 / b, 3)))
    print(json.dumps(dict(tool="score_bench", lib=os.environ.get("ADSR_LIB", "in-tree"), device=torch.cuda.get_device_name(),
                          power_limit_w=power_limit_w(), launches=args.launches, warmup=args.warmup,
                          inputs="L2-resident between calls", cases=cases)))


def alternate(args):
    libs = args.libs.split(",")
    runs = {lib: [] for lib in libs}
    for _ in range(args.rounds):
        for lib in libs:
            env = dict(os.environ)
            env.pop("ADSR_LIB", None)
            if lib != "in-tree":
                env["ADSR_LIB"] = os.path.abspath(lib)
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--cases", args.cases, "--launches", str(args.launches),
                                  "--warmup", str(args.warmup)], env=env, capture_output=True, text=True, check=True).stdout
            runs[lib].append(json.loads(out.strip().splitlines()[-1]))
    first = runs[libs[0]][0]
    summary = []
    for k, case in enumerate(first["cases"]):
        summary.append(dict(batch=case["batch"], shape=case["shape"], windows=case["windows"],
                            median_ms={lib: round(statistics.median(r["cases"][k]["score_images_ms"] for r in runs[lib]), 4)
                                       for lib in libs},
                            all_ms={lib: [r["cases"][k]["score_images_ms"] for r in runs[lib]] for lib in libs}))
    print(json.dumps(dict(tool="score_bench", device=first["device"], power_limit_w=first["power_limit_w"], launches=args.launches,
                          warmup=args.warmup, rounds=args.rounds, inputs="L2-resident between calls", cases=summary)))


if __name__ == "__main__":
    main()
