#!/usr/bin/env python
"""Headline benchmark: DRCT-L x4, 32 px LR -> 128 px HR, RGB, batch 256 per GPU, inference + anomaly scoring
(BASELINE.json configs[2], the configuration the metric is quoted on).

  python bench.py --gpus N --steps K --warmup W            # this repo (torchrun launches N ranks for N > 1)
  python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm's CPU path (oracle port)
  python bench.py --steps K --dump-outputs DIR              # + each workload's last timed step as DIR/*.npy (seeded inputs:
                                                            #   two builds can be compared array for array)

A "step" = one pass of the hot path over one batch: HR uint8 truncation, DRCT forward (uint8 truncation fused into
the last kernel), one scoring launch (13 SSIM window sizes + MSE + PSNR per image) and, when sharded, the NCCL
all_gather of the per-image score rows.  `value` times it with inputs resident in HBM; `e2e` runs the same step
through the public evaluator API from pinned HOST tensors, with the H2D copies and the D2H read of the score
table inside the timed region.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "anomaly-detection-super-resolution_b200"
METRIC = "DRCT-L x4 128px HR images/sec (inference+scoring)"
DOMINANT_KERNEL_NAMES = {"swin_attn": "swin_attn_kernel", "swin_mlp": "swin_mlp_kernel", "tc_gemm": "tc_gemm_rows_kernel",
                         "window_attention": "window_attn_tc_kernel", "conv3x3": "tc_gemm_manual_kernel", "conv3x3_halo": "conv_halo_kernel"}
HR, SCALE, NC = 128, 4, 3


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--batch", type=int, default=None, help="images per GPU per step (default 256 DRCT-L, 64 DRN-L)")
    p.add_argument("--workload", default="drct-l", choices=["drct-l", "drn-l", "drct-l-64"],
                   help="drct-l = BASELINE configs[2] (headline); drn-l = configs[1]; drct-l-64 = configs[3] (64 px LR, 16 x 16 windows)")
    p.add_argument("--no-sub-workloads", action="store_true", help="skip the sub-records of the other BASELINE configs")
    p.add_argument("--cpu-sample", type=int, default=4, help="images per CPU-baseline step")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write each workload's results of its last timed step to DIR/<workload>_<array>.npy")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def synthetic_pairs(n: int, seed: int = 1234, hr: int = 128):
    """MVTec-shaped synthetic pairs (SURVEY.md 8d): low-pass texture, the second half ('bad') gets a 16-32 px constant
    square; LR = PIL LANCZOS / 4 of HR (scripts/prepare_mvtec_data.py:30-33).  -> HR u8 [n,128,128,3], LR u8, labels."""
    from PIL import Image

    HR = hr
    rng = np.random.default_rng(seed)
    hrs, lrs, labels = [], [], []
    for i in range(n):
        noise = rng.random((HR + 4, HR + 4, NC))
        c = np.zeros((HR + 5, HR + 5, NC))
        c[1:, 1:] = noise.cumsum(0).cumsum(1)
        blur = (c[5:, 5:] - c[:-5, 5:] - c[5:, :-5] + c[:-5, :-5]) / 25.0
        blur = (blur - blur.min()) / max(blur.max() - blur.min(), 1e-9)
        img = (blur * 255.0).astype(np.uint8)
        label = 0 if i < n // 2 else 1
        if label:
            sz = int(rng.integers(16, 33))
            y0, x0 = int(rng.integers(0, HR - sz)), int(rng.integers(0, HR - sz))
            img[y0:y0 + sz, x0:x0 + sz] = 255 if rng.random() < 0.5 else 0
        lr = np.asarray(Image.fromarray(img).resize((HR // SCALE, HR // SCALE), Image.LANCZOS))
        hrs.append(img)
        lrs.append(lr)
        labels.append(label)
    return np.stack(hrs), np.stack(lrs), np.asarray(labels)


def to_float_nchw(u8_nhwc: np.ndarray, rgb_range: float = 255.0) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(u8_nhwc.transpose(0, 3, 1, 2))).float().mul_(rgb_range / 255)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          "200", "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return {"burst": d["bf16_tflops"], "sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "hbm": d["hbm_gbs"],
                "source": "measured"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "source": "fallback"}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs.  The reference is pure Python / PyTorch; its own setup.py installs no modules (find_packages on a flat module
# directory), so `pip install --target baseline/_ref` leaves only metadata there.  When a tree with src/drct.py IS present under
# baseline/_ref (e.g. placed there by the driver) the unmodified reference is timed through oracle/ref_shim.py
# (kind "reference"); otherwise the oracle port of the same algorithm is (kind "port").
# ---------------------------------------------------------------------------------------------------------------------
REF_ROOT = os.environ.get("ADSR_BENCH_REF_ROOT", os.path.join(ROOT, "baseline", "_ref"))


def cpu_step(O, S, sd, cfg, lr_f: torch.Tensor, hr_u8: np.ndarray, wss):
    with torch.no_grad():
        sr = O.drct_forward(sd, lr_f, cfg) if hasattr(O, "drct_forward") else O.drn_forward(sd, lr_f, cfg)[-1]
    sr_u8 = S.quantize_u8(sr.numpy(), 255.0)
    return S.score_images(list(sr_u8), list(hr_u8), wss)


def cpu_setup(n: int, workload: str = "drct-l"):
    from oracle import scoring_oracle as S
    if workload == "drct-l":
        from oracle import drct_oracle as O
        cfg = O.DrctCfg()
    else:
        from oracle import drn_oracle as O
        cfg = O.DrnCfg()

    torch.set_num_threads(os.cpu_count() or 1)
    sd = O.make_state_dict(cfg, seed=1)
    hr, lr, _ = synthetic_pairs(n)
    return O, S, sd, cfg, to_float_nchw(lr), hr, S.window_sizes_for(HR)


def reference_setup(n: int, workload: str):
    """The UNMODIFIED reference (src.drct.DRCT / src.drn.DRN in eval mode + src.metrics.ssim_numpy / psnr_numpy) when its tree
    is present under baseline/_ref; returns a step function, or None."""
    if not os.path.isfile(os.path.join(REF_ROOT, "src", "drct.py")):
        return None
    os.environ["ADSR_REFERENCE_ROOT"] = REF_ROOT
    from oracle import ref_shim
    try:
        ref_shim.import_reference()
        rmain, rmetrics = sys.modules["src.main"], sys.modules["src.metrics"]
        torch.set_num_threads(os.cpu_count() or 1)
        torch.manual_seed(1)
        if workload == "drct-l":
            opt = rmain.DRCT()
            opt.img_size, opt.n_colors, opt.window_size, opt.upscale, opt.scale = HR // SCALE, NC, HR // SCALE // 4, SCALE, [SCALE]
            model = sys.modules["src.drct"].DRCT(opt).eval()
        else:
            opt = rmain.DRN()
            opt.n_colors, opt.scale = NC, [2, 4]
            model = sys.modules["src.drn"].DRN(opt).eval()
    except Exception as e:                              # an incomplete tree: fall back to the port
        print(f"[bench] reference under baseline/_ref not usable ({e}); timing the oracle port", file=sys.stderr)
        return None
    hr, lr, _ = synthetic_pairs(n)
    lr_f = to_float_nchw(lr)
    wss = [w for w in range(3, max(3, HR - 3) + 1, 10) if w % 2 == 1]

    def step():
        with torch.no_grad():
            sr = model(lr_f)
        sr = sr[-1] if isinstance(sr, list) else sr
        sr_u8 = sr.mul(1.0).clamp(0, 255).byte().permute(0, 2, 3, 1).numpy()
        for a, b in zip(sr_u8, hr):
            af, bf = a.astype(np.float32) / 255.0, b.astype(np.float32) / 255.0
            for ws in wss:
                rmetrics.ssim_numpy(bf, af, ws)
            rmetrics.psnr_numpy(bf, af)
            float(np.mean((af - bf) ** 2))
    return step


def run_reference_arm(args, rank: int, emit):
    if rank != 0:
        return
    workload = args.workload if args.workload in ("drct-l", "drn-l") else "drct-l"
    drct_wl = workload == "drct-l"
    name = "DRCT-L" if drct_wl else "DRN-L"
    ref_step = reference_setup(1, workload)
    if ref_step is not None:
        n, kind = 1, "reference"
        step = ref_step
        sample = (f"1 image/step x {args.steps} steps: the unmodified reference from baseline/_ref ({name}.eval() fp32 forward, torch CPU, "
                  f"{torch.get_num_threads()} threads, + its ssim_numpy Python loop for the 13 window sizes + psnr_numpy + MSE)")
    else:
        n, kind = args.cpu_sample, "port"
        O, S, sd, cfg, lr_f, hr, wss = cpu_setup(n, workload)
        step = lambda: cpu_step(O, S, sd, cfg, lr_f, hr, wss)
        sample = (f"{n} images/step x {args.steps} steps: oracle {name} fp32 forward (torch CPU, {torch.get_num_threads()} threads) "
                  "+ vectorised box-SSIM sweep/MSE/PSNR (numpy); the reference's own ssim_numpy is a Python "
                  "loop ~100x slower than this port (its setup.py installs no modules, so it cannot travel to this box)")
    for _ in range(max(1, min(args.warmup, 1))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": METRIC if drct_wl else "DRN-L x4 128px HR images/sec (inference+scoring)", "value": value, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": ("configs[2]: DRCT-L" if drct_wl else "configs[1]: DRN-L") + " x4 RGB 32->128 px, inference + scoring",
                   "images_per_step": n},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(json.dumps(line))


def cpu_baseline_record(args) -> dict:
    """Oracle port on a bounded sample (rank 0, N = 1), timed beside the GPU run."""
    workload = args.workload if args.workload in ("drct-l", "drn-l") else "drct-l"
    n = args.cpu_sample
    O, S, sd, cfg, lr_f, hr_np, wss_c = cpu_setup(n, workload)
    cpu_step(O, S, sd, cfg, lr_f, hr_np, wss_c)
    t0 = time.perf_counter()
    reps_c = 3
    for _ in range(reps_c):
        cpu_step(O, S, sd, cfg, lr_f, hr_np, wss_c)
    dtc = time.perf_counter() - t0
    cores = torch.get_num_threads()
    return {"value": n * reps_c / dtc, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{n} images x {reps_c} passes: oracle {'DRCT-L' if workload == 'drct-l' else 'DRN-L'} fp32 forward "
                      f"(torch CPU, {cores} threads) + vectorised SSIM sweep/MSE/PSNR (numpy)"}


# ---------------------------------------------------------------------------------------------------------------------
def _guard_stdout():
    """Everything that libraries print to stdout (e.g. the NCCL version banner) goes to stderr; the returned function
    prints the ONE JSON line to the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)

    def emit(line: str) -> None:
        sys.stdout.flush()
        os.write(real, (line + "\n").encode())

    return emit


WORKLOADS = {
    # name: (model, LR side, default images per GPU per step, GFLOP per image (SURVEY.md 8d), metric, description)
    "drct-l": ("drct", 32, 256, 60.436e9, METRIC, "configs[2]: DRCT-L x4 RGB 32->128 px, batch 256 per GPU"),
    "drn-l": ("drn", 32, 64, 49.877e9, "DRN-L x4 128px HR images/sec (inference+scoring)",
              "configs[1]: DRN-L x4 RGB 32->128 px, batch 64 per GPU"),
    "drct-l-64": ("drct", 64, 128, 287.798e9, "DRCT-L x4 256px HR images/sec (inference+scoring)",
                  "configs[3]: DRCT-L x4 RGB 64->256 px (16 x 16 windows), batch 128 per GPU"),
}


DUMP_SR_SAMPLES = 1 << 20                      # SR pixels kept per workload (4 MiB as float32)


def dump_outputs(dump_dir: str, workload: str, scores: np.ndarray, sr_u8: torch.Tensor) -> None:
    """What the evaluator handed back in the last timed step: the fp64 score table [images, n_ws + 2] (ordered by image id)
    and a fixed sample (seed 0, ascending flat NHWC indices) of the uint8 SR pixels as float32."""
    os.makedirs(dump_dir, exist_ok=True)
    name = workload.replace("-", "_")
    np.save(os.path.join(dump_dir, f"{name}_scores.npy"), np.asarray(scores, dtype=np.float64))
    flat = sr_u8.reshape(-1)
    n = flat.numel()
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SR_SAMPLES), replace=False))
    sample = flat[torch.from_numpy(idx).to(flat.device)].float().cpu().numpy()
    np.save(os.path.join(dump_dir, f"{name}_sr_sample.npy"), sample)


def build_model(mods, workload: str, batch: int, dev):
    model_kind, lr_side, _, _, _, _ = WORKLOADS[workload]
    main_mod = mods["main"]
    hr_side = lr_side * SCALE
    torch.manual_seed(1)
    if model_kind == "drct":
        # the reference's DRCT-L configuration (src/main.py:83-142, setup_opt_drct: window_size = img_size // 4), random init
        opt = main_mod.setup_opt_drct(main_mod.DRCT(), 0.0, 11, "mvtec", "carpet", False, SCALE, True, NC, 1, batch, hr_side,
                                      lr_side, "", "", "", 1, 1, 1, 0.0, 0, ".", "1*L1")
        return mods["drct"].DRCT(opt).to(dev).eval()
    dopt = main_mod.setup_opt_drn(main_mod.DRN(), 0.0, 11, "mvtec", "carpet", False, SCALE, True, NC, 1, batch, hr_side, "",
                                  "", "", 1, 1, 1, 0.0, 0, ".", ".", "1*L1")
    model = mods["drn"].DRN(dopt).to(dev).eval()
    with torch.no_grad():                      # keep 80 residual blocks numerically tame with random weights
        for n_, p_ in model.named_parameters():
            if ".body.0." in n_ or ".body.2." in n_:
                p_.mul_(0.5)
    return model


def run_workload(mods, workload: str, B: int, steps: int, warmup: int, dev, rank: int, world: int, local_rank: int,
                 with_roofline: bool = True, dump_dir: str = None) -> dict:
    """One workload, timed twice: `value` with the inputs resident in HBM (CUDA events, L2 flushed between steps, max over
    ranks) and `e2e` through the public evaluator API from pinned host tensors (H2D copies + D2H read of the score table in
    the timed region).  Returns the fields of a bench record."""
    import torch.distributed as dist

    ops, evaluate, metrics = mods["ops"], mods["evaluate"], mods["metrics"]
    _, lr_side, _, flops_img, metric, wl = WORKLOADS[workload]
    hr_side = lr_side * SCALE
    model = build_model(mods, workload, B, dev)

    # ---- synthetic MVTec-shaped data; every rank gets its own shard of a (world * batch)-image set
    base = min(B, 64)                                   # distinct images generated per rank (tiled up to B)
    hr_u8, lr_u8, labels = synthetic_pairs(base, seed=1234 + rank, hr=hr_side)
    reps = (B + base - 1) // base
    # decoded-PNG bytes (uint8 HWC), exactly what evaluate_on_test hands the evaluator: the float scaling of the loader
    # (src/data.py:11-17) runs on the device, a quarter of the bytes cross PCIe
    lr_h = torch.from_numpy(np.ascontiguousarray(np.tile(lr_u8, (reps, 1, 1, 1))[:B])).pin_memory()
    hr_h = torch.from_numpy(np.ascontiguousarray(np.tile(hr_u8, (reps, 1, 1, 1))[:B])).pin_memory()
    labels = np.tile(labels, reps)[:B]
    lr_d, hr_d = lr_h.to(dev), hr_h.to(dev)
    wss = metrics.window_sizes_for(hr_side)
    ev = evaluate.BatchedEvaluator(model, 255.0, wss)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > L2 (126 MB)
    ids = torch.arange(rank, world * B, world, dtype=torch.int64, device=dev)

    def step_device():
        s = ev.step(lr_d, hr_d)
        if world > 1:                                    # one all_gather of the score rows; no host synchronisation
            return evaluate.gather_scores(s, ids, world * B, to_host=False)
        return s

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        flush.zero_()
        step_device()
    barrier()

    # ---- timed region: K steps, device events, L2 flushed between steps
    launches0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        e0.record()
        for _ in range(steps):
            flush.zero_()
            out = step_device()
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.LAUNCHES - launches0
    if dump_dir is not None and rank == 0:
        table = evaluate.scores_table(out, world * B) if world > 1 else out.cpu().numpy()
        dump_outputs(dump_dir, workload, table, ev.last_sr_u8)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * B * steps / (ms_total / 1e3)

    # ---- end to end through the public evaluator API: pinned host tensors in, score table out (host).  Every step's inputs are
    # copied host -> device inside the timed region (the evaluator keeps one batch of copy look-ahead on its
    # copy stream, exactly as evaluate_on_test drives it) and every step's score table is read back.
    nxt = ev.submit(lr_h, hr_h)
    for _ in range(6):                                   # warm both buffer sets: eager run, graph capture, first replay
        cur, nxt = nxt, ev.submit(lr_h, hr_h)
        ev.step_submitted(cur).cpu()
    ev.step_submitted(nxt).cpu()
    barrier()
    t0 = time.perf_counter()
    nxt = ev.submit(lr_h, hr_h)
    table, pending = None, None

    def consume(p_):                                     # the step's result on the host (every step's table is read back)
        p_[1].synchronize()
        return evaluate.scores_table(p_[0], world * B) if world > 1 else p_[0].numpy().copy()

    for i in range(steps):
        flush.zero_()
        cur, nxt = nxt, (ev.submit(lr_h, hr_h) if i + 1 < steps else None)
        s = ev.step_submitted(cur)
        if world > 1:
            s = evaluate.gather_scores(s, ids, world * B, to_host=False)
        h = ev.to_host_async(s)                          # D2H read of step i starts; the host first enqueues step i + 1 ...
        if pending is not None:
            table = consume(pending)                     # ... and only then waits for step i - 1's table
        pending = h
    table = consume(pending)
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = world * B * steps / float(dt.item())
    h2d = lr_h.numel() * lr_h.element_size() + hr_h.numel() * hr_h.element_size()
    d2h = B * (len(wss) + 2) * 8

    # ---- AUC on the gathered table (host, rank 0): the step's real consumer
    auc = None
    if rank == 0 and table is not None:
        y = labels[np.arange(world * B) // world]          # image id -> (rank = id % world, local index = id // world)
        best_ws, a_ssim, a_mse, a_psnr = metrics.aucs_from_scores(y, np.asarray(table), wss)
        auc = {"best_ws": int(best_ws), "ssim": a_ssim, "mse": a_mse, "psnr": a_psnr}

    # ---- roofline of the dominant (tcgen05) kernels: per-launch CUDA events in one extra, untimed step
    roofline = None
    TENSOR_KINDS = ("tc_gemm", "conv3x3", "conv3x3_halo", "swin_mlp", "swin_attn", "window_attention")
    if rank == 0 and with_roofline:
        ops.PROFILE = []
        torch.cuda.synchronize()
        ev.step(lr_d, hr_d)
        torch.cuda.synchronize()
        prof, ops.PROFILE = ops.PROFILE, None
        peaks = load_peaks()
        gemm = [(p[1], p[2].elapsed_time(p[3])) for p in prof if p[0] in TENSOR_KINDS]
        allk = [(p[0], p[2].elapsed_time(p[3])) for p in prof]
        step_ms = sum(d for _, d in allk)
        by_kind, flops_by_kind, n_by_kind = {}, {}, {}
        for (k, d), p_ in zip(allk, prof):
            by_kind[k] = by_kind.get(k, 0.0) + d
            flops_by_kind[k] = flops_by_kind.get(k, 0.0) + p_[1]
            n_by_kind[k] = n_by_kind.get(k, 0) + 1
        # the dominant kernel of the step (largest share of the device time); algorithmic FLOPs per launch = what ops.py counts
        # for that call (DESIGN.md section 4), duration = CUDA events around the launch on the launching stream
        dom = max(by_kind, key=by_kind.get)
        dom_tf = flops_by_kind[dom] / (by_kind[dom] * 1e-3) / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")     # dram bytes per launch from the committed ncu --set full capture
        if os.path.isfile(tpath) and workload == "drct-l":
            traffic = json.load(open(tpath)).get(DOMINANT_KERNEL_NAMES.get(dom, dom), {}).get("dram_bytes_per_launch")
        flops = sum(f for f, _ in gemm)
        tms = sum(d for _, d in gemm)
        kname = DOMINANT_KERNEL_NAMES.get(dom, dom)
        if dom == "window_attention" and lr_side == 64:
            kname = "window_attn16_tc_kernel"                # 16 x 16 windows: csrc/attention_tc16.cu
        roofline = {"bound": "tensor", "kernel": kname, "achieved": dom_tf, "peak": peaks["sustained"],
                    "unit": "TFLOP/s", "frac": dom_tf / peaks["sustained"], "frac_of_burst": dom_tf / peaks["burst"],
                    "peak_source": peaks["source"] + " (sustained bf16: the kernel is timed inside a long step)",
                    "traffic": traffic, "launches": n_by_kind[dom], "flops_per_launch": flops_by_kind[dom] / n_by_kind[dom],
                    "avg_launch_us": 1e3 * by_kind[dom] / n_by_kind[dom], "share_of_step": by_kind[dom] / step_ms if step_ms else None,
                    "all_tcgen05_kernels": {"kinds": list(TENSOR_KINDS), "achieved": flops / (tms * 1e-3) / 1e12 if tms else None,
                                            "frac": flops / (tms * 1e-3) / 1e12 / peaks["sustained"] if tms else None,
                                            "launches": len(gemm), "flops_per_step": flops, "kernel_ms_per_step": tms,
                                            "share_of_step": tms / step_ms if step_ms else None},
                    "ms_by_kernel": {k: round(v, 3) for k, v in sorted(by_kind.items(), key=lambda kv: -kv[1])},
                    "tflops_by_kernel": {k: round(flops_by_kind[k] / (by_kind[k] * 1e-3) / 1e12, 1) for k in by_kind
                                         if flops_by_kind[k] > 0 and by_kind[k] > 0},
                    "model_flops_per_image": flops_img,
                    "model_tensor_frac": (value / world) * flops_img / (peaks["sustained"] * 1e12)}
    n_ws = len(wss)
    del ev, model, flush
    torch.cuda.empty_cache()
    return {
        "metric": metric, "value": value, "unit": "images/s", "steps": steps, "warmup": max(warmup, 3),
        "ms_per_step": ms_total / steps, "dtype": "bf16",
        "config": {"workload": wl + f", inference + scoring ({n_ws}-window SSIM sweep + MSE + PSNR per image)",
                   "batch_per_gpu": B, "global_batch": world * B, "parallelism": f"dp{world} (images sharded by rank; "
                   "one all_gather of score rows + ids)", "l2": "flushed between steps (256 MiB write)",
                   "weights": "random init, seed 1", "inputs": "uint8 HWC image pairs (decoded-PNG bytes)", "auc": auc},
        "roofline": roofline,
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches, "clocks": clocks.summary(),
    }


def main():
    args = parse()
    emit = _guard_stdout()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, emit)
        return

    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    mods = {n: importlib.import_module(f"{PKG}.{n}") for n in ("ops", "drct", "drn", "evaluate", "metrics", "main")}

    B = args.batch if args.batch is not None else WORKLOADS[args.workload][2]
    head = run_workload(mods, args.workload, B, args.steps, args.warmup, dev, rank, world, local_rank,
                        dump_dir=args.dump_outputs)

    # ---- the other BASELINE configurations ride in the same line as sub-records (same timing rules)
    subs = {}
    if not args.no_sub_workloads:
        for name, key in (("drn-l", "drn_l_b64"), ("drct-l-64", "drct_l_64px_b128"), ("drct-l", "drct_l_b256")):
            if name == args.workload:
                continue
            r = run_workload(mods, name, WORKLOADS[name][2], args.steps, 3, dev, rank, world, local_rank,
                             dump_dir=args.dump_outputs)
            r.pop("clocks", None)
            subs[key] = r
        if world > 1 and args.workload == "drct-l" and 256 % world == 0:
            # strong scaling: the SAME 256 images split over the ranks (SURVEY.md 8d)
            r = run_workload(mods, "drct-l", 256 // world, args.steps, 3, dev, rank, world, local_rank, with_roofline=False)
            subs["strong_scaling_global256"] = {"value": r["value"], "unit": "images/s", "ms_per_step": r["ms_per_step"],
                                                "batch_per_gpu": 256 // world, "global_batch": 256, "e2e": r["e2e"],
                                                "scaling": "strong"}

    # ---- CPU baseline beside it (rank 0, N=1 only): oracle port on a bounded sample
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_record(args)

    if rank == 0:
        line = {
            "metric": head["metric"], "value": head["value"], "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": head["warmup"], "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": head["config"],
            "roofline": head["roofline"], "cpu_baseline": cpu_baseline, "e2e": head["e2e"],
            "gpu_launches": head["gpu_launches"], "clocks": head["clocks"], "workloads": subs,
        }
        emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
