"""Every dispatch branch of the scorer (csrc/scoring.cu, launch_score) against an oracle that follows the kernels' own gray conversion
and per-pixel term (oracle/scoring_oracle.py: gray01_like_kernel, ssim_sweep_like_kernel, mse_like_kernel), at 1e-10 instead of the
reference's fp32 tolerance; the strided entry points through each kernel; that an image's score row does not depend on the batch it
is scored in (the batch size picks the kernel); full window sweeps at MVTec-native sizes; and the rejections."""
import importlib
import math
import zlib

import numpy as np
import pytest
import torch

from oracle import scoring_oracle as S
from gpu_common import PKG, TableModel

pytestmark = pytest.mark.gpu

ops = importlib.import_module(PKG + ".ops")
metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")

SSIM_TOL, MSE_RTOL, PSNR_TOL = 1e-10, 1e-14, 1e-10
SMEM_LIMIT = 227 * 1024


def _sms() -> int:
    return torch.cuda.get_device_properties(0).multi_processor_count


def _kernel_for(B: int, H: int, W: int, n_ws: int, sms: int) -> str:
    """launch_score's choice, restated: the warp-per-window kernel (`fast`, 4 columns a lane: 16-byte loads when W % 4 == 0, scalar
    loads otherwise; two CTAs per image when that saves waves), the 4-warps-per-window kernel (`fast4`) when the batch leaves more
    than half of the SMs idle, and the thread-per-column kernel (`general`) for W > 128, gray planes that do not fit shared memory or
    no window sizes; `general/dyn` when its prefix rows need more than the 48 KB of static shared memory."""
    fast_smem = (32 + 16 * 5 * (W + (W >> 4) + 1)) * 8 + 2 * H * W * 4
    if W <= 128 and fast_smem <= SMEM_LIMIT and n_ws > 0:
        fast4_smem = (32 + 8 * (5 * 32 + 5 * (W + 1))) * 8 + 2 * H * W * 4
        if 2 * B <= sms and n_ws > 8 and fast4_smem <= SMEM_LIMIT:
            return "fast4"

        def cost(parts):
            return -(-B * parts // sms) * (0.3 + -(-n_ws // (16 * parts)))

        if n_ws > 16 and cost(2) < cost(1):
            return "fast/2cta"
        return "fast/w4" if W % 4 == 0 else "fast/scalar"
    if n_ws == 0:
        return "general/psnr"
    if W <= 128:
        return "general/planes-too-big"
    return "general/dyn" if (32 + 2 * 5 * 32 + 2 * 5 * (W + 1)) * 8 > 48 * 1024 else "general"


BRANCHES = {"fast/w4", "fast/scalar", "fast/2cta", "fast4", "general", "general/dyn", "general/planes-too-big", "general/psnr"}
KERNEL_NAME = {"fast": "score_images_fast_kernel", "fast4": "score_images_fast4_kernel", "general": "score_images_kernel"}


def _sweep(h, w):
    """The evaluator's sweep plus ws = 1 and the largest window the kernels take (ws / 2 = min(H, W) - 1)."""
    m = min(h, w)
    return sorted(set(S.window_sizes_for(m)) | {1, 2 * m - 1})


def _cases(sms):
    """(id, B, H, W, C, window sizes).  Batches are sized in SMs so that each case reaches its branch on any SM count."""
    half = sms // 2
    return [
        ("fast-w4-128sq-rgb", half + 1, 128, 128, 3, _sweep(128, 128)),
        ("fast-scalar-61x99-rgb", 4, 61, 99, 3, _sweep(61, 99)),
        ("fast-scalar-127x90-gray", half + 1, 127, 90, 1, _sweep(127, 90)),
        ("fast-scalar-2x3-gray", 4, 2, 3, 1, [1, 3]),
        ("fast-2cta-64sq-rgb", 150 if sms == 148 else sms + 2, 64, 64, 3, WSS20),
        ("fast4-96sq-rgb-b1", 1, 96, 96, 3, _sweep(96, 96)),
        ("fast4-96sq-rgb", half, 96, 96, 3, _sweep(96, 96)),
        ("fast4-128sq-gray-b1", 1, 128, 128, 1, _sweep(128, 128)),
        ("fast4-128sq-gray", half, 128, 128, 1, _sweep(128, 128)),
        ("fast4-127x90-gray", 4, 127, 90, 1, _sweep(127, 90)),
        ("fast4-90x127-rgb", 4, 90, 127, 3, _sweep(90, 127)),
        ("general-129sq-rgb", 4, 129, 129, 3, _sweep(129, 129)),
        ("general-250sq-gray", 4, 250, 250, 1, [1, 3, 11, 249, 499]),
        ("general-256sq-rgb-full", 4, 256, 256, 3, _sweep(256, 256)),
        ("general-planes-1024x120-rgb", 4, 1024, 120, 3, _sweep(1024, 120)),
        ("general-dyn-40x1024-gray", 4, 40, 1024, 1, _sweep(40, 1024)),
        ("general-psnr-only-64x96-rgb", 4, 64, 96, 3, []),
    ]


WSS20 = list(range(1, 38, 2)) + [127]         # 20 window sizes: more than the 16 warps of one fast-kernel CTA
ORACLE_ROWS = (0, 1, 2, 3, 4, 5)                 # random, identical, constant, all-zero, random, noisy; and the batch's last row


def _pairs(B, H, W, C, seed):
    """uint8 NHWC pairs: 0 = independent random images, 1 = an identical pair, 2 = two different constants, 3 = an all-zero pair,
    then SR = HR + noise and independent random images in turn."""
    rng = np.random.default_rng(seed)
    hr = rng.integers(0, 256, (B, H, W, C), dtype=np.uint8)
    sr = np.clip(hr.astype(np.int16) + rng.integers(-24, 25, hr.shape), 0, 255).astype(np.uint8)
    sr[0::2] = rng.integers(0, 256, sr[0::2].shape, dtype=np.uint8)
    if B > 1:
        sr[1] = hr[1]
    if B > 3:
        hr[2], sr[2] = 97, 31
        hr[3], sr[3] = 0, 0
    return sr, hr


def _check_rows(got, sr, hr, wss, rows, *, c1=0.01 * 0.01, c2=0.03 * 0.03, zero_pad=False, peak2=1.0, gray=None, mse_vals=None):
    """got: fp64 [B, n_ws + 2] from the device; the oracle is evaluated for `rows`.  gray / mse_vals map (sr_i, hr_i) to the gray
    planes / the MSE operands (default: the uint8 conventions of adsr_score_images)."""
    gray = gray or (lambda s, h: (S.gray01_like_kernel(h), S.gray01_like_kernel(s)))
    mse_vals = mse_vals or (lambda s, h: (s.astype(np.float32) / np.float32(255.0), h.astype(np.float32) / np.float32(255.0)))
    n = len(wss)
    worst = [0.0, 0.0, 0.0]
    for i in rows:
        if n:
            gh, gs = gray(sr[i], hr[i])
            want = S.ssim_sweep_like_kernel(gh, gs, wss, c1, c2, zero_pad)
            worst[0] = max(worst[0], float(np.abs(got[i, :n] - want).max()))
        a, b = mse_vals(sr[i], hr[i])
        mse = S.mse_like_kernel(a, b)
        assert (got[i, n] == 0.0) == (mse == 0.0), f"row {i}: MSE {got[i, n]!r} vs {mse!r}"
        if mse > 0:
            worst[1] = max(worst[1], abs(got[i, n] - mse) / mse)
            worst[2] = max(worst[2], abs(got[i, n + 1] - 10.0 * math.log10(peak2 / mse)))
        else:
            assert got[i, n + 1] == math.inf, f"row {i}: PSNR of an exact match is {got[i, n + 1]!r}"
    msg = f"largest error: SSIM {worst[0]:.3e}, MSE relative {worst[1]:.3e}, PSNR {worst[2]:.3e} dB"
    assert worst[0] <= SSIM_TOL and worst[1] <= MSE_RTOL and worst[2] <= PSNR_TOL, msg
    return worst


def test_case_list_reaches_every_branch():
    sms = _sms()
    reached = {_kernel_for(B, H, W, len(wss), sms) for _, B, H, W, _, wss in _cases(sms)}
    assert reached == BRANCHES, f"unreached: {sorted(BRANCHES - reached)}"
    for _, B, H, W, _, wss in _cases(sms):                  # and every case exercises the reflection limit in both directions
        if wss:
            assert 1 in wss and max(wss) // 2 == min(H, W) - 1
    shapes = {(_kernel_for(B, H, W, len(w), sms).split("/")[0], (H > W) - (H < W)) for _, B, H, W, _, w in _cases(sms) if w}
    for kernel in ("fast", "fast4", "general"):
        assert {(kernel, 1), (kernel, -1)} <= shapes, f"{kernel}: needs a tall and a wide image"


@pytest.mark.parametrize("case", [c[0] for c in _cases(148)])
def test_branch_matches_faithful_oracle(case):
    sms = _sms()
    _, B, H, W, C, wss = next(c for c in _cases(sms) if c[0] == case)
    sr, hr = _pairs(B, H, W, C, seed=zlib.crc32(case.encode()))
    got = ops.score_images(torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda(), wss).cpu().numpy()
    assert got.shape == (B, len(wss) + 2)
    rows = sorted({i for i in ORACLE_ROWS if i < B} | {B - 1})
    _check_rows(got, sr, hr, wss, rows)
    for i in (1, 3):                                         # identical pairs: exactly 1 / 0 / +inf
        if i < B and np.array_equal(sr[i], hr[i]):
            assert np.all(got[i, :len(wss)] == 1.0) and got[i, len(wss)] == 0.0 and got[i, len(wss) + 1] == math.inf


def test_kernel_names_in_profile():
    """Each case launches the kernel _kernel_for names (when the profiler records CUDA kernels on this runner)."""
    from torch.profiler import ProfilerActivity, profile
    sms = _sms()
    seen = {}
    for case, B, H, W, C, wss in _cases(sms):
        z = torch.zeros(B, H, W, C, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ops.score_images(z, z, wss)
            torch.cuda.synchronize()
        seen[case] = [e.name for e in prof.events() if "score_images" in e.name]
    if not any(seen.values()):
        pytest.skip("torch.profiler recorded no CUDA kernels on this runner")
    for case, B, H, W, C, wss in _cases(sms):
        want = KERNEL_NAME[_kernel_for(B, H, W, len(wss), sms).split("/")[0]]
        names = seen[case]                                  # no kernel name is a substring of another
        assert names and all({k for k in KERNEL_NAME.values() if k in n} == {want} for n in names), (case, want, names)


# ----------------------------------------------------------------------------------------------------------- strided entry points
def test_ssim_numpy_psnr_numpy_fp32_hwc_odd_width():
    """ssim_numpy / psnr_numpy on fp32 HWC (W % 4 != 0: the fast kernel's scalar path; W > 128: the general kernel)."""
    rng = np.random.default_rng(5)
    for h, w in ((70, 97), (33, 150)):
        for c in (1, 3):
            ref = rng.random((h, w, c), dtype=np.float32) * np.float32(1.2)
            img = np.clip(ref + rng.standard_normal(ref.shape).astype(np.float32) * np.float32(0.05), 0, None).astype(np.float32)
            for ws, dr in ((7, None), (2 * min(h, w) - 1, 2.0)):
                got = metrics.ssim_numpy(ref, img, win_size=ws, data_range=dr)
                d = 1.0 if dr is None else dr
                want = S.ssim_sweep_like_kernel(S.gray01_like_kernel(ref), S.gray01_like_kernel(img), [ws], (0.01 * d) ** 2,
                                                (0.03 * d) ** 2)[0]
                assert abs(got - want) <= SSIM_TOL, (h, w, c, ws, got - want)
            mse = S.mse_like_kernel(img, ref)
            assert abs(metrics.psnr_numpy(ref, img) - 10.0 * math.log10(1.0 / mse)) <= PSNR_TOL
            assert abs(metrics.psnr_numpy(ref, img, data_range=2.0) - 10.0 * math.log10(4.0 / mse)) <= PSNR_TOL


def test_ssim_torch_psnr_torch_shaved_views_out_of_range():
    """ssim_torch / psnr_torch on shaved NCHW views (strided) whose values leave [0, rgb_range]: SSIM clamps to [0, 1] and pads
    with zeros, PSNR does not clamp."""
    rng = np.random.default_rng(6)
    rgb = 255.0
    for b, c, h, w in ((2, 3, 72, 72), (2, 1, 60, 140), (3, 3, 136, 40)):
        hr = (rng.random((b, c, h, w)) * 300.0 - 20.0).astype(np.float32)
        sr = (hr + rng.standard_normal(hr.shape).astype(np.float32) * 9.0).astype(np.float32)
        ts, th = torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda()
        a = np.clip(sr[..., 4:-4, 4:-4] / np.float32(rgb), 0, 1).astype(np.float32)
        e = np.clip(hr[..., 4:-4, 4:-4] / np.float32(rgb), 0, 1).astype(np.float32)
        c1, c2 = (0.01 * 1.0) ** 2 * (255.0 ** 2), (0.03 * 1.0) ** 2 * (255.0 ** 2)
        want = np.mean([S.ssim_sweep_like_kernel(S.gray01_like_kernel(e[i].transpose(1, 2, 0)),
                                                 S.gray01_like_kernel(a[i].transpose(1, 2, 0)), [11], c1, c2, zero_pad=True)[0]
                        for i in range(b)])
        assert abs(metrics.ssim_torch(ts, th, rgb) - want) <= SSIM_TOL
        d = (sr[..., 4:-4, 4:-4] / np.float32(rgb) - hr[..., 4:-4, 4:-4] / np.float32(rgb)).astype(np.float32)
        per_image = [float(np.sum((d[i] * d[i]).astype(np.float64)) / d[i].size) for i in range(b)]
        got = ops.score_images_strided(ts[..., 4:-4, 4:-4], th[..., 4:-4, 4:-4], "chw", [], div=rgb).cpu().numpy()[:, 0]
        assert np.abs(got - per_image).max() <= MSE_RTOL * max(per_image)
        assert abs(metrics.psnr_torch(ts, th, rgb) - 10.0 * math.log10(1.0 / np.mean(per_image))) <= PSNR_TOL


@pytest.mark.parametrize("side", [40, 248])
def test_validate_images_round_quantised_zero_padded(side):
    """validate_images (Trainer.test's body) at 40^2 (fast kernel) and at the 248^2 shaved crops of --resolution 256 (general
    kernel), B = 3: round-quantised SR, zero-padded SSIM with the 255^2-scaled constants, unclamped MSE."""
    rng = np.random.default_rng(side)
    rgb = 255.0
    full = side + 8
    hr = (rng.random((3, 3, full, full)) * 280.0 - 10.0).astype(np.float32)
    sr = (hr + rng.standard_normal(hr.shape).astype(np.float32) * 12.0).astype(np.float32)
    sr[1] = hr[1]
    ts, th = torch.from_numpy(sr).cuda()[..., 4:-4, 4:-4], torch.from_numpy(hr).cuda()[..., 4:-4, 4:-4]
    got = ops.validate_images(ts, th, rgb).cpu().numpy()
    q = S.quantize_round(sr[..., 4:-4, 4:-4], rgb)
    h = hr[..., 4:-4, 4:-4]
    qs = (q / np.float32(rgb)).astype(np.float32)
    hs = (h / np.float32(rgb)).astype(np.float32)
    c1, c2 = 0.01 * 0.01 * 255.0 * 255.0, 0.03 * 0.03 * 255.0 * 255.0
    hwc = lambda x: np.clip(x, 0, 1).astype(np.float32).transpose(1, 2, 0)
    _check_rows(got[:, [0, 1, 2]], qs, hs, [11], range(3), c1=c1, c2=c2, zero_pad=True,
                gray=lambda s, r: (S.gray01_like_kernel(hwc(r)), S.gray01_like_kernel(hwc(s))), mse_vals=lambda s, r: (s, r))


# ----------------------------------------------------------------------------------------------------------- batch independence
def test_score_rows_do_not_depend_on_the_batch():
    """Image i's row is bit-identical whether it is scored alone, in a batch that runs the 4-warps-per-window kernel, one that runs
    the warp-per-window kernel, or a batch of 256; and with one or two CTAs per image."""
    sms = _sms()
    g = torch.Generator(device="cuda").manual_seed(3)
    hr = torch.randint(0, 256, (256, 128, 128, 3), generator=g, device="cuda", dtype=torch.uint8)
    sr = (hr.to(torch.int16) + torch.randint(-20, 21, hr.shape, generator=g, device="cuda", dtype=torch.int16)).clamp(0, 255)
    sr = sr.to(torch.uint8)
    wss = metrics.window_sizes_for(128)
    full = ops.score_images(sr, hr, wss)
    kinds = set()
    for b in (1, sms // 2, sms // 2 + 1, 256):
        kinds.add(_kernel_for(b, 128, 128, len(wss), sms))
        for i0 in range(0, 256, b)[:3]:
            part = ops.score_images(sr[i0:i0 + b], hr[i0:i0 + b], wss)
            assert torch.equal(part, full[i0:i0 + part.shape[0]]), f"batch {b}, rows {i0}..: differ from the batch of 256"
    assert kinds == {"fast4", "fast/w4"}

    wss20 = WSS20
    hr, sr = hr[:, :64, :64].contiguous(), sr[:, :64, :64].contiguous()
    big = 150 if sms == 148 else sms + 2
    hr2, sr2 = torch.cat([hr, hr])[:big], torch.cat([sr, sr])[:big]
    two = ops.score_images(sr2, hr2, wss20)
    assert _kernel_for(big, 64, 64, len(wss20), sms) == "fast/2cta"
    for b in (1, sms // 2, sms // 2 + 1):
        assert _kernel_for(b, 64, 64, len(wss20), sms) in ("fast4", "fast/w4")
        assert torch.equal(ops.score_images(sr2[:b], hr2[:b], wss20), two[:b]), f"batch {b} differs from two CTAs per image"


def test_evaluator_tables_equal_at_batch_64_and_256():
    n = 300
    g = torch.Generator(device="cuda").manual_seed(8)
    hr = torch.randint(0, 256, (n, 128, 128, 3), generator=g, device="cuda", dtype=torch.uint8)
    sr = (hr.to(torch.int16) + torch.randint(-12, 13, hr.shape, generator=g, device="cuda", dtype=torch.int16)).clamp(0, 255)
    sr = sr.to(torch.uint8)
    wss = metrics.window_sizes_for(128)
    tables = []
    for bs in (64, 256):
        ev = evaluate.BatchedEvaluator(TableModel(sr), 255.0, wss)
        ev.use_graph = False
        rows, ids = [], []
        for i0 in range(0, n, bs):
            m = min(bs, n - i0)
            rows.append(ev.step(torch.full((m, 1, 1, 1), float(i0), device="cuda"), hr[i0:i0 + m]).clone())
            ids += list(range(i0, i0 + m))
        tables.append(evaluate.gather_scores(torch.cat(rows), torch.tensor(ids, device="cuda"), n))
    assert np.array_equal(tables[0], tables[1]), f"{int((tables[0] != tables[1]).any(1).sum())} of {n} rows differ"


# ----------------------------------------------------------------------------------------------------------- MVTec-native sizes
@pytest.mark.parametrize("b,h,w,c", [(2, 700, 700, 1), (1, 700, 1024, 3)])
def test_full_sweep_at_mvtec_native_sizes(b, h, w, c):
    """700 px and larger images: the evaluator's full sweep has 70 window sizes (102 at 1024 px)."""
    sr, hr = _pairs(b, h, w, c, seed=h + w)
    wss = metrics.window_sizes_for(min(h, w))
    assert len(wss) == 70
    got = metrics.score_batch(torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda(), wss).cpu().numpy()
    _check_rows(got, sr, hr, wss, range(b))


# ----------------------------------------------------------------------------------------------------------- rejections
def test_window_count_limit_and_rejections():
    z = lambda b, h, w, c: torch.zeros(b, h, w, c, dtype=torch.uint8, device="cuda")
    a = z(1, 1024, 1024, 1)
    wss = metrics.window_sizes_for(1024)
    assert len(wss) == 102
    got = ops.score_images(a, a, wss).cpu().numpy()
    assert np.all(got[0, :102] == 1.0) and got[0, 102] == 0.0 and got[0, 103] == math.inf
    x = z(1, 300, 300, 1)
    with pytest.raises(RuntimeError, match="unsupported shape"):
        ops.score_images(x, x, [3] * 129)                    # more window sizes than the kernels take
    ops.score_images(x, x, [3] * 128)
    for bad, wss in ((z(1, 8, 1025, 1), [3]),                # wider than a CTA
                     (z(1, 1, 8, 1), [1]),                   # one row
                     (z(1, 8, 8, 2), [3]),                   # two channels
                     (z(1, 8, 8, 1), [4]),                   # even window
                     (z(1, 8, 8, 1), [0]),
                     (z(1, 8, 20, 1), [17]),                 # H < W: ws / 2 = 8 >= H
                     (z(1, 20, 8, 1), [17])):                # H > W: ws / 2 = 8 >= W
        with pytest.raises(RuntimeError, match="unsupported shape"):
            ops.score_images(bad, bad, wss)
    empty = z(0, 16, 16, 3)
    out = torch.full((0, 3), 7.0, dtype=torch.float64, device="cuda")
    assert ops.score_images(empty, empty, [3], out).shape == (0, 3)
    torch.cuda.synchronize()
