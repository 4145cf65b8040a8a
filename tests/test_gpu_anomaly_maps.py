"""GPU tests of the anomaly maps (csrc/anomaly_maps.cu): per-pixel 1 - SSIM and squared-error maps of uint8 SR / HR pairs, their
Gaussian smoothing and per-image maxima, against a numpy oracle (fp64 reflect-padded box sums as oracle/scoring_oracle.py,
scipy.ndimage.gaussian_filter for the smoothing) and against the existing scorer; then the evaluator and CLI paths."""
import importlib
import os

import numpy as np
import pytest
import torch
from PIL import Image
from scipy.ndimage import gaussian_filter

from oracle import drct_oracle as O
from oracle import scoring_oracle as S
from gpu_common import PKG, DrctOpt

pytestmark = pytest.mark.gpu

ops = importlib.import_module(PKG + ".ops")
metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")


# ------------------------------------------------------------------------------------------------------------- oracle
def oracle_maps(sr_u8: np.ndarray, hr_u8: np.ndarray, ws: int, sigma: float):
    """One uint8 HWC pair -> (1 - SSIM map, squared-error map) as float32 [H, W]; smoothed with scipy when sigma > 0."""
    gs, gh = S.to_gray01(sr_u8), S.to_gray01(hr_u8)
    C1, C2 = 1e-4, 9e-4
    mu1, mu2 = S._box_mean_f64(gh, ws), S._box_mean_f64(gs, ws)
    s1 = S._box_mean_f64(gh * gh, ws) - mu1 * mu1
    s2 = S._box_mean_f64(gs * gs, ws) - mu2 * mu2
    s12 = S._box_mean_f64(gh * gs, ws) - mu1 * mu2
    ssim = ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 * mu1 + mu2 * mu2 + C1) * (s1 + s2 + C2))
    m_ssim = (1.0 - ssim).astype(np.float32)
    d = sr_u8.astype(np.float32) / np.float32(255.0) - hr_u8.astype(np.float32) / np.float32(255.0)
    m_se = (d * d).astype(np.float64).mean(axis=2).astype(np.float32)
    if sigma > 0:
        m_ssim = gaussian_filter(m_ssim, sigma, mode="reflect", truncate=4.0)
        m_se = gaussian_filter(m_se, sigma, mode="reflect", truncate=4.0)
    return m_ssim, m_se


def _pairs(h, w, c, seed):
    """4 pairs: random SR / HR, an identical pair, a constant HR, SR = HR + noise."""
    rng = np.random.default_rng(seed)
    hr = rng.integers(0, 256, (4, h, w, c), dtype=np.uint8)
    sr = rng.integers(0, 256, (4, h, w, c), dtype=np.uint8)
    sr[1] = hr[1]
    hr[2] = 97
    sr[3] = np.clip(hr[3].astype(np.int16) + rng.integers(-6, 7, (h, w, c)), 0, 255).astype(np.uint8)
    return sr, hr


# a partial last band of 16 rows (100, 130, 17), partially active warps (84, 33), the dynamic shared memory of W >= 582 (1024) and a
# Gaussian radius of H - 1 (sigma 4 on 17 rows: r = 16); "max" is the largest window, ws / 2 = min(H, W) - 1
MAP_SHAPES = [(128, 128, 3), (128, 128, 1), (64, 96, 3), (256, 256, 3), (100, 84, 3), (130, 33, 3), (17, 1024, 1)]


@pytest.mark.parametrize("sigma", [0.0, 4.0])
@pytest.mark.parametrize("ws", [3, 11, 33, "max"])
@pytest.mark.parametrize("h,w,c", MAP_SHAPES)
def test_maps_match_oracle(h, w, c, ws, sigma):
    ws = 2 * min(h, w) - 1 if ws == "max" else ws
    sr, hr = _pairs(h, w, c, seed=h + w + c + ws)
    m_ssim, m_se, m_max = (t.cpu().numpy() for t in ops.anomaly_maps(torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda(), ws, sigma))
    assert m_ssim.shape == (4, h, w) and m_se.shape == (4, h, w) and m_max.shape == (4, 2)
    for i in range(4):
        raw_ssim, raw_se = oracle_maps(sr[i], hr[i], ws, 0.0)
        want_ssim, want_se = (raw_ssim, raw_se) if sigma == 0 else oracle_maps(sr[i], hr[i], ws, sigma)
        if sigma == 0:
            # the kernels' own gray and per-pixel term: 1 - SSIM in fp64, rounded once to fp32
            exact = 1.0 - next(S.ssim_maps_like_kernel(S.gray01_like_kernel(hr[i]), S.gray01_like_kernel(sr[i]), [ws]))
            ulp = np.spacing(np.abs(exact).astype(np.float32)).astype(np.float64)
            worst = float((np.abs(m_ssim[i] - exact) / ulp).max())
            assert worst <= 1.0, f"image {i}: 1-SSIM map off by {worst:.2f} fp32 ulp of the kernel-faithful oracle"
        assert np.abs(m_ssim[i] - want_ssim).max() <= 1e-5, f"image {i}: 1-SSIM map"
        assert np.abs(m_se[i] - want_se).max() <= (1e-7 if sigma == 0 else 1e-5), f"image {i}: SE map"
    assert not m_ssim[1].any() and not m_se[1].any(), "an identical pair must give all-zero maps"
    assert np.array_equal(m_max, np.stack([m_ssim.reshape(4, -1).max(1), m_se.reshape(4, -1).max(1)], 1).astype(np.float64))


@pytest.mark.parametrize("h,w,c", MAP_SHAPES)
def test_map_means_equal_scorer_columns(h, w, c):
    """The unsmoothed 1 - SSIM map averages to 1 - the scorer's SSIM of that window size, the SE map to its MSE column."""
    sr, hr = _pairs(h, w, c, seed=3)
    sr_d, hr_d = torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda()
    wss = [3, 11, 33]
    scores = ops.score_images(sr_d, hr_d, wss).cpu().numpy()
    for j, ws in enumerate(wss):
        m_ssim, m_se, _ = ops.anomaly_maps(sr_d, hr_d, ws, 0.0)
        mean_ssim = m_ssim.double().mean(dim=(1, 2)).cpu().numpy()
        mean_se = m_se.double().mean(dim=(1, 2)).cpu().numpy()
        assert np.abs(mean_ssim - (1.0 - scores[:, j])).max() <= 1e-6
        assert np.abs(mean_se - scores[:, len(wss)]).max() <= 1e-7


@pytest.mark.parametrize("sigma", [0.0, 4.0])
def test_deterministic_and_batch_independent(sigma):
    rng = np.random.default_rng(11)
    sr = torch.from_numpy(rng.integers(0, 256, (6, 128, 128, 3), dtype=np.uint8)).cuda()
    hr = torch.from_numpy(rng.integers(0, 256, (6, 128, 128, 3), dtype=np.uint8)).cuda()
    first = [t.clone() for t in ops.anomaly_maps(sr, hr, 11, sigma)]
    again = ops.anomaly_maps(sr, hr, 11, sigma)
    for a, b in zip(first, again):
        assert torch.equal(a, b)
    for i in (0, 3, 5):
        alone = ops.anomaly_maps(sr[i:i + 1], hr[i:i + 1], 11, sigma)
        for a, b in zip(first, alone):
            assert torch.equal(a[i:i + 1], b)


def test_rejections():
    rng = np.random.default_rng(2)
    img = lambda h, w, c: torch.from_numpy(rng.integers(0, 256, (2, h, w, c), dtype=np.uint8)).cuda()
    a, b = img(16, 16, 3), img(16, 16, 3)
    with pytest.raises(RuntimeError):
        ops.anomaly_maps(a, b, 10, 0.0)                      # even window size
    with pytest.raises(RuntimeError):
        ops.anomaly_maps(a, b, 33, 0.0)                      # ws / 2 >= min(H, W)
    with pytest.raises(RuntimeError):
        ops.anomaly_maps(a, b, 11, 4.0)                      # Gaussian radius 16 >= min(H, W)
    with pytest.raises(RuntimeError):
        ops.anomaly_maps(img(16, 16, 2), img(16, 16, 2), 3, 0.0)   # two channels
    f32 = dict(dtype=torch.float32, device="cuda")
    out = (torch.empty(2, 16, 16, **f32), torch.empty(2, 16, 16, **f32), torch.empty(2, 2, dtype=torch.float64, device="cuda"), None)
    with pytest.raises(RuntimeError):
        ops.anomaly_maps(a, b, 3, 1.0, out=out)              # smoothing without scratch
    ops.anomaly_maps(a, b, 3, 0.0, out=out)                  # no smoothing: no scratch needed
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------- evaluator
def _small_drct(seed=6):
    drct = importlib.import_module(PKG + ".drct")
    cfg = O.DrctCfg(num_layers=1)
    sd = O.make_state_dict(cfg, seed=seed)
    model = drct.DRCT(DrctOpt(layers=1))
    model.load_state_dict(sd, strict=True)
    return model.to("cuda").eval()


def test_evaluator_maps_graph_and_pipelined_match_eager():
    """BatchedEvaluator(maps=...): eager steps, CUDA-graph replays and run_pipelined give bit-identical maps and scores; a
    maps-off evaluator gives the same score table."""
    model = _small_drct()
    hr, lr, _ = S.synthetic_dataset(12, hr=128, nc=3, scale=4, seed=5)
    to_t = lambda a: torch.from_numpy(np.ascontiguousarray(a.transpose(0, 3, 1, 2))).float()
    batches = [(to_t(lr[i:i + 4]).pin_memory(), to_t(hr[i:i + 4]).pin_memory()) for i in (0, 4, 8)]
    wss = metrics.window_sizes_for(128)
    maps = (11, 4.0)

    eager = evaluate.BatchedEvaluator(model, 255.0, wss, maps=maps)
    eager.use_graph = False
    want = []
    for l, h in batches:
        s = eager.step(l, h).cpu()
        want.append((s, [t.cpu() for t in eager.last_maps], eager.last_sr_u8.cpu(), eager.last_hr_u8.cpu()))
        # the maps are those of the step's own uint8 SR / HR
        ref = ops.anomaly_maps(eager.last_sr_u8, eager.last_hr_u8, *maps)
        for a, b in zip(ref, want[-1][1]):
            assert torch.equal(a.cpu(), b)

    off = evaluate.BatchedEvaluator(model, 255.0, wss)
    off.use_graph = False
    for (l, h), w in zip(batches, want):
        assert torch.equal(off.step(l, h).cpu(), w[0])
        assert off.last_maps is None

    ev = evaluate.BatchedEvaluator(model, 255.0, wss, maps=maps)
    for rep in range(4):                                    # eager warm-up, capture, then replays
        for s, w in zip(ev.run_pipelined(batches), want):
            assert torch.equal(s.cpu(), w[0])
            for a, b in zip(ev.last_maps, w[1]):
                assert torch.equal(a.cpu(), b)
            assert torch.equal(ev.last_hr_u8.cpu(), w[3])
    assert any(e["graph"] is not None for e in ev._graphs.values()), "no CUDA graph was captured"
    dl, dh = batches[0][0].cuda(), batches[0][1].cuda()
    for _ in range(3):                                      # device-resident inputs: graph keyed by the buffer pair
        assert torch.equal(ev.step(dl, dh).cpu(), want[0][0])
        for a, b in zip(ev.last_maps, want[0][1]):
            assert torch.equal(a.cpu(), b)


def _dataset_with_masks(root, classe, nc, n, seed):
    """S.synthetic_dataset's images (same generator, same draws) written as PNG folders, plus the defect-square masks of the bad
    images under <root>/masks (bad image i -> <stem>_mask.png, 255 inside the square)."""
    rng = np.random.default_rng(seed)
    hr_side, scale = 128, 4
    hrs, lrs, labels, masks = [], [], [], []
    for i in range(n):
        noise = rng.random((hr_side + 4, hr_side + 4, nc))
        c = np.zeros((hr_side + 5, hr_side + 5, nc))
        c[1:, 1:] = noise.cumsum(0).cumsum(1)
        blur = (c[5:, 5:] - c[:-5, 5:] - c[5:, :-5] + c[:-5, :-5]) / 25.0
        blur = (blur - blur.min()) / max(blur.max() - blur.min(), 1e-9)
        img = (blur * 255.0).astype(np.uint8)
        label = 0 if i < n // 2 else 1
        mask = np.zeros((hr_side, hr_side), dtype=np.uint8)
        if label:
            sz = int(rng.integers(16, 33))
            y0, x0 = int(rng.integers(0, hr_side - sz)), int(rng.integers(0, hr_side - sz))
            img[y0:y0 + sz, x0:x0 + sz] = 255 if rng.random() < 0.5 else 0
            mask[y0:y0 + sz, x0:x0 + sz] = 255
        pil = Image.fromarray(img if nc == 3 else img[:, :, 0])
        lr = np.asarray(pil.resize((hr_side // scale, hr_side // scale), Image.LANCZOS))
        lr = lr[:, :, None] if nc == 1 else lr
        split = "good" if label == 0 else "bad"
        for sub, arr in (("HR", img), ("LR_4", lr)):
            d = os.path.join(root, classe, "test", split, sub)
            os.makedirs(d, exist_ok=True)
            Image.fromarray(arr if nc == 3 else arr[:, :, 0]).save(os.path.join(d, f"{i:03d}.png"))
        if label:
            os.makedirs(os.path.join(root, "masks"), exist_ok=True)
            Image.fromarray(mask).save(os.path.join(root, "masks", f"{i:03d}_mask.png"))
        hrs.append(img), lrs.append(lr), labels.append(label), masks.append(mask)
    return np.stack(hrs), np.stack(lrs), np.asarray(labels), np.stack(masks)


def test_evaluate_cli_anomaly_maps_match_oracle(tmp_path, capsys, monkeypatch):
    n = 16
    root = str(tmp_path / "mvtec_128")
    hr, lr, labels, masks = _dataset_with_masks(root, "carpet", 3, n, seed=77)
    assert np.array_equal(hr, S.synthetic_dataset(n, hr=128, nc=3, scale=4, seed=77)[0])
    cfg = O.DrctCfg(num_layers=1)
    sd = O.make_state_dict(cfg, seed=4)
    ckpt = str(tmp_path / "model_best.pt")
    torch.save(sd, ckpt)
    orig = evaluate.setup_opt_drct

    def one_rdg(*a, **k):                                   # a 1-RDG DRCT keeps the test short; the evaluator logic is unchanged
        opt = orig(*a, **k)
        opt.depths, opt.num_heads = (6,), (6,)
        return opt

    monkeypatch.setattr(evaluate, "setup_opt_drct", one_rdg)
    out_dir = str(tmp_path / "out")
    argv = ["--model-type", "drct", "--classe", "carpet", "--scale", "4", "--resolution", "128", "--data-root", root,
            "--checkpoint", ckpt, "--batch-size", "8", "--output-dir", out_dir]
    plain = evaluate.main(argv)
    plain_lines = capsys.readouterr().out.strip().splitlines()
    res = evaluate.main(argv + ["--anomaly-maps", "--mask-dir", os.path.join(root, "masks"), "--save-maps"])
    lines = capsys.readouterr().out.strip().splitlines()
    assert lines[-1] == plain_lines[-1] and lines[-1].startswith("Test AUCs - SSIM(best ws=")
    assert lines[-2].startswith("Map AUCs - max 1-SSIM(ws=11, sigma=4.0): ") and "pixel AUROC 1-SSIM" in lines[-2]
    assert np.array_equal(res["scores"], plain["scores"])
    assert res["map_max"].shape == (n, 2)

    # oracle pipeline in the evaluator's order (good first, then bad; names sorted)
    order = np.argsort(labels, kind="stable")
    x = torch.from_numpy(np.ascontiguousarray(lr[order].transpose(0, 3, 1, 2))).float()
    with torch.no_grad():
        sr = torch.cat([O.drct_forward(sd, x[i:i + 8], cfg) for i in range(0, n, 8)])
    sr_u8 = S.quantize_u8(sr.numpy(), 255.0)
    om = [oracle_maps(sr_u8[k], hr[order][k], 11, 4.0) for k in range(n)]
    y = labels[order]
    mx = np.array([[a.max(), b.max()] for a, b in om])
    assert abs(res["auc_map_ssim"] - S.roc_auc(y, mx[:, 0])) <= 1e-3
    assert abs(res["auc_map_se"] - S.roc_auc(y, mx[:, 1])) <= 1e-3
    mk = masks[order]
    for j, key in ((0, "pixel_auroc_ssim"), (1, "pixel_auroc_se")):
        want = S.roc_auc((mk != 0).ravel().astype(int), np.stack([m[j] for m in om]).ravel())
        assert abs(res[key] - want) <= 1e-3, key

    for split, i in (("good", 0), ("bad", n - 1)):
        for kind in ("ssim", "se"):
            a = np.load(os.path.join(out_dir, "maps", split, f"{i:03d}_{kind}.npy"))
            assert a.shape == (128, 128) and a.dtype == np.float32

    os.remove(os.path.join(root, "masks", f"{n - 1:03d}_mask.png"))
    with pytest.raises(FileNotFoundError, match=f"{n - 1:03d}_mask.png"):
        evaluate.main(argv + ["--mask-dir", os.path.join(root, "masks")])
