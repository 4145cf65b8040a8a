"""GPU tests of the MSGMS map (csrc/anomaly_maps.cu adsr_gms_map): against the numpy reference oracle/gms_oracle.py, determinism
and batch independence, rejections; then BatchedEvaluator(gms=True) on its eager, graph and pipelined paths and `--gms-map` on the
command line, with masks and with calibration."""
import importlib
import os
import shutil

import numpy as np
import pytest
import torch
from PIL import Image

from gpu_common import PKG, DrctOpt
from oracle import drct_oracle as O
from oracle import gms_oracle as G
from oracle import scoring_oracle as S

pytestmark = pytest.mark.gpu

ops = importlib.import_module(PKG + ".ops")
metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")
_abi = importlib.import_module(PKG + "._abi")


def _pairs(h, w, c, seed):
    """4 pairs: random SR / HR, an identical pair, a constant HR, SR = HR + noise."""
    rng = np.random.default_rng(seed)
    hr = rng.integers(0, 256, (4, h, w, c), dtype=np.uint8)
    sr = rng.integers(0, 256, (4, h, w, c), dtype=np.uint8)
    sr[1] = hr[1]
    hr[2] = 97
    sr[3] = np.clip(hr[3].astype(np.int16) + rng.integers(-6, 7, (h, w, c)), 0, 255).astype(np.uint8)
    return sr, hr


@pytest.mark.parametrize("sigma", [0.0, 4.0])
@pytest.mark.parametrize("h,w,c", [(128, 128, 3), (128, 128, 1), (64, 96, 3), (100, 84, 1), (256, 256, 3), (8, 8, 1)])
def test_gms_map_matches_oracle(h, w, c, sigma):
    if int(4 * sigma + 0.5) >= min(h, w):
        pytest.skip("the Gaussian radius does not fit the image")
    sr, hr = _pairs(h, w, c, seed=h + w + c)
    launches = ops.LAUNCHES
    m, mx = (t.cpu().numpy() for t in ops.gms_map(torch.from_numpy(sr).cuda(), torch.from_numpy(hr).cuda(), sigma))
    assert ops.LAUNCHES - launches == (6 if sigma > 0 else 4)
    assert m.shape == (4, h, w) and m.dtype == np.float32 and mx.shape == (4,) and mx.dtype == np.float64
    for i in range(4):
        assert np.abs(m[i] - G.gms_map(sr[i], hr[i], sigma)).max() <= 1e-5, f"image {i}"
    assert not m[1].any(), "an identical pair must give an all-zero map"
    assert np.array_equal(mx, m.reshape(4, -1).max(1).astype(np.float64))


@pytest.mark.parametrize("sigma", [0.0, 4.0])
def test_deterministic_and_batch_independent(sigma):
    rng = np.random.default_rng(12)
    sr = torch.from_numpy(rng.integers(0, 256, (6, 100, 84, 3), dtype=np.uint8)).cuda()
    hr = torch.from_numpy(rng.integers(0, 256, (6, 100, 84, 3), dtype=np.uint8)).cuda()
    first = [t.clone() for t in ops.gms_map(sr, hr, sigma)]
    for a, b in zip(first, ops.gms_map(sr, hr, sigma)):
        assert torch.equal(a, b)
    for i in (0, 3, 5):
        for a, b in zip(first, ops.gms_map(sr[i:i + 1], hr[i:i + 1], sigma)):
            assert torch.equal(a[i:i + 1], b)


def test_rejections():
    rng = np.random.default_rng(2)
    img = lambda h, w, c: torch.from_numpy(rng.integers(0, 256, (2, h, w, c), dtype=np.uint8)).cuda()
    a, b = img(16, 16, 3), img(16, 16, 3)
    for x, y in ((img(7, 16, 3), img(7, 16, 3)), (img(16, 7, 1), img(16, 7, 1)), (img(16, 16, 2), img(16, 16, 2))):
        with pytest.raises(RuntimeError, match="adsr_gms_map"):
            ops.gms_map(x, y)                                   # H or W < 8, two channels
    with pytest.raises(RuntimeError, match="adsr_gms_map"):
        ops.gms_map(a, b, float("nan"))
    with pytest.raises(RuntimeError, match="adsr_gms_map"):
        ops.gms_map(a, b, 4.0)                                  # Gaussian radius 16 >= min(H, W)
    need = ops.gms_workspace_bytes(2, 16, 16)
    out = (torch.empty(2, 16, 16, device="cuda"), torch.empty(2, dtype=torch.float64, device="cuda"),
           torch.empty(need - 4, dtype=torch.uint8, device="cuda"))
    with pytest.raises(ValueError, match="workspace"):
        ops.gms_map(a, b, 1.0, out=out)                         # smoothing with too small a workspace
    st = _abi.stream_ptr()
    assert _abi.lib().adsr_gms_map(a.data_ptr(), b.data_ptr(), 2, 16, 16, 3, 1.0, out[0].data_ptr(), out[1].data_ptr(), 0, st) == 1
    assert _abi.lib().adsr_gms_map(0, 0, 1 << 15, 256, 256, 3, 0.0, 0, 0, 0, st) == 1      # B H W >= 2^31
    ops.gms_map(a, b, 1.0, out=out[:2] + (torch.empty(need, dtype=torch.uint8, device="cuda"),))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------- evaluator
def _small_drct(seed=6):
    drct = importlib.import_module(PKG + ".drct")
    sd = O.make_state_dict(O.DrctCfg(num_layers=1), seed=seed)
    model = drct.DRCT(DrctOpt(layers=1))
    model.load_state_dict(sd, strict=True)
    return model.to("cuda").eval()


def test_evaluator_gms_graph_and_pipelined_match_eager():
    model = _small_drct()
    hr, lr, _ = S.synthetic_dataset(12, hr=128, nc=3, scale=4, seed=5)
    to_t = lambda a: torch.from_numpy(np.ascontiguousarray(a.transpose(0, 3, 1, 2))).float()
    batches = [(to_t(lr[i:i + 4]).pin_memory(), to_t(hr[i:i + 4]).pin_memory()) for i in (0, 4, 8)]
    wss = metrics.window_sizes_for(128)
    maps = (11, 4.0)

    eager = evaluate.BatchedEvaluator(model, 255.0, wss, maps=maps, gms=True)
    eager.use_graph = False
    two = evaluate.BatchedEvaluator(model, 255.0, wss, maps=maps)
    two.use_graph = False
    want = []
    for l, h in batches:
        s = eager.step(l, h).cpu()
        got = [t.cpu() for t in eager.last_maps]
        assert len(got) == 4 and got[3].shape == (4, 3)
        gms, gms_max = ops.gms_map(eager.last_sr_u8, eager.last_hr_u8, maps[1])   # the step's own uint8 SR / HR
        assert torch.equal(gms.cpu(), got[2]) and torch.equal(gms_max.cpu(), got[3][:, 2])
        assert torch.equal(two.step(l, h).cpu(), s)                               # the maps-only evaluator: same table and maps
        for a, b in zip(two.last_maps[:2], got[:2]):
            assert torch.equal(a.cpu(), b)
        assert torch.equal(two.last_maps[2].cpu(), got[3][:, :2])
        want.append((s, got))

    ev = evaluate.BatchedEvaluator(model, 255.0, wss, maps=maps, gms=True)
    for rep in range(4):                                        # eager warm-up, capture, then replays
        for s, w in zip(ev.run_pipelined(batches), want):
            assert torch.equal(s.cpu(), w[0])
            for a, b in zip(ev.last_maps, w[1]):
                assert torch.equal(a.cpu(), b)
    assert any(e["graph"] is not None for e in ev._graphs.values()), "no CUDA graph was captured"
    dl, dh = batches[0][0].cuda(), batches[0][1].cuda()
    for _ in range(3):                                          # device-resident inputs: graph keyed by the buffer pair
        assert torch.equal(ev.step(dl, dh).cpu(), want[0][0])
        for a, b in zip(ev.last_maps, want[0][1]):
            assert torch.equal(a.cpu(), b)
    with pytest.raises(ValueError, match="needs maps"):
        evaluate.BatchedEvaluator(model, 255.0, wss, gms=True)


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


def _cli_setup(tmp_path, monkeypatch, seed):
    n = 16
    root = str(tmp_path / "mvtec_128")
    hr, lr, labels, masks = _dataset_with_masks(root, "carpet", 3, n, seed=seed)
    sd = O.make_state_dict(O.DrctCfg(num_layers=1), seed=4)
    ckpt = str(tmp_path / "model_best.pt")
    torch.save(sd, ckpt)
    orig = evaluate.setup_opt_drct

    def one_rdg(*a, **k):                                       # a 1-RDG DRCT keeps the test short; the evaluator logic is unchanged
        opt = orig(*a, **k)
        opt.depths, opt.num_heads = (6,), (6,)
        return opt

    monkeypatch.setattr(evaluate, "setup_opt_drct", one_rdg)
    argv = ["--model-type", "drct", "--classe", "carpet", "--scale", "4", "--resolution", "128", "--data-root", root,
            "--checkpoint", ckpt, "--batch-size", "8", "--output-dir", str(tmp_path / "out")]
    return root, argv, sd, hr, lr, labels, masks


def test_evaluate_cli_gms_map_matches_oracle(tmp_path, capsys, monkeypatch):
    root, argv, sd, hr, lr, labels, masks = _cli_setup(tmp_path, monkeypatch, seed=77)
    n, out_dir, mask_dir = len(labels), str(tmp_path / "out"), os.path.join(root, "masks")
    plain = evaluate.main(argv)
    plain_lines = capsys.readouterr().out.strip().splitlines()
    flags = ["--mask-dir", mask_dir, "--au-pro", "--pr-metrics", "--save-maps", "--save-segmentation"]
    two = evaluate.main(argv + flags)
    two_lines = capsys.readouterr().out.strip().splitlines()
    res = evaluate.main(argv + flags + ["--gms-map"])
    lines = capsys.readouterr().out.strip().splitlines()
    assert lines[-1] == plain_lines[-1] and lines[-1].startswith("Test AUCs - SSIM(best ws=")
    assert np.array_equal(res["scores"], plain["scores"])
    assert res["map_max"].shape == (n, 3) and np.array_equal(res["map_max"][:, :2], two["map_max"])
    for key in ("auc_map", "pixel_auroc", "au_pro", "pixel_ap", "f1_max", "f1_threshold"):
        assert res[f"{key}_ssim"] == two[f"{key}_ssim"] and res[f"{key}_se"] == two[f"{key}_se"], key
        assert f"{key}_gms" in res and f"{key}_gms" not in two, key

    # every Map line is that of the maps-only run with the MSGMS entry right after each SE entry
    f = lambda key: f"{res[key]:.4f}"
    inserts = [(f"max SE: {f('auc_map_se')}", f"max MSGMS: {f('auc_map_gms')}"),
               (f"pixel AUROC SE: {f('pixel_auroc_se')}", f"pixel AUROC MSGMS: {f('pixel_auroc_gms')}"),
               (f"pixel AP SE: {f('pixel_ap_se')}", f"pixel AP MSGMS: {f('pixel_ap_gms')}"),
               (f"F1-max SE: {f('f1_max_se')} (thr {res['f1_threshold_se']:g})",
                f"F1-max MSGMS: {f('f1_max_gms')} (thr {res['f1_threshold_gms']:g})"),
               (f"AU-PRO@0.3 SE: {f('au_pro_se')}", f"AU-PRO@0.3 MSGMS: {f('au_pro_gms')}")]
    want = [l for l in two_lines if l.startswith("Map ")]
    assert [l.split(" - ")[0] for l in want] == ["Map PR", "Map PRO", "Map AUCs"]
    for se, gms in inserts:
        assert sum(l.count(se) for l in want) == 1, se
        want = [l.replace(se, f"{se}, {gms}") for l in want]
    assert [l for l in lines if l.startswith("Map ")] == want

    # oracle pipeline in the evaluator's order (good first, then bad; names sorted)
    order = np.argsort(labels, kind="stable")
    cfg = O.DrctCfg(num_layers=1)
    x = torch.from_numpy(np.ascontiguousarray(lr[order].transpose(0, 3, 1, 2))).float()
    with torch.no_grad():
        sr = torch.cat([O.drct_forward(sd, x[i:i + 8], cfg) for i in range(0, n, 8)])
    sr_u8 = S.quantize_u8(sr.numpy(), 255.0)
    om = [G.gms_map(sr_u8[k], hr[order][k], 4.0) for k in range(n)]
    y = labels[order]
    assert abs(res["auc_map_gms"] - S.roc_auc(y, [m.max() for m in om])) <= 1e-3
    want = S.roc_auc((masks[order] != 0).ravel().astype(int), np.stack(om).ravel())
    assert abs(res["pixel_auroc_gms"] - want) <= 1e-3

    for split, i in (("good", 0), ("bad", n - 1)):
        a = np.load(os.path.join(out_dir, "maps", split, f"{i:03d}_gms.npy"))
        assert a.shape == (128, 128) and a.dtype == np.float32
        png = np.array(Image.open(os.path.join(out_dir, "segmentation", split, f"{i:03d}_gms.png")))
        assert png.shape == (128, 128) and png.dtype == np.uint8 and set(np.unique(png)) <= {0, 255}
        assert np.array_equal(png == 255, a >= np.float32(res["f1_threshold_gms"]))


def test_evaluate_cli_gms_calibration(tmp_path, capsys, monkeypatch):
    q = 0.99
    root, argv, sd, hr, lr, labels, masks = _cli_setup(tmp_path, monkeypatch, seed=78)
    other = str(tmp_path / "other")
    _dataset_with_masks(other, "carpet", 3, 12, seed=79)        # its 6 good images become the defect-free calibration split
    cal_dir = os.path.join(root, "carpet", "train", "good")
    shutil.move(os.path.join(other, "carpet", "test", "good"), cal_dir)
    built = []

    class Recording(evaluate.BatchedEvaluator):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            built.append(self)

    monkeypatch.setattr(evaluate, "BatchedEvaluator", Recording)
    mask_dir = os.path.join(root, "masks")
    base = evaluate.main(argv + ["--mask-dir", mask_dir, "--calibration-dir", cal_dir, "--calibration-quantile", str(q)])
    base_lines = capsys.readouterr().out.strip().splitlines()
    res = evaluate.main(argv + ["--mask-dir", mask_dir, "--calibration-dir", cal_dir, "--calibration-quantile", str(q), "--gms-map",
                                "--save-calibrated-masks"])
    lines = capsys.readouterr().out.strip().splitlines()

    # the calibration maps, recomputed from the evaluator's own SR output: the threshold is their numpy quantile
    ev = evaluate.BatchedEvaluator(built[-1].model, 255.0, built[-1].window_sizes, maps=(11, 4.0))
    ev.use_graph = False
    pairs = [evaluate.load_pair(h, l, 4, 3, 255.0, raw_u8=True) for h, l in zip(*evaluate.scan_split(cal_dir, 4))]
    with torch.no_grad():
        ev.step(torch.stack([p[0] for p in pairs]), torch.stack([p[1] for p in pairs]))
    cal_gms, cal_max = (t.cpu().numpy() for t in ops.gms_map(ev.last_sr_u8, ev.last_hr_u8, 4.0))
    t_px = res["calib_pixel_threshold_gms"]
    assert t_px == float(np.quantile(cal_gms.astype(np.float64), q, method="inverted_cdf"))
    assert res["calib_image_threshold_gms"] == float(np.quantile(cal_max, q, method="inverted_cdf"))
    for k in ("pixel_threshold", "image_threshold", "image_tpr", "image_fpr", "pixel_precision", "pixel_recall", "pixel_fpr",
              "pixel_f1", "pixel_iou", "pixel_pro"):
        assert f"calib_{k}_gms" in res and f"calib_{k}_gms" not in base, k
        assert res[f"calib_{k}_ssim"] == base[f"calib_{k}_ssim"] and res[f"calib_{k}_se"] == base[f"calib_{k}_se"], k
    cal_line = next(l for l in lines if l.startswith("Map CAL - "))
    base_cal = next(l for l in base_lines if l.startswith("Map CAL - "))
    assert cal_line.startswith(base_cal + "; MSGMS t_px ")
    assert f"MSGMS t_px {t_px:g}, t_img {res['calib_image_threshold_gms']:g}" in cal_line
    png = np.array(Image.open(os.path.join(str(tmp_path / "out"), "calibrated", "bad", f"{len(labels) - 1:03d}_gms.png")))
    assert png.shape == (128, 128) and set(np.unique(png)) <= {0, 255}
