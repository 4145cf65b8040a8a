"""GPU tests of the localisation metrics (csrc/localisation.cu through metrics.LocalisationAccumulator / au_pro / pixel_auroc): pixel
AUROC against sklearn (|d| <= 1e-9) and AU-PRO against oracle/localisation_oracle.py (|d| <= 1e-7) on ties, smoothed maps, negative
scores and -0.0, tiny and border regions, defect-free and all-defect images, mixed image sizes and more than 2^24 pixels; errors;
determinism and batch independence; then the `--au-pro` option of the evaluator end to end."""
import importlib
import os

import numpy as np
import pytest
import torch
from scipy.ndimage import gaussian_filter

from gpu_common import PKG
from oracle import drct_oracle as O
from oracle import localisation_oracle as L
from test_gpu_anomaly_maps import _dataset_with_masks

pytestmark = pytest.mark.gpu

metrics = importlib.import_module(PKG + ".metrics")
evaluate = importlib.import_module(PKG + ".evaluate")

ALPHAS = (0.3, 1.0, 0.05)


def _device(maps):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in maps]


def check(maps, masks, alphas=ALPHAS):
    """Device metrics of host maps / masks (list input) against sklearn and the oracle, for every alpha."""
    want_auc = L.pixel_auroc(maps, masks)
    curve = L.curve(maps, masks)
    for alpha in alphas:
        acc = metrics.LocalisationAccumulator(1)
        acc.append([_device(maps)], masks)
        (auc, pro), = acc.finish(alpha)
        assert abs(auc - want_auc) <= 1e-9, (alpha, auc, want_auc)
        assert abs(pro - L.area(*curve, alpha)) <= 1e-7, (alpha, pro, L.area(*curve, alpha))


def _blob_masks(rng, n, h, w, p_defect=0.7):
    masks = []
    for _ in range(n):
        m = np.zeros((h, w), np.uint8)
        if rng.random() < p_defect:
            for _ in range(rng.integers(1, 4)):
                y, x = rng.integers(0, h), rng.integers(0, w)
                m[y:y + rng.integers(1, max(2, h // 3)), x:x + rng.integers(1, max(2, w // 3))] = 255
            yy, xx = np.mgrid[:h, :w]
            cy, cx, r = rng.integers(0, h), rng.integers(0, w), rng.integers(2, 8)
            m[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = 255
        masks.append(m)
    if not any(m.any() for m in masks):
        masks[0][0, 0] = 255
    return masks


def test_many_ties():
    rng = np.random.default_rng(0)
    masks = _blob_masks(rng, 12, 64, 64)
    maps = [(np.round(rng.random((64, 64)) * 12 + 4 * (m != 0)) / 8).astype(np.float32) for m in masks]
    check(maps, masks)


def test_smoothed_maps():
    rng = np.random.default_rng(1)
    masks = _blob_masks(rng, 10, 96, 80)
    maps = [gaussian_filter((rng.random((96, 80)) + 0.8 * (m != 0)).astype(np.float32), 4.0, mode="reflect") for m in masks]
    check(maps, masks)


def test_negative_scores_and_negative_zero():
    rng = np.random.default_rng(2)
    masks = _blob_masks(rng, 6, 40, 40)
    maps = []
    for m in masks:
        a = (rng.integers(-3, 4, (40, 40)) / 2.0).astype(np.float32)
        a[rng.random((40, 40)) < 0.3] = -0.0
        a[rng.random((40, 40)) < 0.1] = np.float32(-3.0e38)        # the most negative keys (sklearn refuses infinities)
        maps.append(a)
    assert any(np.signbit(a[a == 0]).any() for a in maps)
    check(maps, masks)
    # -0.0 and +0.0 are one score: flipping every zero's sign changes nothing
    flipped = [np.where(a == 0, np.float32(0.0), a) for a in maps]
    acc1, acc2 = metrics.LocalisationAccumulator(1), metrics.LocalisationAccumulator(1)
    acc1.append([_device(maps)], masks)
    acc2.append([_device(flipped)], masks)
    assert acc1.finish() == acc2.finish()


def test_single_pixel_and_border_regions():
    rng = np.random.default_rng(3)
    masks = []
    for i in range(5):
        m = np.zeros((32, 48), np.uint8)
        m[rng.integers(0, 32, 6), rng.integers(0, 48, 6)] = 1       # single pixels (some may touch diagonally)
        m[0, :5] = m[-1, -3:] = m[10:14, 0] = m[:2, -1] = 1          # regions on every border
        masks.append(m)
    maps = [(rng.random((32, 48)) + 0.3 * (m != 0)).astype(np.float32) for m in masks]
    check(maps, masks)


def test_defect_free_and_all_defect_images():
    rng = np.random.default_rng(4)
    masks = [np.zeros((32, 32), np.uint8), np.ones((32, 32), np.uint8) * 255, np.zeros((32, 32), np.uint8)]
    masks[2][5:9, 20:30] = 1
    maps = [np.round(rng.random((32, 32)) * 50).astype(np.float32) / 10 for _ in masks]
    check(maps, masks)


def test_mixed_image_sizes_and_tensor_input():
    rng = np.random.default_rng(5)
    shapes = [(17, 33), (64, 40), (5, 7), (128, 96)]
    masks = [_blob_masks(rng, 1, h, w, 1.0)[0] for h, w in shapes]
    maps = [(np.round(rng.random(s) * 30) / 7).astype(np.float32) for s in shapes]
    check(maps, masks)
    # au_pro / pixel_auroc: one [N, H, W] tensor or a list, same numbers
    same = [np.zeros((24, 24), np.uint8) for _ in range(4)]
    same[1][3:8, 3:8] = same[3][20:, 10:12] = 1
    stack = np.stack([rng.random((24, 24)).astype(np.float32) for _ in range(4)])
    d = torch.from_numpy(stack).cuda()
    assert metrics.au_pro(d, np.stack(same)) == metrics.au_pro(list(d.unbind(0)), same)
    assert abs(metrics.au_pro(d, same, 0.3) - L.au_pro(list(stack), same, 0.3)) <= 1e-7
    got = metrics.pixel_auroc(d, np.stack(same))
    assert abs(got - metrics.pixel_auroc(stack, np.stack(same))) <= 1e-9      # host path, unchanged
    with pytest.raises(ValueError):
        metrics.pixel_auroc(d, np.stack(same)[:, :16])


def test_more_than_2_pow_24_pixels():
    """17.3 M pixels: prefix counts past 2^24 (where fp32 counting would lose pixels), 4 radix passes over many tiles."""
    rng = np.random.default_rng(6)
    n_img, h, w = 264, 256, 256
    masks = np.zeros((n_img, h, w), np.uint8)
    for i in range(0, n_img, 3):
        y, x = rng.integers(0, h - 40, 2)
        masks[i, y:y + rng.integers(4, 40), x:x + rng.integers(4, 40)] = 1
    maps = (np.round(rng.random((n_img, h, w)) * 4000) / 1000 + 0.5 * masks).astype(np.float32)
    assert maps.size > 2 ** 24
    acc = metrics.LocalisationAccumulator(1)
    for s in range(0, n_img, 64):
        acc.append([torch.from_numpy(maps[s:s + 64]).cuda()], masks[s:s + 64])
    (auc, pro), = acc.finish(0.3)
    assert abs(auc - L.pixel_auroc(list(maps), list(masks))) <= 1e-9
    assert abs(pro - L.au_pro(list(maps), list(masks), 0.3)) <= 1e-7


def test_errors():
    m = np.zeros((2, 16, 16), np.uint8)
    m[1, 4:6, 4:6] = 1
    a = torch.rand(2, 16, 16, device="cuda")
    bad = a.clone()
    bad[0, 3, 3] = float("nan")
    with pytest.raises(ValueError, match="NaN"):
        metrics.au_pro(bad, m)
    with pytest.raises(ValueError, match="defect region"):
        metrics.au_pro(a, np.zeros_like(m))                           # R == 0
    with pytest.raises(ValueError, match="defect-free"):
        metrics.au_pro(a, np.ones_like(m))                            # N_ok == 0
    with pytest.raises(ValueError, match="fpr_limit"):
        metrics.au_pro(a, m, 1.5)
    with pytest.raises(ValueError):
        metrics.au_pro(a, m[:, :8])                                   # shape mismatch
    with pytest.raises(TypeError):
        metrics.au_pro(a.double(), m)


def test_bitwise_deterministic_and_batch_independent():
    rng = np.random.default_rng(7)
    n = 128
    masks = _blob_masks(rng, n, 64, 64)
    ssim = np.stack([gaussian_filter(rng.random((64, 64)).astype(np.float32), 2.0) for _ in range(n)])
    se = (np.round(rng.random((n, 64, 64)) * 100) / 100).astype(np.float32)
    d_ssim, d_se = torch.from_numpy(ssim).cuda(), torch.from_numpy(se).cuda()
    results = []
    for bs in (8, 64, 128, 8):
        acc = metrics.LocalisationAccumulator(2)
        for s in range(0, n, bs):
            acc.append([d_ssim[s:s + bs], d_se[s:s + bs]], masks[s:s + bs])
        results.append(acc.finish(0.3))
    assert all(r == results[0] for r in results), results
    for j, maps in enumerate((ssim, se)):
        assert abs(results[0][j][0] - L.pixel_auroc(list(maps), masks)) <= 1e-9
        assert abs(results[0][j][1] - L.au_pro(list(maps), masks, 0.3)) <= 1e-7


# ------------------------------------------------------------------------------------------------------------- evaluator
def test_evaluate_cli_au_pro_matches_oracle(tmp_path, capsys, monkeypatch):
    n = 16
    root = str(tmp_path / "mvtec_128")
    _, _, labels, masks = _dataset_with_masks(root, "carpet", 3, n, seed=77)
    sd = O.make_state_dict(O.DrctCfg(num_layers=1), seed=4)
    ckpt = str(tmp_path / "model_best.pt")
    torch.save(sd, ckpt)
    orig = evaluate.setup_opt_drct

    def one_rdg(*a, **k):
        opt = orig(*a, **k)
        opt.depths, opt.num_heads = (6,), (6,)
        return opt

    monkeypatch.setattr(evaluate, "setup_opt_drct", one_rdg)
    out_dir = str(tmp_path / "out")
    mask_dir = os.path.join(root, "masks")
    argv = ["--model-type", "drct", "--classe", "carpet", "--scale", "4", "--resolution", "128", "--data-root", root,
            "--checkpoint", ckpt, "--batch-size", "8", "--output-dir", out_dir, "--mask-dir", mask_dir]
    plain = evaluate.main(argv)
    plain_lines = capsys.readouterr().out.strip().splitlines()
    res = evaluate.main(argv + ["--au-pro", "--save-maps"])
    lines = capsys.readouterr().out.strip().splitlines()

    # without --au-pro: the parent's two last lines, no PRO line; with it: the PRO line right before them
    assert not any(l.startswith("Map PRO") for l in plain_lines) and "au_pro_ssim" not in plain
    assert plain_lines[-1].startswith("Test AUCs - SSIM(best ws=")
    assert plain_lines[-2] == (f"Map AUCs - max 1-SSIM(ws=11, sigma=4.0): {plain['auc_map_ssim']:.4f}, max SE: {plain['auc_map_se']:.4f}, "
                               f"pixel AUROC 1-SSIM: {plain['pixel_auroc_ssim']:.4f}, pixel AUROC SE: {plain['pixel_auroc_se']:.4f}")
    assert lines[-2:] == plain_lines[-2:]
    assert lines[-3] == f"Map PRO - AU-PRO@0.3 1-SSIM: {res['au_pro_ssim']:.4f}, AU-PRO@0.3 SE: {res['au_pro_se']:.4f}"
    assert res["pro_fpr_limit"] == 0.3

    # the saved maps, in the evaluator's order (good first, then bad; names sorted), against the oracle and sklearn
    order = np.argsort(labels, kind="stable")
    mk = [masks[i] for i in order]
    for kind in ("ssim", "se"):
        maps = [np.load(os.path.join(out_dir, "maps", "good" if labels[i] == 0 else "bad", f"{i:03d}_{kind}.npy")) for i in order]
        assert abs(res[f"au_pro_{kind}"] - L.au_pro(maps, mk, 0.3)) <= 1e-7, kind
        assert abs(res[f"pixel_auroc_{kind}"] - L.pixel_auroc(maps, mk)) <= 1e-9, kind
        assert res[f"pixel_auroc_{kind}"] == plain[f"pixel_auroc_{kind}"]

    res = evaluate.main(argv + ["--au-pro", "0.1"])
    assert capsys.readouterr().out.strip().splitlines()[-3].startswith("Map PRO - AU-PRO@0.1 1-SSIM: ")
    assert res["pro_fpr_limit"] == 0.1
