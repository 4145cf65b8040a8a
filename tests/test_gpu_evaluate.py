"""GPU end-to-end parity of the batched evaluator (`python -m src.evaluate` path): PNG folders in the reference's
on-disk layout -> AUC line, against the oracle pipeline (oracle forward + quantise + scoring + AUC) on the same files
and checkpoint.  North-star bar: identical AUC to 1e-3 and the same best SSIM window (or an AUC tie)."""
import importlib
import os

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import drct_oracle as O
from oracle import scoring_oracle as S
from gpu_common import PKG, TableModel

pytestmark = pytest.mark.gpu


def _write_dataset(root, classe, nc, n):
    hr, lr, labels = S.synthetic_dataset(n, hr=128, nc=nc, scale=4, seed=77)
    for i in range(n):
        split = "good" if labels[i] == 0 else "bad"
        for sub, arr in (("HR", hr[i]), ("LR_4", lr[i])):
            d = os.path.join(root, classe, "test", split, sub)
            os.makedirs(d, exist_ok=True)
            Image.fromarray(arr if nc == 3 else arr[:, :, 0]).save(os.path.join(d, f"{i:03d}.png"))
    return hr, lr, labels


@pytest.mark.parametrize("classe,nc", [("carpet", 3), ("grid", 1)])
def test_evaluate_cli_matches_oracle(tmp_path, classe, nc, capsys):
    evaluate = importlib.import_module(PKG + ".evaluate")
    n = 24
    root = str(tmp_path / "mvtec_128")
    hr, lr, labels = _write_dataset(root, classe, nc, n)
    cfg = O.DrctCfg(n_colors=nc)
    sd = O.make_state_dict(cfg, seed=4)
    ckpt = str(tmp_path / "model_best.pt")
    torch.save(sd, ckpt)

    res = evaluate.main(["--model-type", "drct", "--classe", classe, "--scale", "4", "--resolution", "128", "--data-root",
                         root, "--checkpoint", ckpt, "--batch-size", "16", "--output-dir", str(tmp_path / "out")])
    line = capsys.readouterr().out.strip().splitlines()[-1]
    assert line.startswith("Test AUCs - SSIM(best ws=")

    # oracle pipeline in the evaluator's order: good first (sorted names), then bad
    order = np.argsort(labels, kind="stable")
    x = torch.from_numpy(np.ascontiguousarray(lr[order].transpose(0, 3, 1, 2))).float()
    with torch.no_grad():
        sr = torch.cat([O.drct_forward(sd, x[i:i + 8], cfg) for i in range(0, n, 8)])
    sr_u8 = S.quantize_u8(sr.numpy(), 255.0)
    wss = S.window_sizes_for(128)
    ssim, mse, psnr = S.score_images(list(sr_u8), list(hr[order]), wss)
    y = labels[order]
    best_ws, a_ssim, a_mse, a_psnr = S.aucs_from_scores(y, ssim, mse, psnr, wss)

    assert abs(res["auc_mse"] - a_mse) <= 1e-3 and abs(res["auc_psnr"] - a_psnr) <= 1e-3
    assert abs(res["auc_ssim"] - a_ssim) <= 1e-3
    if res["best_ws"] != best_ws:       # allowed only as an AUC tie between window sizes
        j, jo = wss.index(res["best_ws"]), wss.index(best_ws)
        assert abs(S.roc_auc(y, 1 - ssim[:, j]) - S.roc_auc(y, 1 - ssim[:, jo])) <= 1e-3
    # per-image scores: bf16 noise flips a few uint8 levels, so compare with a tolerance (SURVEY 7.3)
    assert np.abs(res["scores"][:, :len(wss)] - ssim).max() < 5e-3
    assert np.abs(res["scores"][:, len(wss)] - mse).max() < 1e-3 * max(mse.max(), 1e-3) + 1e-5
    # SR PNGs were written like the reference does (output_dir/<split>/x4/<name>.png)
    assert os.path.isfile(os.path.join(str(tmp_path / "out"), "good", "x4", "000.png"))


def test_evaluator_graph_and_pipelined_paths_match_eager():
    """BatchedEvaluator: the CUDA-graph replay of a step and the double-buffered host-input path (copy stream + persistent
    buffers) return bit-identical score tables and SR images to the eager, synchronous step; launches are still counted."""
    evaluate = importlib.import_module(PKG + ".evaluate")
    drct = importlib.import_module(PKG + ".drct")
    metrics = importlib.import_module(PKG + ".metrics")
    ops = importlib.import_module(PKG + ".ops")
    from gpu_common import DrctOpt

    cfg = O.DrctCfg(num_layers=2)
    sd = O.make_state_dict(cfg, seed=6, affine_jitter=0.05)
    model = drct.DRCT(DrctOpt(layers=2))
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda").eval()
    hr, lr, _ = S.synthetic_dataset(12, hr=128, nc=3, scale=4, seed=5)
    to_t = lambda a: torch.from_numpy(np.ascontiguousarray(a.transpose(0, 3, 1, 2))).float()
    batches = [(to_t(lr[i:i + 4]).pin_memory(), to_t(hr[i:i + 4]).pin_memory()) for i in (0, 4, 8)]
    wss = metrics.window_sizes_for(128)

    eager = evaluate.BatchedEvaluator(model, 255.0, wss)
    eager.use_graph = False
    want = [(eager.step(l, h).cpu(), eager.last_sr_u8.cpu()) for l, h in batches]

    ev = evaluate.BatchedEvaluator(model, 255.0, wss)
    got = [s.cpu() for s in ev.run_pipelined(batches)]                 # two buffer sets: eager warm-up runs, no graph yet
    for (w, _), g in zip(want, got):
        assert torch.equal(w, g)
    n0 = ops.LAUNCHES
    for rep in range(3):                                               # same buffer sets again: capture, then replay
        got = []
        for s in ev.run_pipelined(batches):
            got.append((s.cpu(), ev.last_sr_u8.cpu()))
        for (w, wu8), (g, gu8) in zip(want, got):
            assert torch.equal(w, g) and torch.equal(wu8, gu8)
    assert any(e["graph"] is not None for e in ev._graphs.values()), "no CUDA graph was captured"
    assert ops.LAUNCHES > n0, "graph replays must still be counted as kernel launches"
    dl, dh = batches[0][0].cuda(), batches[0][1].cuda()                # device-resident inputs: graph keyed by the buffer pair
    for _ in range(3):
        assert torch.equal(ev.step(dl, dh).cpu(), want[0][0])


def test_evaluate_cli_drn_l_matches_oracle(tmp_path, capsys):
    """`--model-type drn-l` through the CLI (src/evaluate.py:210-211: the LAST element of DRN's output list is scored)."""
    from oracle import drn_oracle as DO

    evaluate = importlib.import_module(PKG + ".evaluate")
    n = 24
    root = str(tmp_path / "mvtec_128")
    hr, lr, labels = _write_dataset(root, "carpet", 3, n)
    cfg = DO.DrnCfg()
    sd = DO.make_state_dict(cfg, seed=4)
    for k in sd:                                   # keep 80 residual blocks numerically tame with random weights
        if ".body.0." in k or ".body.2." in k:
            sd[k] = sd[k] * 0.5
    ckpt = str(tmp_path / "model_best.pt")
    torch.save(sd, ckpt)
    res = evaluate.main(["--model-type", "drn-l", "--classe", "carpet", "--scale", "4", "--resolution", "128", "--data-root",
                         root, "--checkpoint", ckpt, "--batch-size", "8", "--output-dir", str(tmp_path / "out")])
    assert capsys.readouterr().out.strip().splitlines()[-1].startswith("Test AUCs - SSIM(best ws=")

    order = np.argsort(labels, kind="stable")
    x = torch.from_numpy(np.ascontiguousarray(lr[order].transpose(0, 3, 1, 2))).float()
    with torch.no_grad():
        sr = torch.cat([DO.drn_forward(sd, x[i:i + 8], cfg)[-1] for i in range(0, n, 8)])
    sr_u8 = S.quantize_u8(sr.numpy(), 255.0)
    wss = S.window_sizes_for(128)
    ssim, mse, psnr = S.score_images(list(sr_u8), list(hr[order]), wss)
    y = labels[order]
    best_ws, a_ssim, a_mse, a_psnr = S.aucs_from_scores(y, ssim, mse, psnr, wss)
    assert np.abs(res["scores"][:, :len(wss)] - ssim).max() < 2e-2
    assert np.abs(res["scores"][:, len(wss)] - mse).max() < 2e-2 * max(mse.max(), 1e-3) + 1e-5
    # AUC is a rank statistic: identical unless bf16 noise swaps a near-tie; with 12 x 12 pairs one swap moves it by 0.007
    assert abs(res["auc_mse"] - a_mse) <= 1.5e-2 and abs(res["auc_psnr"] - a_psnr) <= 1.5e-2 and abs(res["auc_ssim"] - a_ssim) <= 1.5e-2


@pytest.mark.timeout(900)
def test_auc_over_1024_images_matches_oracle():
    """SURVEY.md 8d: >= 1024 images for the AUC check.  Synthetic good / bad uint8 pairs (SR = HR + reconstruction noise; bad
    images keep a residual defect) go through BatchedEvaluator batches of 128 + gather_scores; best window and the three AUCs
    must equal the oracle's (numpy SSIM sweep + rank-statistic AUC) on the same uint8 inputs."""
    evaluate = importlib.import_module(PKG + ".evaluate")
    metrics = importlib.import_module(PKG + ".metrics")
    n, bs = 1024, 128
    hr, _, labels = S.synthetic_dataset(n, hr=128, nc=3, scale=4, seed=31)
    rng = np.random.default_rng(7)
    sr = hr.astype(np.int16) + rng.integers(-5, 6, hr.shape)
    for i in np.nonzero(labels)[0]:                       # the SR model "repairs" the defect only partly
        y0, x0 = rng.integers(0, 96, 2)
        sr[i, y0:y0 + 24, x0:x0 + 24] += rng.integers(4, 40)
    sr = np.clip(sr, 0, 255).astype(np.uint8)
    wss = S.window_sizes_for(128)
    ev = evaluate.BatchedEvaluator(TableModel(torch.from_numpy(sr).cuda()), 255.0, wss)
    ev.use_graph = False
    rows, ids = [], []
    for i0 in range(0, n, bs):
        lr_tag = torch.full((bs, 1, 1, 1), float(i0), device="cuda")
        rows.append(ev.step(lr_tag, torch.from_numpy(hr[i0:i0 + bs]).cuda()).clone())
        ids += list(range(i0, i0 + bs))
    table = evaluate.gather_scores(torch.cat(rows), torch.tensor(ids, device="cuda"), n)
    got = metrics.aucs_from_scores(labels, table, wss)
    ssim, mse, psnr = S.score_images(list(sr), list(hr), wss)
    want = S.aucs_from_scores(labels, ssim, mse, psnr, wss)
    assert np.abs(table[:, :len(wss)] - ssim).max() < 1e-5 and np.abs(table[:, len(wss)] - mse).max() < 1e-7
    assert got[0] == want[0], f"best window {got[0]} != oracle {want[0]}"
    assert np.allclose(got[1:], want[1:], atol=1e-3), f"AUCs {got[1:]} vs oracle {want[1:]}"


def test_evaluate_on_test_many_equal_batches_match_eager(tmp_path, capsys, monkeypatch):
    """evaluate_on_test over >= 6 equal-shape batches: CUDA-graph replays reuse ONE static output tensor per buffer set, so the
    per-batch score rows must be copied before the next replay.  The table must equal the eager (no graph) run bit for bit."""
    evaluate = importlib.import_module(PKG + ".evaluate")
    n = 28                                               # batch 4 -> 7 batches per run
    root = str(tmp_path / "mvtec_128")
    _write_dataset(root, "carpet", 3, n)
    cfg = O.DrctCfg(num_layers=1)
    sd = O.make_state_dict(cfg, seed=9)
    ckpt = str(tmp_path / "model_best.pt")
    torch.save(sd, ckpt)
    main_mod = importlib.import_module(PKG + ".main")
    orig = main_mod.setup_opt_drct

    def one_rdg(*a, **k):                                # a 1-RDG DRCT keeps the test short; the evaluator logic is unchanged
        opt = orig(*a, **k)
        opt.depths, opt.num_heads = (6,), (6,)
        return opt

    monkeypatch.setattr(evaluate, "setup_opt_drct", one_rdg)
    argv = ["--model-type", "drct", "--classe", "carpet", "--scale", "4", "--resolution", "128", "--data-root", root,
            "--checkpoint", ckpt, "--batch-size", "4", "--output-dir", str(tmp_path / "out")]
    monkeypatch.setenv("ADSR_CUDA_GRAPH", "0")
    want = evaluate.main(argv)
    monkeypatch.setenv("ADSR_CUDA_GRAPH", "1")
    got = evaluate.main(argv)
    capsys.readouterr()
    assert np.array_equal(got["scores"], want["scores"])
    assert len({tuple(r) for r in got["scores"].round(9).tolist()}) > n // 2     # rows are not copies of one batch


def test_u8_inputs_equal_float_inputs():
    """uint8 HWC batches (decoded PNG bytes; the loader's float scaling runs on the device) give bit-identical scores and SR
    images to the float NCHW tensors the reference's loader yields (rgb_range 255)."""
    evaluate, drct, metrics, ops = (importlib.import_module(f"{PKG}.{m}") for m in ("evaluate", "drct", "metrics", "ops"))
    from gpu_common import DrctOpt

    cfg = O.DrctCfg(num_layers=1)
    sd = O.make_state_dict(cfg, seed=6)
    model = drct.DRCT(DrctOpt(layers=1))
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda").eval()
    hr, lr, _ = S.synthetic_dataset(6, hr=128, nc=3, scale=4, seed=15)
    lr_u8, hr_u8 = torch.from_numpy(lr).cuda(), torch.from_numpy(hr).cuda()
    to_t = lambda a: torch.from_numpy(np.ascontiguousarray(a.transpose(0, 3, 1, 2))).float().mul_(255.0 / 255)
    got_f = ops.u8_to_float(lr_u8, 255.0)
    assert torch.equal(got_f.cpu(), to_t(lr))
    assert torch.equal(ops.u8_to_float(lr_u8, 1.0).cpu(), torch.from_numpy(np.ascontiguousarray(lr.transpose(0, 3, 1, 2))).float().mul_(1.0 / 255))
    wss = metrics.window_sizes_for(128)
    ev = evaluate.BatchedEvaluator(model, 255.0, wss)
    ev.use_graph = False
    a = ev.step(to_t(lr).cuda(), to_t(hr).cuda()).cpu()
    a_sr = ev.last_sr_u8.cpu()
    b = ev.step(lr_u8, hr_u8).cpu()
    assert torch.equal(a, b) and torch.equal(a_sr, ev.last_sr_u8.cpu())
