"""GPU parity of the DRN path: DRN-only kernels against torch fp32, and the full DRN forward against the reference's own
outputs (tests/golden/drn_*.npz) and the oracle."""
import copy
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import drn_oracle as DO
from oracle import hotpath_oracle as R
from gpu_common import mod

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 2e-2                      # golden cases; the seeded n_blocks = 6 forwards carry measured bounds (DRN_TOL)
# about twice the largest max|dSR|/rgb_range measured on a B200 (1000 W power limit): 6.9e-4 at 32 px LR, 7.5e-4 at 64 px
DRN_TOL = {32: 1.5e-3, 64: 1.5e-3}


class DrnOpt:
    def __init__(self, cfg: DO.DrnCfg):
        self.scale = [2 ** (i + 1) for i in range(cfg.phase)]
        self.n_blocks, self.n_feats, self.n_colors = cfg.n_blocks, cfg.n_feats, cfg.n_colors
        self.rgb_range, self.negval = 255, cfg.negval


def _model(cfg, sd):
    drn = mod("drn")
    m = drn.DRN(DrnOpt(cfg))
    assert set(m.state_dict().keys()) == set(sd.keys())
    res = m.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    return m.to(DEV).eval()


@pytest.mark.parametrize("nc,scale", [(3, 4), (1, 4), (3, 2)])
def test_bicubic_affine(nc, scale):
    ops = mod("ops")
    torch.manual_seed(nc)
    x = torch.rand(2, nc, 12, 20, device=DEV) * 255
    mat = torch.eye(nc, device=DEV) + 0.01 * torch.randn(nc, nc, device=DEV)
    bias = torch.randn(nc, device=DEV) * 10
    out = torch.empty(2, nc, 12 * scale, 20 * scale, device=DEV)
    ops.bicubic_affine(x, scale, mat.contiguous(), bias, out)
    want = F.conv2d(F.interpolate(x, scale_factor=scale, mode="bicubic", align_corners=False), mat.view(nc, nc, 1, 1), bias)
    assert (out - want).abs().max() < 2e-3


def _verdict(tag, got, ref, shortcut=None, kernel="conv"):
    b, rb = R.TOL[kernel]
    v = R.compare(got.cpu(), ref, None if shortcut is None else shortcut.cpu(), b=b, rms_b=rb)
    print(f"[drn] {tag}: {v}")
    assert v.ok, f"{tag}: {v}"


def test_conv3x3_small_two_destinations():
    ops = mod("ops")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 3, 16, 24, generator=g)
    w, b = torch.randn(20, 3, 3, 3, generator=g) * 0.3, torch.randn(20, generator=g)
    o1 = torch.full((2 * 16 * 24, 32), 7.0, device=DEV, dtype=torch.bfloat16)
    o2 = torch.full((2 * 16 * 24, 48), 7.0, device=DEV, dtype=torch.bfloat16)
    ops.conv3x3_small(x.to(DEV), w.to(DEV), b.to(DEV), 20, o1, o2, 20)
    torch.cuda.synchronize()
    ref = R.conv3x3_small(x, w, b)
    _verdict("conv3x3_small out1", o1[:, :20], ref)
    assert torch.equal(o1[:, :20], o2[:, 20:40])
    assert float(o1[:, 20:].float().abs().max()) == 0.0
    assert float((o2[:, :20].float() - 7).abs().max()) == 0.0 and float((o2[:, 40:].float() - 7).abs().max()) == 0.0


def test_channel_mean_and_ca_scale():
    ops = mod("ops")
    g = torch.Generator().manual_seed(1)
    B, HW, C, Cr = 3, 1024, 80, 5
    t2 = (torch.randn(B * HW, C, generator=g) + torch.randn(B, 1, C, generator=g).repeat_interleave(HW, 0).view(-1, C)).to(torch.bfloat16)
    x = (torch.randn(B * HW, C, generator=g) * 4.0).to(torch.bfloat16)        # the shortcut dominates the output
    mlp = [torch.randn(Cr, C, generator=g) * 0.3, torch.randn(Cr, generator=g), torch.randn(C, Cr, generator=g) * 0.3,
           torch.randn(C, generator=g)]
    n_parts = ops.channel_mean_slices(HW)
    parts = torch.full((B * n_parts + 2, C), float("nan"), device=DEV)         # one guard row: written rows only
    scale = torch.empty(B, C, device=DEV)
    mean = torch.empty(B, C, device=DEV)
    t2d, xd, mlpd = t2.to(DEV), x.to(DEV), [t.to(DEV) for t in mlp]
    ops.channel_sums(t2d, B, HW, C, parts[1:-1])
    ops.channel_mean_parts(parts[1:-1], B, n_parts, C, HW, scale, *mlpd, Cr)
    ops.channel_mean(t2d, B, HW, C, mean)
    torch.cuda.synchronize()
    assert bool(torch.isnan(parts[0]).all()) and bool(torch.isnan(parts[-1]).all()) and bool(torch.isfinite(parts[1:-1]).all())
    want_mean = R.channel_mean(t2, B, HW, C)
    assert float((R.channel_mean_parts(parts[1:-1].cpu(), B, n_parts, C, HW) - want_mean).abs().max()) < 1e-5
    assert float((mean.cpu() - want_mean).abs().max()) < 1e-5
    want_s = R.ca_scale(want_mean, *mlp)
    assert float((scale.cpu() - want_s).abs().max()) < 1e-5
    out = torch.empty(B * HW, C, device=DEV, dtype=torch.bfloat16)
    ops.rcab_ca_scale(t2d, xd, out, scale, *mlpd, B, HW, C, 0)                  # scales given
    out2 = torch.empty_like(out)
    ops.rcab_ca_scale(t2d, xd, out2, mean, *mlpd, B, HW, C, Cr)                 # means given: the MLP runs first
    torch.cuda.synchronize()
    _verdict("rcab_ca_scale", out, R.rcab_ca_scale(t2, x, scale.cpu(), B, HW, C), x)
    assert torch.equal(out, out2)


def test_conv_into_channel_slice():
    ops = mod("ops")
    B, H, Cin, Cout = 2, 16, 20, 40
    c = R.conv_case(B, H, H, Cin, Cout, 2, ld=32)
    pw = mod("pack").to_device(c["pw"], DEV)
    out = torch.full((B * H * H, 80), 3.0, device=DEV, dtype=torch.bfloat16)
    ops.conv3x3(c["x"].to(DEV), B, H, H, Cin, pw, out, ocol0=40, n_store=40)
    torch.cuda.synchronize()
    _verdict("conv into columns [40, 80)", out[:, 40:80], R.conv3x3(c["x"], B, H, H, Cin, c["pw"]))
    assert float((out[:, :40].float() - 3).abs().max()) == 0.0
    # the slice is also a valid conv INPUT (view with a 16-byte aligned column offset): DownBlock's stride-2 conv + LeakyReLU
    c2 = R.conv_case(B, H, H, 40, 40, 3)
    pw2 = mod("pack").to_device(c2["pw"], DEV)
    o2 = torch.full((B * (H // 2) ** 2, 56), -7.0, device=DEV, dtype=torch.bfloat16)
    ops.conv3x3(out[:, 40:], B, H, H, 40, pw2, o2, stride=2, act=ops.ACT_LRELU, slope=0.2)
    torch.cuda.synchronize()
    _verdict("stride-2 conv from a column slice", o2[:, :40], R.conv3x3(out[:, 40:].cpu(), B, H, H, 40, c2["pw"], stride=2, act="lrelu",
                                                                       slope=0.2))
    assert bool((o2[:, 48:] == -7.0).all())


def test_gemm_partial_store_20_columns():
    ops, pack = mod("ops"), mod("pack")
    g = torch.Generator().manual_seed(3)
    a = torch.randn(300, 80, generator=g).to(torch.bfloat16)
    pw = pack.pack_gemm_weight(torch.randn(20, 80, generator=g) * 0.1, torch.randn(20, generator=g))
    out = torch.full((300, 48), 5.0, device=DEV, dtype=torch.bfloat16)
    ops.tc_gemm(a.to(DEV), 80, pack.to_device(copy.copy(pw), DEV), out, n_store=20)
    torch.cuda.synchronize()
    _verdict("1x1 GEMM, 20 stored columns", out[:, :20], R.gemm(a, 80, pw), kernel="gemm")
    assert float((out[:, 20:].float() - 5).abs().max()) == 0.0


@pytest.mark.parametrize("B,H,W,C,path", [(4, 64, 64, 40, "halo"), (4, 32, 32, 80, "halo"), (2, 128, 128, 40, "fallback")])
def test_rcab_against_reference(B, H, W, C, path):
    """One RCAB the way drn.py runs it: c1 + ReLU, c2, CALayer, x + t2 * s -- on the halo path the pooled means leave c2's epilogue
    as partial sums, on the fallback (W > 126) the implicit GEMM is followed by channel_mean.  Both end in channel_mean_parts with
    the squeeze-excite MLP and rcab_ca_scale."""
    ops, pack = mod("ops"), mod("pack")
    case = R.rcab_case(B, H, W, C, H + C)
    x = case["x"].to(DEV)
    c1, c2 = pack.to_device(copy.copy(case["c1"]), DEV), pack.to_device(copy.copy(case["c2"]), DEV)
    mlp = [t.to(DEV) for t in case["mlp"]]
    t1 = torch.empty_like(x)
    t2 = torch.empty_like(x)
    n_parts = ops.halo_parts(H, W)
    parts = torch.empty(B * n_parts, x.shape[1], device=DEV)
    scale = torch.empty(B, C, device=DEV)
    ops.conv3x3(x, B, H, W, C, c1, t1, act=ops.ACT_RELU)
    halo = ops.conv3x3(t1, B, H, W, C, c2, t2, chan_part=parts)
    assert halo == (path == "halo")
    if not halo:
        n_parts = ops.channel_mean_slices(H * W)
        ops.channel_sums(t2, B, H * W, C, parts)
    ops.channel_mean_parts(parts, B, n_parts, C, H * W, scale, *mlp, C // 16)
    ops.rcab_ca_scale(t2, x, x, scale, *mlp, B, H * W, C, 0)
    torch.cuda.synchronize()
    ref = R.rcab(case["x"], B, H, W, case["c1"], case["c2"], case["mlp"])
    _verdict(f"RCAB {B}x{H}x{W}x{C} {path}", x[:, :C], ref, case["x"][:, :C], kernel="rcab")


@pytest.mark.parametrize("name,cfg", [("drn_small_gray", DO.DrnCfg(n_blocks=3, n_colors=1)), ("drn_l_rgb", DO.DrnCfg())])
def test_drn_golden(golden_dir, name, cfg):
    g = np.load(os.path.join(golden_dir, f"{name}.npz"))
    sd = DO.make_state_dict(cfg, seed=5)
    assert abs(DO.state_dict_checksum(sd) - float(g["checksum"])) < 1e-6 * float(g["checksum"])
    m = _model(cfg, sd)
    outs = m(torch.from_numpy(g["x"]).to(DEV))
    assert len(outs) == cfg.phase + 1
    for i, o in enumerate(outs):
        err = np.abs(o.cpu().numpy() - g[f"sr{i}"]).max() / 255.0
        print(f"[drn] golden {name} output {i}: max|dSR|/rgb_range = {err:.3g}")
        assert err < TOL, f"output {i}: max|dSR|/rgb_range = {err}"


def _u8_check(u8, want_last):
    """uint8 output against the reference's truncation: at most one grey level off, and the share of equal pixels."""
    from oracle import scoring_oracle as S
    ref = S.quantize_u8(want_last.numpy(), 255.0).astype(np.int16)
    d = np.abs(u8.cpu().numpy().astype(np.int16) - ref)
    print(f"[drn] uint8: max |d| {d.max()}, equal share {float((d == 0).mean()):.4f}")
    assert d.max() <= 1 and float((d == 0).mean()) >= 0.97


def _drn_forward_checks(lr, B):
    """DRN forward (n_blocks 6) against the oracle, batch independence and run-to-run bits.  At 64 px LR (HR 256) level 1 is 128 px
    wide, past the halo conv's 126, so its RCABs take the implicit GEMM + channel_mean branch.  The end-to-end bound cannot see
    CA-level defects (a squeeze-excite bias off by 0.5 in every CALayer moves the outputs by 2.3e-4 rgb_range, a DownBlock slope
    of 0.22 by 1.1e-3): the kernel tests above carry that weight."""
    cfg = DO.DrnCfg(n_blocks=6)
    sd = DO.make_state_dict(cfg, seed=9)
    m = _model(cfg, sd)
    x = torch.rand(B, 3, lr, lr, generator=torch.Generator().manual_seed(1)) * 255.0
    with torch.no_grad():
        want = DO.drn_forward(sd, x, cfg)
    outs, u8 = m.run(x.to(DEV), want_float=True, want_u8=True)
    for i, (o, wv) in enumerate(zip(outs, want)):
        err = float((o.cpu() - wv).abs().max()) / 255.0
        print(f"[drn] {lr} px LR output {i}: max|dSR|/rgb_range = {err:.3g}")
        assert err < DRN_TOL[lr]
    _u8_check(u8, want[-1])
    again, u8_again = m.run(x.to(DEV), want_float=True, want_u8=True)
    assert all(torch.equal(a, b) for a, b in zip(outs, again)) and torch.equal(u8, u8_again), "two runs differ"
    alone, u8_alone = m.run(x[B - 1:].to(DEV), want_float=True, want_u8=True)
    assert all(torch.equal(a[B - 1:], b) for a, b in zip(outs, alone)) and torch.equal(u8[B - 1:], u8_alone), "depends on the batch"


def test_drn_batch_vs_oracle_and_u8():
    _drn_forward_checks(32, 5)


def test_drn_64px_lr_fallback_branch():
    _drn_forward_checks(64, 2)
