"""GPU parity of the fused Swin MLP kernel (norm2 + fc1 + GELU + fc2 + residual, csrc/swin_mlp.cu) and its folded adjust /
folded wide-conv epilogues against the fp64 reference of oracle/hotpath_oracle.py (weights unpacked from the kernel's
slabs), with the comparator in units of the MLP branch."""
import pytest
import torch

from oracle import hotpath_oracle as R
from gpu_common import mod

pytestmark = pytest.mark.gpu
DEV = "cuda"
B_TOL, RMS_TOL = R.TOL["swin_mlp"]


def _inputs(M, C, H, seed, **kw):
    case = R.mlp_case(M, C, H, seed, **kw)
    pm = mod("pack").to_device(case["pm"], DEV)
    ld = 320
    y = torch.full((M, ld), 5.0, device=DEV, dtype=torch.bfloat16)            # poison beyond C
    y[:, :C] = case["y"].to(DEV)
    return case, pm, y, case["stats"].to(DEV)


def _check(tag, got, ref, shortcut):
    assert bool(torch.isfinite(got.float()).all()), f"{tag}: non-finite output"
    v = R.compare(got, ref, shortcut, b=B_TOL, rms_b=RMS_TOL)
    print(f"[swin_mlp] {tag}: {v}")
    assert v.ok, f"{tag}: {v}"


def _mlp_case(M, C, H, seed=0, **kw):
    ops = mod("ops")
    _, pm, y, stats = _inputs(M, C, H, seed, **kw)
    ld = y.shape[1]
    z = torch.full((M, ld), -7.0, device=DEV, dtype=torch.bfloat16)
    ops.swin_mlp(y, C, pm, z, stats_in=(stats, 2))
    torch.cuda.synchronize()
    z_rev = torch.full((M, ld), -7.0, device=DEV, dtype=torch.bfloat16)     # tiles walked from the last one down: same bits
    ops.swin_mlp(y, C, pm, z_rev, stats_in=(stats, 2), reverse=True)
    torch.cuda.synchronize()
    assert torch.equal(z, z_rev), "reverse tile order must not change the result"
    _check(f"M={M} C={C} H={H} {kw}", z[:, :C], R.swin_mlp(y, stats, 2, pm), y[:, :C])
    # the TMA store clips at the tensor-map width C rounded up to a 16-byte chunk: pad columns inside that chunk receive
    # exact zeros (zero weight rows, zero bias, zero-filled residual), everything beyond stays untouched
    c8 = (C + 7) // 8 * 8
    tail = z[:, C:c8].float()
    assert bool(((tail == 0.0) | (tail == -7.0)).all()), "pad columns must be zero or untouched"
    assert float((z[:, c8:].float() + 7.0).abs().max()) == 0.0, "wrote past the 16-byte chunk holding column C-1"


@pytest.mark.parametrize("C,H", [(180, 360), (212, 424), (244, 488), (276, 276), (308, 308)])
def test_mlp_drct_shapes(C, H):
    _mlp_case(128 * 5 + 37, C, H, seed=C)


@pytest.mark.parametrize("C,H", [(180, 360), (244, 488), (308, 308)])
def test_mlp_scaled_shortcut(C, H):
    """y scaled by 2^-6 (exact; LayerNorm is scale-invariant apart from eps, which the reference carries): z is mostly branch."""
    _mlp_case(128 * 5 + 37, C, H, seed=C, shortcut_scale=2.0 ** -6)


def test_mlp_single_tile():
    _mlp_case(128, 180, 360)


def test_mlp_small_dims():
    _mlp_case(300, 60, 120)        # DRCT-small widths: one hidden chunk, one K panel
    _mlp_case(300, 92, 184)


def test_mlp_many_tiles_per_cta():
    _mlp_case(128 * 148 * 3 + 5, 180, 360, seed=3)


def _adjust_case(C, H, M, seed, **kw):
    ops = mod("ops")
    case, pm, y, stats = _inputs(M, C, H, seed, kind="adjust", **kw)
    ld = y.shape[1]
    stats1 = torch.zeros(M, 2, 2, device=DEV)
    stats1[:, 0] = stats[:, :2].sum(1)
    slab = torch.full((M, ld), -7.0, device=DEV, dtype=torch.bfloat16)
    st_out = torch.full((M, 6, 2), 1e9, device=DEV)
    ops.swin_mlp_adjust(y, C, pm, slab, C, stats_in=(stats1, 1), stats_out=(st_out, 2))
    torch.cuda.synchronize()
    slab_rev = torch.full((M, ld), -7.0, device=DEV, dtype=torch.bfloat16)
    ops.swin_mlp_adjust(y, C, pm, slab_rev, C, stats_in=(stats1, 1), stats_out=(torch.empty_like(st_out), 2), reverse=True)
    torch.cuda.synchronize()
    assert torch.equal(slab, slab_rev), "reverse tile order must not change the result"
    got = slab[:, C:C + 32]
    _check(f"adjust M={M} C={C} H={H} {kw}", got, R.swin_mlp(y, stats1, 1, pm), None)
    outside = torch.cat([slab[:, :C], slab[:, C + 32:]], dim=1).float()
    assert float((outside + 7.0).abs().max()) == 0.0, "wrote outside the 32-column slice"
    r = R.stats_bound_check(st_out[:, 2], got)
    assert r <= 1.0, f"stats_out off by {r:.3g} x its bound"
    assert float(st_out[:, 3].abs().max()) == 0.0
    assert float((st_out[:, :2] - 1e9).abs().max()) == 0.0 and float((st_out[:, 4:] - 1e9).abs().max()) == 0.0


@pytest.mark.parametrize("C,H,M", [(180, 360, 677), (212, 424, 677), (244, 488, 677), (276, 276, 677), (288, 288, 677), (60, 120, 677),
                                   (180, 360, 128), (180, 360, 128 * 148 * 3 + 5)])
def test_mlp_fused_adjust(C, H, M):
    """Adjust 1x1 conv (src/drct.py:389-393) folded into fc2: slab[:, C:C+32] = LReLU_0.2(adjust(z)) computed as
    y W_adj^T + g (W_adj W2)^T + bias, z never exists; row statistics of the 32 new columns in the given slot, the next slot zeroed."""
    _adjust_case(C, H, M, C)


def _conv_res_case(C, H, Co, M, inplace, seed, **kw):
    ops = mod("ops")
    case, pm, y, stats = _inputs(M, C, H, seed, kind="conv_res", Co=Co, **kw)
    ld = y.shape[1]
    assert pm.plan.tolist()[23] == 2 and pm.plan.tolist()[4] == (Co + 15) // 16 * 16
    res = torch.full((M, ld), -7.0, device=DEV, dtype=torch.bfloat16)
    res[:, :Co] = case["res"].to(DEV)
    rf = res[:, :Co].clone()
    stats1 = torch.zeros(M, 2, 2, device=DEV)
    stats1[:, 0] = stats[:, :2].sum(1)
    ref = R.swin_mlp(y, stats1, 1, pm, res=res)
    st_out = torch.full((M, 6, 2), 1e9, device=DEV)
    out = res if inplace else torch.full((M, ld), -3.0, device=DEV, dtype=torch.bfloat16)
    ops.swin_mlp_conv_res(y, C, pm, res, out, stats_in=(stats1, 1), stats_out=(st_out, 2))
    torch.cuda.synchronize()
    got = out[:, :Co]
    _check(f"conv_res M={M} C={C} Co={Co} {kw}", got, ref, rf)
    fill = -7.0 if inplace else -3.0
    c8 = (Co + 7) // 8 * 8              # the TMA store clips at Co rounded up to a 16-byte chunk; pad columns there receive exact zeros
    tail = out[:, Co:c8].float()
    assert bool(((tail == 0.0) | (tail == fill)).all()) and float((out[:, c8:].float() - fill).abs().max()) == 0.0, "wrote outside the output columns"
    if not inplace:
        assert torch.equal(res[:, :Co], rf) and float((res[:, Co:].float() + 7.0).abs().max()) == 0.0
    r = R.stats_bound_check(st_out[:, 2:6].sum(1), got)                                    # four partial slots
    assert r <= 1.0, f"stats_out off by {r:.3g} x its bound"
    assert float((st_out[:, :2] - 1e9).abs().max()) == 0.0
    if not inplace:                                                         # reverse tile order: same bits
        out2 = torch.full((M, ld), -3.0, device=DEV, dtype=torch.bfloat16)
        ops.swin_mlp_conv_res(y, C, pm, res, out2, stats_in=(stats1, 1), reverse=True)
        torch.cuda.synchronize()
        assert torch.equal(out, out2)


@pytest.mark.parametrize("C,H,Co,M,inplace", [(308, 308, 180, 677, True), (308, 308, 180, 128 * 148 * 2 + 9, True), (244, 488, 180, 677, False),
                                              (128, 256, 60, 300, True)])
def test_mlp_folded_conv_with_residual(C, H, Co, M, inplace):
    """adjust5 + the RDG residual folded into the MLP kernel (src/drct.py:394-396): out[:, :Co] = res[:, :Co] + 0.2 (W_a z + b_a), z never
    written; in place on the slab (out is res) or into another tensor; row statistics of the Co output columns in the given slot."""
    _conv_res_case(C, H, Co, M, inplace, C + Co)


def test_mlp_folded_conv_scaled_residual():
    """y and the residual scaled by 2^-6: the output is mostly branch."""
    _conv_res_case(308, 308, 180, 677, False, 488, shortcut_scale=2.0 ** -6)


@pytest.mark.parametrize("mean_std", [10, 100])
@pytest.mark.parametrize("kind", ["plain", "adjust", "conv_res"])
def test_mlp_row_mean_over_std(kind, mean_std):
    """Rows whose mean is mean_std standard deviations, through all three entry points: the one-pass fp32 variance from
    (sum, sumsq) loses ~2^-24 (mean/std)^2 of var.  100 is the edge of the supported range (DESIGN.md section 2)."""
    if kind == "plain":
        _mlp_case(677, 180, 360, seed=mean_std, mean_std=mean_std, shortcut_scale=2.0 ** -6)
    elif kind == "adjust":
        _adjust_case(180, 360, 677, mean_std, mean_std=mean_std)
    else:
        _conv_res_case(308, 308, 180, 677, False, mean_std, mean_std=mean_std, shortcut_scale=2.0 ** -6)
