"""GPU parity of the fused attention half (norm1 + qkv + shifted-window attention + proj + residual, csrc/swin_attn.cu)
against the fp64 reference built from the packed bytes (oracle/hotpath_oracle.py), with the per-element and RMS
comparator in units of the attention branch.  Each case id names the plan branch of swin_attn_plan it runs."""
import pytest
import torch

from oracle import hotpath_oracle as R
from gpu_common import mod

pytestmark = pytest.mark.gpu
DEV = "cuda"
B_TOL, RMS_TOL = R.TOL["swin_attn"]

BRANCH = {(180, 6): "pipelined", (212, 4): "fused", (276, 6): "two-proj-pieces", (244, 2): "one-region", (308, 4): "two-regions"}


def _case(B, H, W, C, heads, shift, fuse, seed=0, **kw):
    ops = mod("ops")
    b_tol = R.PEAKED_B if "qk_gain" in kw else B_TOL
    case = R.swin_attn_case(B, H, W, C, heads, shift, seed, **kw)
    pa = mod("pack").to_device(case["pa"], DEV)
    hd, hdp = pa.hd, pa.hdp
    mode = ops.swin_attn_mode(C, heads, hdp, fuse)
    assert mode == (2 if fuse else 1), f"C={C} heads={heads}: mode {mode}"
    M, ld = B * H * W, 320
    x = torch.full((M, ld), 3.0, device=DEV, dtype=torch.bfloat16)            # columns >= C hold other slab data: must be ignored
    x[:, :C] = case["x"].to(DEV)
    stats, table = case["stats"].to(DEV), case["table"].to(DEV)
    att_ref, y_ref = R.swin_attn(x, stats, 2, pa, table, B, H, W, shift, fuse)
    tag = f"C={C} heads={heads} shift={shift} {kw}"
    if fuse:
        out = torch.full((M, ld), -7.0, device=DEV, dtype=torch.bfloat16)
        st_out = torch.full((M, 4, 2), 1e9, device=DEV)
        ops.swin_attn(x, pa, table, out, B, H, W, shift, (stats, 2), True, stats_out=(st_out, 1))
        torch.cuda.synchronize()
        assert bool(torch.isfinite(out[:, :C].float()).all()), f"{tag}: non-finite y"
        v = R.compare(out[:, :C], y_ref, x[:, :C], b=b_tol, rms_b=RMS_TOL)
        print(f"[swin_attn y] {tag}: {v}")
        assert v.ok, f"{tag}: y {v}"
        # the TMA store clips at the tensor-map width C rounded up to a 16-byte chunk: pad columns inside that chunk receive exact
        # zeros (zero weight rows, zero bias, zero-filled shortcut), everything beyond stays untouched
        c8 = (C + 7) // 8 * 8
        tail = out[:, C:c8].float()
        assert bool(((tail == 0.0) | (tail == -7.0)).all()), "pad columns must be zero or untouched"
        assert float((out[:, c8:].float() + 7.0).abs().max()) == 0.0, "wrote past the 16-byte chunk holding column C-1"
        # (sum, sumsq) of the fp32 values the epilogue rounded into y: within half an ulp per element of the stored row
        r = R.stats_bound_check(st_out[:, 1], out[:, :C])
        assert r <= 1.0, f"{tag}: stats_out off by {r:.3g} x its bound"
        assert float((st_out[:, 0] - 1e9).abs().max()) == 0.0 and float((st_out[:, 2:] - 1e9).abs().max()) == 0.0
    else:
        out = torch.full((M, heads * hdp), -7.0, device=DEV, dtype=torch.bfloat16)
        ops.swin_attn(x, pa, table, out, B, H, W, shift, (stats, 2), False)
        torch.cuda.synchronize()
        got = out.view(M, heads, hdp)
        assert bool(torch.isfinite(got.float()).all()), f"{tag}: non-finite attention rows"
        v = R.compare(got[:, :, :hd], att_ref[:, :, :hd], b=b_tol, rms_b=RMS_TOL)
        print(f"[swin_attn att] {tag}: {v}")
        assert v.ok, f"{tag}: attention {v}"
        if hdp > hd:
            assert float(got[:, :, hd:].float().abs().max()) == 0.0, "head padding columns must be exact zeros"


@pytest.mark.parametrize("C,heads,shift", [pytest.param(C, h, s, id=f"{BRANCH[(C, h)]}-{C}-{h}-{s}")
                                           for C, h, s in [(180, 6, 0), (212, 4, 4), (276, 6, 4), (180, 6, 4), (212, 4, 0)]])
@pytest.mark.parametrize("shortcut", [pytest.param(1.0, id="x"), pytest.param(2.0 ** -6, id="x_over_64")])
def test_swin_attn_fused_proj(C, heads, shift, shortcut):
    """shortcut 2^-6 (exact in bf16; LayerNorm is scale-invariant apart from eps, which the reference carries): y is then mostly
    branch, and its bf16 rounding resolves the branch instead of the shortcut."""
    _case(3, 32, 32, C, heads, shift, True, seed=C + shift, shortcut_scale=shortcut)


@pytest.mark.parametrize("C,heads,shift", [pytest.param(C, h, s, id=f"{'two-regions' if (C, h) == (180, 6) else BRANCH[(C, h)]}-{C}-{h}-{s}")
                                           for C, h, s in [(244, 2, 0), (308, 4, 0), (244, 2, 4), (308, 4, 4), (180, 6, 4)]])
def test_swin_attn_qkv_attention_only(C, heads, shift):
    _case(3, 32, 32, C, heads, shift, False, seed=C + shift)


def test_swin_attn_many_tiles_per_cta_and_rect():
    _case(40, 32, 32, 180, 6, 4, True, seed=7)          # 320 window pairs on 148 SMs: several tiles per CTA
    _case(2, 16, 40, 212, 4, 4, True, seed=8)           # rectangular image, wrap in both directions
    _case(1, 8, 16, 276, 6, 0, True, seed=9)            # a single tile


@pytest.mark.parametrize("C,heads", [(180, 6), (212, 4), (276, 6)])
@pytest.mark.parametrize("B,H,W,shift", [
    (40, 32, 32, 0), (40, 32, 32, 4),        # 320 window pairs on 148 SMs: several tiles per CTA
    (1, 8, 16, 0),                           # a single tile
    (3, 16, 24, 0), (3, 16, 24, 4),          # 9 tiles on 148 SMs: one tile per CTA, rectangular
])
def test_swin_attn_qkv_attention_only_geometries(C, heads, B, H, W, shift):
    """qkv + attention only (proj stays a GEMM) on the DRCT-L block shapes the model runs with proj fused, over tile counts
    from one to several per CTA: the fused kernel with two TMEM head regions (the next head's q|k|v runs one head ahead)."""
    _case(B, H, W, C, heads, shift, False, seed={40: C + shift, 1: 3, 3: 5}[B])


@pytest.mark.parametrize("mean_std", [10, 100])
@pytest.mark.parametrize("C,heads,fuse", [pytest.param(180, 6, True, id="pipelined-180-6"), pytest.param(276, 6, True, id="two-proj-pieces-276-6"),
                                          pytest.param(308, 4, False, id="two-regions-308-4")])
def test_swin_attn_row_mean_over_std(C, heads, fuse, mean_std):
    """Rows whose mean is mean_std standard deviations: the one-pass fp32 variance from (sum, sumsq) loses
    ~2^-24 (mean/std)^2 of var.  100 is the edge of the supported range (DESIGN.md section 2)."""
    _case(3, 32, 32, C, heads, 4, fuse, seed=C + mean_std, mean_std=mean_std, shortcut_scale=2.0 ** -6 if fuse else 1.0)


@pytest.mark.parametrize("edge", ["peaked", "masked_max"])
@pytest.mark.parametrize("C,heads,fuse", [pytest.param(180, 6, True, id="pipelined-180-6"), pytest.param(244, 2, False, id="one-region-244-2"),
                                          pytest.param(308, 4, False, id="two-regions-308-4")])
def test_swin_attn_softmax_edges(C, heads, fuse, edge):
    """peaked: logits about 10 apart (q, k weights x3) and a bias table from U(-8, 8); masked_max: every offset that crosses a
    region boundary of the wrap windows gets +10 of bias, so rows there take their largest logit from a masked key (the kernel
    shifts by that maximum and zeroes the masked probabilities, the reference adds -100)."""
    kw = dict(qk_gain=3.0, bias_range=8.0) if edge == "peaked" else dict(masked_max=True)
    _case(3, 32, 32, C, heads, 4, fuse, seed=C + 17, shortcut_scale=2.0 ** -6 if fuse else 1.0, **kw)
