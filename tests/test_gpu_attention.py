"""GPU parity of the standalone (shifted-)window attention kernels -- mma.sync (csrc/attention.cu), tcgen05 for 8 x 8
windows (csrc/attention_tc.cu) and for 16 x 16 windows (csrc/attention_tc16.cu) -- against the fp64 reference of
oracle/hotpath_oracle.py on the same bf16 q | k | v, with the comparator in units of rms(O)."""
import ctypes

import pytest
import torch

from oracle import hotpath_oracle as R
from gpu_common import mod

pytestmark = pytest.mark.gpu
DEV = "cuda"
B_TOL, RMS_TOL = R.TOL["attention"]


def _run(B, H, W, ws, shift, heads, hd, seed, mode=None, **kw):
    """mode None: the dispatcher's choice; else forced through adsr_debug_set_attention_tc (0 mma.sync, 1 default, 2 tcgen05)."""
    ops, abi = mod("ops"), mod("_abi")
    case = R.attention_case(B, H, W, ws, shift, heads, hd, seed, **kw)
    hdp, M = case["hdp"], B * H * W
    qkv, table = case["qkv"].to(DEV), case["table"].to(DEV)
    out = torch.full((M, heads * hdp), 3.0, device=DEV, dtype=torch.bfloat16)
    setter = abi.lib().adsr_debug_set_attention_tc
    setter.restype, setter.argtypes = None, [ctypes.c_int]
    if mode is not None:
        setter(mode)
    try:
        ops.window_attention(qkv, out, table, B, H, W, ws, shift, heads, hd, hdp)
        torch.cuda.synchronize()
    finally:
        setter(1)
    ref = R.attention_ref(dict(case, qkv=qkv, table=table))
    got = out.view(M, heads, hdp)
    tag = f"B={B} {H}x{W} ws={ws} shift={shift} heads={heads} hd={hd} mode={mode} {kw}"
    assert bool(torch.isfinite(got.float()).all()), f"{tag}: non-finite output"
    v = R.compare(got[:, :, :hd], ref[:, :, :hd], b=R.PEAKED_B if "bias_range" in kw else B_TOL, rms_b=RMS_TOL)
    print(f"[attention] {tag}: {v}")
    assert v.ok, f"{tag}: {v}"
    if hdp > hd:
        assert float(got[:, :, hd:].float().abs().max()) == 0.0, "head padding columns must be exact zeros"


@pytest.mark.parametrize("H,ws,shift,heads,hd", [
    (32, 8, 0, 6, 30), (32, 8, 4, 4, 53), (32, 8, 0, 2, 122), (32, 8, 4, 6, 46), (32, 8, 0, 4, 77),
    (16, 4, 2, 4, 23), (16, 4, 0, 6, 10), (64, 16, 8, 4, 53), (64, 16, 0, 6, 30),
])
def test_window_attention(H, ws, shift, heads, hd):
    B = 2 if H < 64 else 1
    _run(B, H, H, ws, shift, heads, hd, H + hd, qk_scale=1.5)


@pytest.mark.parametrize("heads,hd,shift", [(6, 30, 0), (6, 30, 4), (4, 53, 4), (2, 122, 0), (2, 122, 4), (6, 46, 4), (4, 77, 0)])
@pytest.mark.parametrize("mode", [0, 2])
def test_window_attention_both_kernels(heads, hd, shift, mode):
    """ws = 8: the tcgen05 kernel (mode 2, forced for every head width) and the mma.sync kernel (mode 0) against torch,
    several tiles per CTA (B = 40 -> 320 window pairs on 148 SMs)."""
    _run(40, 32, 32, 8, shift, heads, hd, hd + shift, mode=mode)


@pytest.mark.parametrize("heads,hd", [(6, 30), (4, 53), (2, 122), (6, 46), (4, 77)])
@pytest.mark.parametrize("shift", [0, 8])
@pytest.mark.parametrize("mode", [1, 0])
def test_window_attention_ws16_batch(heads, hd, shift, mode):
    """BASELINE configs[3] (64 px LR, 16 x 16 windows, N = 256): the tcgen05 kernel of csrc/attention_tc16.cu (mode 1) and the
    mma.sync kernel (mode 0) against torch for the five DRCT-L block widths, shifted and unshifted, at batch 5
    (80 windows: several units per CTA, so the K / V / Q rings wrap and both TMEM halves are reused)."""
    _run(5, 64, 64, 16, shift, heads, hd, hd + shift, mode=mode, qk_scale=1.5)


@pytest.mark.parametrize("H,W,B,shift", [(32, 64, 3, 8), (48, 16, 2, 8), (16, 16, 1, 0)])
def test_window_attention_ws16_rect_and_tiny(H, W, B, shift):
    """16 x 16 windows on rectangular grids and on a single window (fewer windows than CTAs per head)."""
    _run(B, H, W, 16, shift, 4, 53, H + W)


@pytest.mark.parametrize("edge", ["peaked", "masked_max"])
@pytest.mark.parametrize("ws,mode", [pytest.param(8, 0, id="ws8-mma_sync"), pytest.param(8, 2, id="ws8-tcgen05"),
                                     pytest.param(16, 1, id="ws16-tcgen05"), pytest.param(16, 0, id="ws16-mma_sync")])
@pytest.mark.parametrize("heads,hd", [(6, 30), (2, 122)])
def test_window_attention_softmax_edges(heads, hd, ws, mode, edge):
    """peaked: logits about 10 apart (q, k x 3.5) and a bias table from U(-8, 8) (attention_tc16 shifts by max(S) + max(bias));
    masked_max: every offset that crosses a region boundary of the wrap windows gets +10 of bias, so rows there take their
    largest logit from a masked key: the tcgen05 kernels shift by it and zero the masked probabilities, the reference adds -100."""
    kw = dict(qk_scale=3.5, bias_range=8.0) if edge == "peaked" else dict(masked_max=True)
    B, H = (6, 32) if ws == 8 else (2, 64)
    _run(B, H, H, ws, ws // 2, heads, hd, 11 * hd + ws, mode=mode, **kw)
