"""GPU parity of the tcgen05 GEMM kernels (csrc/tc_gemm.cu, the row-tile csrc/tc_gemm_rows.cu) against the fp64 reference of
oracle/hotpath_oracle.py on the packed weights, with the comparator in units of the GEMM output; the implicit-GEMM convs
against fp32 torch on bf16-rounded inputs."""
import pytest
import torch
import torch.nn.functional as F

from oracle import hotpath_oracle as R
from gpu_common import bf16_round, mod, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
B_TOL, RMS_TOL = R.TOL["gemm"]


def _check(tag, got, ref, shortcut=None):
    assert bool(torch.isfinite(got.float()).all()), f"{tag}: non-finite output"
    v = R.compare(got, ref, shortcut, b=B_TOL, rms_b=RMS_TOL)
    print(f"[gemm] {tag}: {v}")
    assert v.ok, f"{tag}: {v}"


def _gemm_case(M, K, N, act="none", res=False, alpha=1.0, ocol0=0, n_store=None, seed=0, rows=False):
    ops, pack = mod("ops"), mod("pack")
    torch.manual_seed(seed)
    lda = (K + 63) // 64 * 64 + 64
    a = torch.full((M, lda), 9.0, device=DEV, dtype=torch.bfloat16)          # poison beyond K
    a[:, :K] = torch.randn(M, K, device=DEV).to(torch.bfloat16)
    k8 = (K + 7) // 8 * 8
    a[:, K:k8] = 3.0                                                          # finite junk in the K tail
    w = torch.randn(N, K, device=DEV) * 0.1
    bias = torch.randn(N, device=DEV)
    pw = pack.pack_gemm_weight(w, bias, rows_kernel=rows)
    ldo = 1024
    out = torch.full((M, ldo), -7.0, device=DEV, dtype=torch.bfloat16)
    r = torch.randn(M, 512, device=DEV).to(torch.bfloat16) if res else None
    code = {"none": ops.ACT_NONE, "gelu": ops.ACT_GELU, "lrelu": ops.ACT_LRELU, "relu": ops.ACT_RELU}[act]
    ops.tc_gemm(a, K, pw, out, act=code, slope=0.2, alpha=alpha, res=r, ocol0=ocol0, n_store=n_store)
    torch.cuda.synchronize()
    ns = (N + 15) // 16 * 16 if n_store is None else n_store
    got = out[:, ocol0:ocol0 + N]
    ref = R.gemm(a, K, pw, act=act, slope=0.2, alpha=alpha, res=r)
    _check(f"M={M} K={K} N={N} act={act} res={res} rows={rows}", got, ref, r[:, :N] if res else None)
    if ns > N:
        assert float(out[:, ocol0 + N:ocol0 + ns].float().abs().max()) == 0.0, "padded columns must be exact zeros"
    assert float((out[:, ocol0 + ns:].float() + 7.0).abs().max()) == 0.0, "wrote past n_store"
    if ocol0:
        assert float((out[:, :ocol0].float() + 7.0).abs().max()) == 0.0, "wrote before ocol0"


def test_gemm_single_tile_k64():
    _gemm_case(128, 64, 64)


def test_gemm_k16_steps():
    _gemm_case(128, 16, 16)
    _gemm_case(128, 48, 32)


@pytest.mark.parametrize("K", [180, 212, 244, 276, 308, 488])
def test_gemm_k_tails(K):
    _gemm_case(256, K, 192, seed=K)


@pytest.mark.parametrize("N", [32, 180, 360, 576, 768, 864, 960])
def test_gemm_n_tiles(N):
    _gemm_case(384, 180, N, seed=N)


def test_gemm_row_tail_and_many_tiles():
    _gemm_case(128 * 301 + 77, 212, 424, act="gelu", seed=5)     # > 148 tiles: persistent loop + TMEM double buffer


def test_gemm_epilogues():
    _gemm_case(300, 244, 244, act="none", res=True, seed=6)
    _gemm_case(300, 308, 180, act="none", res=True, alpha=0.2, seed=7)
    _gemm_case(300, 180, 32, act="lrelu", ocol0=180, n_store=32, seed=8)     # slab slice at an 8-byte aligned column
    _gemm_case(300, 276, 276, act="relu", seed=9)


@pytest.mark.parametrize("K", [64, 180, 212, 244, 276, 308])
@pytest.mark.parametrize("N", [32, 180, 308, 576, 864, 960])
def test_gemm_rows_kernel_shapes(K, N):
    """row-tile kernel (tc_gemm_rows.cu): weights packed in 128-row N tiles, M tail, several tiles per CTA on small grids"""
    _gemm_case(128 * 3 + 77, K, N, seed=K + N, rows=True)


def test_gemm_rows_kernel_many_tiles_per_cta():
    _gemm_case(128 * 148 * 5 + 9, 180, 576, seed=31, rows=True)            # 5 N tiles x 3 K slabs, A double buffered
    _gemm_case(128 * 148 * 4 + 9, 308, 308, res=True, seed=32, rows=True)  # 5 K slabs, single A buffer, residual


def test_gemm_rows_kernel_epilogues():
    _gemm_case(128 * 160 + 5, 256, 244, act="none", res=True, seed=16, rows=True)       # proj: residual, > 148 tiles
    _gemm_case(700, 308, 180, act="none", res=True, alpha=0.2, seed=17, rows=True)      # adjust5: 0.2 * v + x
    _gemm_case(700, 180, 360, act="gelu", seed=18, rows=True)
    _gemm_case(700, 192, 96, act="lrelu", ocol0=64, n_store=96, seed=19, rows=True)     # column offset, exact n_store
    _gemm_case(700, 276, 276, act="relu", res=True, seed=20, rows=True)


def _conv_case(B, H, W, Cin, Cout, stride=1, act="none", res=False, ps=False, seed=0):
    ops, pack = mod("ops"), mod("pack")
    torch.manual_seed(seed)
    ld = (Cin + 15) // 16 * 16
    x = torch.zeros(B * H * W, ld, device=DEV, dtype=torch.bfloat16)
    x[:, :Cin] = torch.randn(B * H * W, Cin, device=DEV).to(torch.bfloat16)
    w = torch.randn(Cout, Cin, 3, 3, device=DEV) * 0.05
    bias = torch.randn(Cout, device=DEV)
    pw = pack.pack_conv3x3_weight(w, bias)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    xin = x[:, :Cin].float().view(B, H, W, Cin).permute(0, 3, 1, 2)
    want = F.conv2d(xin, bf16_round(w), bias, stride=stride, padding=1)
    code = {"none": ops.ACT_NONE, "lrelu": ops.ACT_LRELU}[act]
    if act == "lrelu":
        want = F.leaky_relu(want, 0.01)
    r = None
    if res:
        r = torch.randn(B * Ho * Wo, (Cout + 15) // 16 * 16, device=DEV).to(torch.bfloat16)
        want = want + r[:, :Cout].float().view(B, Ho, Wo, Cout).permute(0, 3, 1, 2)
    if ps:
        want = F.pixel_shuffle(want, 2)
        out = torch.zeros(B * 4 * Ho * Wo, Cout // 4, device=DEV, dtype=torch.bfloat16)
        ops.conv3x3(x, B, H, W, Cin, pw, out, out_mode=ops.OUT_PIXEL_SHUFFLE2)
        got = out.float().view(B, 2 * Ho, 2 * Wo, Cout // 4).permute(0, 3, 1, 2)
    else:
        out = torch.zeros(B * Ho * Wo, (Cout + 15) // 16 * 16, device=DEV, dtype=torch.bfloat16)
        ops.conv3x3(x, B, H, W, Cin, pw, out, stride=stride, act=code, slope=0.01, res=r)
        got = out[:, :Cout].float().view(B, Ho, Wo, Cout).permute(0, 3, 1, 2)
    torch.cuda.synchronize()
    err = rel_err(got, want)
    assert err < 0.012, f"conv B={B} H={H} Cin={Cin} Cout={Cout} s={stride} ps={ps}: rel err {err}"


def test_conv_64_to_64():
    _conv_case(1, 16, 16, 64, 64)


def test_conv_after_body_shape():
    _conv_case(2, 32, 32, 180, 180, res=True, seed=1)


def test_conv_before_upsample_shape():
    _conv_case(2, 32, 32, 180, 64, act="lrelu", seed=2)


def test_conv_upsample_pixelshuffle():
    _conv_case(2, 32, 32, 64, 256, ps=True, seed=3)
    _conv_case(1, 64, 64, 64, 256, ps=True, seed=4)


def test_conv_stride2_and_odd_sizes():
    _conv_case(2, 32, 32, 80, 80, stride=2, seed=5)
    _conv_case(3, 20, 12, 16, 32, seed=6)        # M not a multiple of 128, tiles straddle images


@pytest.mark.parametrize("B,H,W,Cin,Cout,act", [(3, 32, 32, 80, 80, "relu"), (2, 64, 64, 80, 80, "none"), (5, 17, 24, 40, 48, "lrelu"),
                                                (1, 9, 126, 128, 16, "none"), (150, 16, 16, 64, 64, "relu"), (2, 8, 8, 20, 20, "none")])
def test_conv_halo_tile_kernel(B, H, W, Cin, Cout, act):
    """Halo-tile conv with resident weights (csrc/conv_halo.cu), called directly: every tap offset / tile phase / image border,
    poison in the untouched output columns, and equality with the streaming implicit GEMM on the same inputs."""
    ops, pack, abi = mod("ops"), mod("pack"), mod("_abi")
    torch.manual_seed(B * 131 + W)
    ld = (Cin + 15) // 16 * 16 + 16
    x = torch.full((B * H * W, ld), 7.0, device=DEV, dtype=torch.bfloat16)      # columns >= Cin must not matter beyond round8
    x[:, :Cin] = torch.randn(B * H * W, Cin, device=DEV).to(torch.bfloat16)
    x[:, Cin:(Cin + 7) // 8 * 8] = 0
    w = torch.randn(Cout, Cin, 3, 3, device=DEV) * 0.05
    bias = torch.randn(Cout, device=DEV)
    pw = pack.pack_conv3x3_weight(w, bias)
    assert pw.compact is not None
    wc = pw.compact
    code = {"none": ops.ACT_NONE, "lrelu": ops.ACT_LRELU, "relu": ops.ACT_RELU}[act]
    n_store = (Cout + 15) // 16 * 16
    out_g = torch.full((B * H * W + 64, n_store + 24), -3.0, device=DEV, dtype=torch.bfloat16)     # 32 guard rows on either side
    out = out_g[32:-32]
    n_parts = ops.halo_parts(H, W)
    parts_g = torch.full((B * n_parts + 16, wc.BN), float("nan"), device=DEV)   # every entry must be written, none outside
    parts = parts_g[8:-8]
    st = abi.lib().adsr_conv3x3_halo_bf16(abi.ptr(x), x.stride(0), B, H, W, Cin, abi.ptr(wc.data), abi.ptr(wc.bias), wc.N, wc.BN, code,
                                          0.1, abi.ptr(out), out.stride(0), 8, n_store, abi.ptr(parts), abi.num_sms(), abi.stream_ptr())
    assert st == 0, f"status {st}"
    mean = torch.zeros(B, Cout, device=DEV)
    ops.channel_mean_parts(parts, B, n_parts, Cout, H * W, mean)
    torch.cuda.synchronize()
    xin = x[:, :Cin].float().view(B, H, W, Cin).permute(0, 3, 1, 2)
    want = F.conv2d(xin, bf16_round(w), bias, padding=1)
    want = {"none": lambda t: t, "lrelu": lambda t: F.leaky_relu(t, 0.1), "relu": F.relu}[act](want)
    got = out[:, 8:8 + Cout].float().view(B, H, W, Cout).permute(0, 3, 1, 2)
    err = rel_err(got, want)
    assert err < 0.012, f"halo conv rel err {err}"
    # pooled means from the epilogue's partial sums (fp32 values before the bf16 rounding): AdaptiveAvgPool2d(1) of the output
    want_mean = want.mean(dim=(2, 3))
    assert float((mean - want_mean).abs().max()) < 2e-3 * max(1.0, float(want_mean.abs().max())), "pooled mean"
    assert bool(torch.isfinite(parts).all())
    # the same kernel continuing with CALayer's squeeze-excite MLP: sigmoid(W2 relu(W1 mean + b1) + b2)   (src/drn.py:128-139)
    cr = max(1, Cout // 16)
    w1, b1 = torch.randn(cr, Cout, device=DEV) * 0.3, torch.randn(cr, device=DEV) * 0.1
    w2, b2 = torch.randn(Cout, cr, device=DEV) * 0.3, torch.randn(Cout, device=DEV) * 0.1
    scale = torch.zeros(B, Cout, device=DEV)
    ops.channel_mean_parts(parts, B, n_parts, Cout, H * W, scale, w1, b1, w2, b2, cr)
    torch.cuda.synchronize()
    want_scale = torch.sigmoid(F.relu(mean @ w1.t() + b1) @ w2.t() + b2)
    assert float((scale - want_scale).abs().max()) < 1e-5
    assert bool((out[:, :8] == -3.0).all()) and bool((out[:, 8 + n_store:] == -3.0).all())
    assert bool((out_g[:32] == -3.0).all()) and bool((out_g[-32:] == -3.0).all())
    assert bool(torch.isnan(parts_g[:8]).all()) and bool(torch.isnan(parts_g[-8:]).all())
    assert bool((out[:, 8 + Cout:8 + n_store] == 0).all())                      # padded output channels: zero weights, zero bias
    # the streaming kernel computes the same sums in a different K order: equal to bf16 rounding
    ref = torch.zeros(B * H * W, n_store, device=DEV, dtype=torch.bfloat16)
    old = ops._HALO_CONV
    ops._HALO_CONV = False
    try:
        ops.conv3x3(x, B, H, W, Cin, pw, ref, act=code, slope=0.1)
    finally:
        ops._HALO_CONV = old
    torch.cuda.synchronize()
    assert rel_err(out[:, 8:8 + Cout].float(), ref[:, :Cout].float()) < 0.006


def _row_stats(t: torch.Tensor, slots: int) -> torch.Tensor:
    """(sum, sumsq) of each row in slot 0, zeros elsewhere: what a producing epilogue leaves behind."""
    st = torch.zeros(t.shape[0], slots, 2, device=t.device)
    st[:, 0, 0] = t.float().sum(1)
    st[:, 0, 1] = (t.float() ** 2).sum(1)
    return st


@pytest.mark.parametrize("rows", [False, True])
@pytest.mark.parametrize("K,N,act", [(180, 576, "none"), (212, 424, "gelu"), (308, 960, "none"), (60, 120, "gelu")])
def test_gemm_with_folded_layernorm(K, N, act, rows):
    """LayerNorm(K) folded into the GEMM: raw rows in, row statistics from the (sum, sumsq) slots."""
    ops, pack = mod("ops"), mod("pack")
    torch.manual_seed(K + N)
    M = 128 * 150 + 37
    a = torch.full((M, 320), 50.0, device=DEV, dtype=torch.bfloat16)          # columns >= K must not influence anything
    a[:, :K] = (torch.randn(M, K, device=DEV) * 2.5 + 1.5 * torch.randn(M, 1, device=DEV)).to(torch.bfloat16)
    w, b = torch.randn(N, K, device=DEV) * 0.1, torch.randn(N, device=DEV)
    g, bt = torch.rand(K, device=DEV) + 0.5, torch.randn(K, device=DEV) * 0.3
    pw = pack.pack_ln_gemm_weight(w, b, g, bt, 1e-5, rows_kernel=rows)
    st = _row_stats(a[:, :K], 4)
    st[:, 1] = st[:, 0] * 0.25                                                  # statistics split over two slots
    st[:, 0] = st[:, 0] * 0.75
    out = torch.zeros(M, 1024, device=DEV, dtype=torch.bfloat16)
    ops.tc_gemm(a, K, pw, out, act=ops.ACT_GELU if act == "gelu" else ops.ACT_NONE, stats_in=(st, 2))
    torch.cuda.synchronize()
    out_rev = torch.zeros(M, 1024, device=DEV, dtype=torch.bfloat16)           # row tiles walked from the last one down: same bits
    ops.tc_gemm(a, K, pw, out_rev, act=ops.ACT_GELU if act == "gelu" else ops.ACT_NONE, stats_in=(st, 2), reverse=True)
    torch.cuda.synchronize()
    assert torch.equal(out, out_rev)
    ref = R.gemm(a, K, pw, act=act, stats=st, slots=2)
    _check(f"LN-folded K={K} N={N} act={act} rows={rows}", out[:, :N], ref)


@pytest.mark.parametrize("rows", [False, True])
@pytest.mark.parametrize("mean_std", [10, 100])
@pytest.mark.parametrize("K,N,act", [(180, 576, "none"), (212, 424, "gelu")])
def test_gemm_folded_layernorm_row_mean_over_std(K, N, act, mean_std, rows):
    """Rows whose mean is mean_std standard deviations: the one-pass fp32 variance from (sum, sumsq) loses ~2^-24 (mean/std)^2
    of var.  100 is the edge of the supported range (DESIGN.md section 2)."""
    ops = mod("ops")
    case = R.ln_gemm_case(128 * 20 + 37, K, N, K + N + mean_std, rows=rows, mean_std=mean_std)
    pw = mod("pack").to_device(case["pw"], DEV)
    a = torch.full((case["a"].shape[0], 320), 50.0, device=DEV, dtype=torch.bfloat16)
    a[:, :K] = case["a"].to(DEV)
    st = case["stats"].to(DEV)
    out = torch.zeros(a.shape[0], 1024, device=DEV, dtype=torch.bfloat16)
    ops.tc_gemm(a, K, pw, out, act=ops.ACT_GELU if act == "gelu" else ops.ACT_NONE, stats_in=(st, 2))
    torch.cuda.synchronize()
    _check(f"LN-folded K={K} N={N} mean/std={mean_std} rows={rows}", out[:, :N], R.gemm(a, K, pw, act=act, stats=st, slots=2))


@pytest.mark.parametrize("rows", [False, True])
@pytest.mark.parametrize("N,res", [(32, False), (180, True), (308, True)])
def test_gemm_emits_row_statistics(N, res, rows):
    """stats_out: per-row (sum, sumsq) partials of the stored output, in deterministic slots."""
    ops, pack = mod("ops"), mod("pack")
    torch.manual_seed(N)
    M, K = 1000, 244
    a = torch.randn(M, 256, device=DEV).to(torch.bfloat16)
    w, b = torch.randn(N, K, device=DEV) * 0.1, torch.randn(N, device=DEV)
    pw = pack.pack_gemm_weight(w, b, rows_kernel=rows)
    r = torch.randn(M, 320, device=DEV).to(torch.bfloat16) if res else None
    out = torch.zeros(M, 320, device=DEV, dtype=torch.bfloat16)
    st = torch.full((M, 10, 2), 7.0, device=DEV)
    ops.tc_gemm(a, K, pw, out, res=r, stats_out=(st, 2))
    torch.cuda.synchronize()
    out_rev, st_rev = torch.zeros_like(out), torch.full((M, 10, 2), 7.0, device=DEV)
    ops.tc_gemm(a, K, pw, out_rev, res=r, stats_out=(st_rev, 2), reverse=True)
    torch.cuda.synchronize()
    assert torch.equal(out, out_rev) and torch.equal(st, st_rev)
    used = 2 * pw.n_tiles
    o = out[:, :N]
    _check(f"stats N={N} res={res} rows={rows}", o, R.gemm(a, K, pw, res=r), r[:, :N] if res else None)
    r_ = R.stats_bound_check(st[:, 2:2 + used].sum(1), o)
    assert r_ <= 1.0, f"stats_out off by {r_:.3g} x its bound"
    assert float((st[:, :2] - 7).abs().max()) == 0.0 and float((st[:, 2 + used:] - 7).abs().max()) == 0.0
