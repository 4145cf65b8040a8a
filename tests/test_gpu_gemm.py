"""GPU parity of the tcgen05 GEMM kernels (csrc/tc_gemm.cu, the row-tile csrc/tc_gemm_rows.cu) and of the 3x3 convs (the
implicit GEMM on its three branches, the halo-tile csrc/conv_halo.cu) against the fp64 reference of oracle/hotpath_oracle.py on
the packed weights, with the comparator in units of the output (of the conv branch when a residual is added)."""
import pytest
import torch

from oracle import hotpath_oracle as R
from gpu_common import mod

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


CONV_TOL = R.TOL["conv"]
# conv dispatch (ops.conv3x3 -> conv_halo.cu, tc_gemm.cu): the kernel each branch launches, as torch.profiler names it
CONV_KERNEL = {"halo": r"conv_halo_kernel", "tma_box": r"tc_gemm_manual_kernel<\d+, 4>", "gather_tma_epi": r"tc_gemm_kernel<",
               "gather_manual": r"tc_gemm_manual_kernel<\d+, 3>"}


def _run_conv(c, B, H, W, Cin, Cout, *, stride=1, act="none", slope=0.01, res=False, ps=False, ocol0=0, n_store=None, ld_out=None,
              halo=True, chan_part=None):
    """ops.conv3x3 on the case's bf16 rows into a poisoned output; returns (out, got rows, Ho, Wo)."""
    ops = mod("ops")
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    pw = mod("pack").to_device(c["pw"], DEV)
    x = c["x"].to(DEV)
    r = c["res"][:B * Ho * Wo].to(DEV) if res else None
    code = {"none": ops.ACT_NONE, "lrelu": ops.ACT_LRELU, "relu": ops.ACT_RELU}[act]
    old = ops._HALO_CONV
    ops._HALO_CONV = halo
    try:
        if ps:
            out = torch.full((B * 4 * Ho * Wo, Cout // 4 + 8), -7.0, device=DEV, dtype=torch.bfloat16)
            ops.conv3x3(x, B, H, W, Cin, pw, out[:, :Cout // 4], out_mode=ops.OUT_PIXEL_SHUFFLE2, act=code, slope=slope)
            got = out[:, :Cout // 4]
        else:
            ns = (Cout + 15) // 16 * 16 if n_store is None else n_store
            out = torch.full((B * Ho * Wo, ld_out or ocol0 + ns + 16), -7.0, device=DEV, dtype=torch.bfloat16)
            ran_halo = ops.conv3x3(x, B, H, W, Cin, pw, out, stride=stride, act=code, slope=slope, res=r, ocol0=ocol0, n_store=n_store,
                                   chan_part=chan_part)
            got = out[:, ocol0:ocol0 + Cout]
    finally:
        ops._HALO_CONV = old
    torch.cuda.synchronize()
    return out, got, Ho, Wo


def _conv_case(B, H, W, Cin, Cout, stride=1, act="none", res=False, ps=False, seed=0, slope=0.01, halo=True, branch=None):
    """Implicit-GEMM / halo conv against the fp64 reference from the packed image.  `branch` names the dispatch branch when a
    residual is added: the manual epilogue (TMA-box A tiles) rounds the conv branch to bf16 before it adds the residual, and the
    comparator charges that rounding."""
    c = R.conv_case(B, H, W, Cin, Cout, seed, res=res)
    out, got, Ho, Wo = _run_conv(c, B, H, W, Cin, Cout, stride=stride, act=act, slope=slope, res=res, ps=ps, halo=halo)
    r = c["res"][:B * Ho * Wo] if res else None
    if branch is None and res:
        branch = "tma_box" if stride == 1 and W <= 128 and 128 % W == 0 and (H * W) % 128 == 0 else "gather_tma_epi"
    ref = R.conv3x3(c["x"], B, H, W, Cin, c["pw"], stride=stride, act=act, slope=slope, res=r, ps=ps)
    tag = f"conv B={B} H={H} W={W} Cin={Cin} Cout={Cout} s={stride} act={act} res={res} ps={ps} halo={halo}"
    assert bool(torch.isfinite(got.float()).all()), f"{tag}: non-finite output"
    rounded = res and branch in ("tma_box", "gather_manual")
    # two roundings in a row are not two independent uniform noises: B200 measured rms 0.00094 on tma_box_res
    v = R.compare(got.cpu(), ref, r[:, :Cout] if res else None, b=CONV_TOL[0], rms_b=0.0015 if rounded else CONV_TOL[1],
                  rounded_branch=rounded)
    print(f"[conv] {tag}: {v}")
    assert v.ok, f"{tag}: {v}"
    ns = Cout // 4 if ps else (Cout + 15) // 16 * 16
    if not ps and ns > Cout:
        assert float(out[:, Cout:ns].float().abs().max()) == 0.0, "padded columns must be exact zeros"
    assert bool((out[:, ns:] == -7.0).all()), "wrote past n_store"


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


# (name, expected branch, shape and epilogue).  The halo kernel takes stride 1 without residual at 8 <= W <= 126 when its weights
# and halo tile fit in shared memory; the TMA-box implicit GEMM stride-1 convs whose 128-pixel tiles are whole rows; a residual
# elsewhere the TMA epilogue; everything else the gather producers with the manual epilogue.
CONV_DISPATCH = [
    ("halo_w8", "halo", dict(B=3, H=8, W=8, Cin=20, Cout=20, act="relu")),
    ("halo_w126_h1", "halo", dict(B=4, H=1, W=126, Cin=40, Cout=40, act="lrelu", slope=0.2)),
    ("halo_tail_panel", "halo", dict(B=5, H=17, W=24, Cin=72, Cout=48, act="lrelu", slope=0.1, seed=72)),
    ("halo_second_panel", "halo", dict(B=2, H=16, W=40, Cin=100, Cout=48, seed=100)),
    ("halo_many_tiles", "halo", dict(B=160, H=16, W=16, Cin=96, Cout=32, act="relu")),
    ("halo_bad_shape", "gather_manual", dict(B=1, H=9, W=126, Cin=128, Cout=48)),             # 110 KB weights + 160 KB halo
    ("tma_box_w128", "tma_box", dict(B=2, H=3, W=128, Cin=64, Cout=64, halo=False)),
    ("tma_box_res", "tma_box", dict(B=2, H=24, W=32, Cin=64, Cout=64, act="lrelu", slope=0.2, res=True, seed=24)),
    ("tma_box_ps", "tma_box", dict(B=2, H=32, W=32, Cin=64, Cout=256, ps=True, seed=3)),
    ("tma_box_tail_panel", "tma_box", dict(B=2, H=16, W=16, Cin=72, Cout=40, act="lrelu", slope=0.01, halo=False)),
    ("gather_res_w24", "gather_tma_epi", dict(B=2, H=24, W=24, Cin=64, Cout=64, act="lrelu", slope=0.2, res=True, seed=24)),
    ("gather_res_w40", "gather_tma_epi", dict(B=3, H=16, W=40, Cin=96, Cout=96, res=True, seed=9)),
    ("gather_hw_off128", "gather_manual", dict(B=2, H=17, W=32, Cin=100, Cout=64, halo=False)),   # W | 128, H*W % 128 != 0
    ("gather_stride2_33x17", "gather_manual", dict(B=2, H=33, W=17, Cin=80, Cout=80, stride=2, act="lrelu", slope=0.2, seed=33)),
    ("gather_ps_w40", "gather_manual", dict(B=2, H=20, W=40, Cin=40, Cout=160, ps=True)),
    ("gather_many_tiles", "gather_manual", dict(B=40, H=33, W=33, Cin=40, Cout=40, act="relu", halo=False)),
]


def _profile_dispatch():
    """{case name: names of the CUDA kernels torch.profiler records while the case's conv runs}."""
    from torch.profiler import ProfilerActivity, profile
    seen = {}
    for name, _, kw in CONV_DISPATCH:
        kw = dict(kw)
        c = R.conv_case(kw["B"], kw["H"], kw["W"], kw["Cin"], kw["Cout"], kw.pop("seed", 0), res=kw.get("res", False))
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _run_conv(c, **kw)
        seen[name] = sorted({e.name for e in prof.events() if "kernel" in e.name})
    return seen


@pytest.fixture(scope="module")
def dispatch_kernels():
    """The kernel names of every dispatch case, profiled in a child process: after CUDA activity tracing has run in a process,
    a later profiling session there can miss kernels (tests/test_gpu_scoring_dispatch.py recorded an empty trace after these
    sessions), so this module leaves the test process's profiler untouched."""
    import json
    import os
    import subprocess
    import sys
    tests = os.path.dirname(os.path.abspath(__file__))
    code = (f"import json, sys; sys.path[:0] = [{os.path.dirname(tests)!r}, {tests!r}]; import test_gpu_gemm as T; "
            "print('KERNELS ' + json.dumps(T._profile_dispatch()))")
    p = subprocess.run([sys.executable, *subprocess._args_from_interpreter_flags(), "-c", code], capture_output=True, text=True,
                       timeout=900)
    assert p.returncode == 0, p.stderr[-4000:]
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("KERNELS ")][-1]
    return json.loads(line[len("KERNELS "):])


@pytest.mark.parametrize("name,branch,kw", CONV_DISPATCH, ids=[c[0] for c in CONV_DISPATCH])
def test_conv_dispatch_branches(dispatch_kernels, name, branch, kw):
    """Every conv branch against the reference; torch.profiler confirms the kernel the case names."""
    import re
    kw = dict(kw)
    seed = kw.pop("seed", 0)
    _conv_case(seed=seed, branch=branch, **kw)
    names = dispatch_kernels[name]
    print(f"[conv dispatch] {name}: {names}")
    if not any(dispatch_kernels.values()):
        pytest.skip("torch.profiler recorded no CUDA kernels on this runner")
    hits = {b for b, pat in CONV_KERNEL.items() if any(re.search(pat, n) for n in names)}
    assert hits == {branch}, (name, branch, names)


def test_conv_dispatch_cases_cover_every_branch():
    assert {c[1] for c in CONV_DISPATCH} == set(CONV_KERNEL)


@pytest.mark.parametrize("halo", [True, False])
def test_drn_conv_shapes_on_both_paths(halo):
    """DRN's convs on the halo kernel and on the implicit GEMM: 40 -> 40 into columns [40, 80) of an 80-wide buffer, and 80 -> 80
    with the CALayer partial sums."""
    ops = mod("ops")
    B, H, W = 2, 32, 32
    c = R.conv_case(B, H, W, 40, 40, 40)
    out, got, _, _ = _run_conv(c, B, H, W, 40, 40, ocol0=40, n_store=40, ld_out=80, halo=halo)
    v = R.compare(got.cpu(), R.conv3x3(c["x"], B, H, W, 40, c["pw"]), b=CONV_TOL[0], rms_b=CONV_TOL[1])
    print(f"[conv] DRN 40->40 slice halo={halo}: {v}")
    assert v.ok and bool((out[:, :40] == -7.0).all())
    c = R.conv_case(B, H, W, 80, 80, 80)
    n_parts = ops.halo_parts(H, W)
    parts = torch.full((B * n_parts, 80), float("nan"), device=DEV)
    out, got, _, _ = _run_conv(c, B, H, W, 80, 80, act="relu", halo=halo, chan_part=parts)
    ref = R.conv3x3(c["x"], B, H, W, 80, c["pw"], act="relu")
    v = R.compare(got.cpu(), ref, b=CONV_TOL[0], rms_b=CONV_TOL[1])
    print(f"[conv] DRN 80->80 halo={halo}: {v}")
    assert v.ok
    if halo:
        mean = R.channel_mean_parts(parts.cpu(), B, n_parts, 80, H * W)
        assert float((mean - R.channel_mean(ref, B, H * W, 80)).abs().max()) < 1e-5


@pytest.mark.parametrize("B,H,W,Cin,Cout,act", [(3, 32, 32, 80, 80, "relu"), (2, 64, 64, 80, 80, "none"), (5, 17, 24, 40, 48, "lrelu"),
                                                (1, 9, 126, 128, 16, "none"), (150, 16, 16, 64, 64, "relu"), (2, 8, 8, 20, 20, "none")])
def test_conv_halo_tile_kernel(B, H, W, Cin, Cout, act):
    """Halo-tile conv with resident weights (csrc/conv_halo.cu), called directly: every tap offset / tile phase / image border,
    poison in the untouched output columns, and the same reference on the streaming implicit GEMM."""
    ops, abi = mod("ops"), mod("_abi")
    ld = (Cin + 15) // 16 * 16 + 16
    c = R.conv_case(B, H, W, Cin, Cout, B * 131 + W, ld=ld, fill=7.0)   # columns >= Cin must not matter beyond round8
    x = c["x"].to(DEV)
    pw = mod("pack").to_device(c["pw"], DEV)
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
    ref = R.conv3x3(c["x"], B, H, W, Cin, pw, act=act, slope=0.1, compact=True)
    v = R.compare(out[:, 8:8 + Cout].cpu(), ref, b=CONV_TOL[0], rms_b=CONV_TOL[1])
    print(f"[conv] halo B={B} H={H} W={W} Cin={Cin} Cout={Cout} act={act}: {v}")
    assert v.ok, v
    # pooled means from the epilogue's partial sums (fp32 values before the bf16 rounding): AdaptiveAvgPool2d(1) of the output
    want_mean = R.channel_mean(ref, B, H * W, Cout)
    assert float((mean.cpu() - want_mean).abs().max()) < 1e-5 * max(1.0, float(want_mean.abs().max())), "pooled mean"
    assert bool(torch.isfinite(parts).all())
    # the same kernel continuing with CALayer's squeeze-excite MLP: sigmoid(W2 relu(W1 mean + b1) + b2)   (src/drn.py:128-139)
    cr = max(1, Cout // 16)
    g = torch.Generator().manual_seed(Cout)
    mlp = [torch.randn(cr, Cout, generator=g) * 0.3, torch.randn(cr, generator=g) * 0.1, torch.randn(Cout, cr, generator=g) * 0.3,
           torch.randn(Cout, generator=g) * 0.1]
    scale = torch.zeros(B, Cout, device=DEV)
    ops.channel_mean_parts(parts, B, n_parts, Cout, H * W, scale, *[t.to(DEV) for t in mlp], cr)
    torch.cuda.synchronize()
    assert float((scale.cpu() - R.channel_mean_parts(parts.cpu(), B, n_parts, Cout, H * W, mlp)).abs().max()) < 1e-5
    assert bool((out[:, :8] == -3.0).all()) and bool((out[:, 8 + n_store:] == -3.0).all())
    assert bool((out_g[:32] == -3.0).all()) and bool((out_g[-32:] == -3.0).all())
    assert bool(torch.isnan(parts_g[:8]).all()) and bool(torch.isnan(parts_g[-8:]).all())
    assert bool((out[:, 8 + Cout:8 + n_store] == 0).all())                      # padded output channels: zero weights, zero bias
    # the streaming kernel: the same reference, its own summation order
    o2 = torch.full((B * H * W, n_store + 16), -3.0, device=DEV, dtype=torch.bfloat16)
    old = ops._HALO_CONV
    ops._HALO_CONV = False
    try:
        ops.conv3x3(x, B, H, W, Cin, pw, o2, act=code, slope=0.1)
    finally:
        ops._HALO_CONV = old
    torch.cuda.synchronize()
    v = R.compare(o2[:, :Cout].cpu(), ref, b=CONV_TOL[0], rms_b=CONV_TOL[1])
    print(f"[conv] igemm B={B} H={H} W={W} Cin={Cin} Cout={Cout} act={act}: {v}")
    assert v.ok, v
    assert bool((o2[:, n_store:] == -3.0).all()) and bool((o2[:, Cout:n_store] == 0).all())


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
