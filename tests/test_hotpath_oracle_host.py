"""CPU checks of the fp64 hot-path reference (oracle/hotpath_oracle.py) and of its comparator:
  * unpack . pack is the identity on bf16-representable weights, for every packed layout;
  * with its bf16 roundings switched off, the reference equals plain torch restatements from the fp32 parameters;
  * every defect of the mutation table fails the comparator at the GPU tests' shapes, seeds and tolerances, and the
    simulated kernel noise passes it -- the tolerances are bounded from both sides without a GPU."""
import copy
import importlib

import pytest
import torch
import torch.nn.functional as F

from oracle import drct_oracle as O
from oracle import hotpath_oracle as R

pack = importlib.import_module("anomaly-detection-super-resolution_b200.pack")


def _bfw(*shape, scale=0.1, g=None):
    return (torch.randn(*shape, generator=g) * scale).to(torch.bfloat16).float()


# ------------------------------------------------------------------------------------------------ unpack . pack
@pytest.mark.parametrize("N,K,rows", [(40, 100, False), (576, 180, False), (960, 308, False), (308, 212, True), (32, 64, True)])
def test_unpack_tiles_inverts_pack(N, K, rows):
    g = torch.Generator().manual_seed(N + K)
    w = _bfw(N, K, g=g)
    pw = pack.pack_gemm_weight(w, None, rows_kernel=rows)
    u = R.unpack_tiles(pw)
    assert torch.equal(u[:N, :K], w.double()) and float(u[N:].abs().sum()) == 0.0 and float(u[:, K:].abs().sum()) == 0.0


@pytest.mark.parametrize("C,heads", [(180, 6), (212, 4), (276, 6), (244, 2), (308, 4), (60, 6)])
def test_unpack_attn_inverts_pack(C, heads):
    g = torch.Generator().manual_seed(C)
    qkv_w, proj_w = _bfw(3 * C, C, g=g), _bfw(C, C, g=g)
    pa = pack.pack_swin_attn(qkv_w, None, torch.ones(C), torch.zeros(C), 1e-5, proj_w, None, heads)
    u = R.unpack_attn(pa)
    hd, hdp = C // heads, pa.hdp
    want = torch.zeros(heads, 3, hdp, C, dtype=torch.float64)
    want[:, :, :hd] = qkv_w.double().view(3, heads, hd, C).permute(1, 0, 2, 3)
    assert torch.equal(u.wqkv, want.reshape(heads, 3 * hdp, C))
    if hdp <= 64:
        wp = torch.zeros(C, heads, hdp, dtype=torch.float64)
        wp[:, :, :hd] = proj_w.double().view(C, heads, hd)
        assert torch.equal(u.wproj, wp)
    else:
        assert u.wproj is None


@pytest.mark.parametrize("C,H,kind,Co", [(180, 360, "plain", 0), (244, 488, "plain", 0), (308, 308, "plain", 0), (60, 120, "plain", 0),
                                         (180, 360, "adjust", 0), (288, 288, "adjust", 0), (308, 308, "conv_res", 180),
                                         (244, 488, "conv_res", 180), (128, 256, "conv_res", 60)])
def test_unpack_mlp_inverts_pack(C, H, kind, Co):
    g = torch.Generator().manual_seed(C + H)
    w1, w2 = _bfw(H, C, g=g), _bfw(C, H, g=g)
    args = (w1, None, torch.ones(C), torch.zeros(C), 1e-5, w2, None)
    if kind == "plain":
        pm = pack.pack_swin_mlp(*args)
    elif kind == "adjust":
        wa = _bfw(32, C, g=g)
        pm = pack.pack_swin_mlp(*args, wa, None)
    else:
        wa = _bfw(Co, C, g=g)
        pm = pack.pack_swin_mlp_conv_res(*args, wa, None, 0.25)             # 0.25: alpha W_a stays exact in bf16
    u = R.unpack_mlp(pm)
    h_idx = torch.arange(H)                                                # hidden index j * hc + row: linear in the chunking
    assert torch.equal(u.w1[h_idx], w1.double()) and float(u.w1[H:].abs().sum()) == 0.0
    if kind == "plain":
        assert torch.equal(u.w2[:C, :H], 0.5 * w2.double()) and float(u.w2[:, H:].abs().sum()) == 0.0
    elif kind == "adjust":
        assert torch.equal(u.wadj, wa.double())
        assert torch.equal(u.w2[:, :H], R.bf16((wa.double() @ (0.5 * w2.double())).float().double()))
    else:
        assert torch.equal(u.wy[:Co], 0.25 * wa.double()) and float(u.wy[Co:].abs().sum()) == 0.0
        assert torch.equal(u.w2[:Co, :H], R.bf16(((0.25 * wa.double()) @ (0.5 * w2.double())).float().double()))


# ------------------------------------------------------------------------------------------------ pinned to plain restatements
def _swin_attn_restated(x, gamma, beta, qkv_w, qkv_b, proj_w, proj_b, table, B, H, W, ws, shift, heads):
    """The restatement the attention-half tests used: F.layer_norm + F.linear + softmax on the oracle's index maps."""
    M, C = x.shape
    hd = C // heads
    N, L = ws * ws, H * W
    qkv = F.linear(F.layer_norm(x, (C,), gamma, beta, 1e-5), qkv_w, qkv_b).view(M, 3, heads, hd)
    src = O.window_source_index(H, W, ws, shift)
    nW = src.shape[0]

    def win(t):
        return t.reshape(B, L, heads, hd)[:, src.reshape(-1)].view(B * nW, N, heads, hd).permute(0, 2, 1, 3)

    q, k, v = win(qkv[:, 0]) * (hd ** -0.5), win(qkv[:, 1]), win(qkv[:, 2])
    attn = q @ k.transpose(-2, -1)
    attn = attn + table[O.relative_position_index(ws).reshape(-1)].view(N, N, heads).permute(2, 0, 1).unsqueeze(0)
    if shift:
        attn = (attn.view(B, nW, heads, N, N) + O.attention_mask(H, W, ws, shift).to(x.dtype)[None, :, None]).view(B * nW, heads, N, N)
    o = (torch.softmax(attn, -1) @ v).permute(0, 2, 1, 3).reshape(B, nW * N, heads, hd)
    att = torch.empty(B, L, heads, hd, dtype=x.dtype)
    att[:, src.reshape(-1)] = o
    att = att.view(M, heads, hd)
    return att, x + F.linear(att.reshape(M, C), proj_w, proj_b)


@pytest.fixture
def no_rounding(monkeypatch):
    monkeypatch.setattr(R, "bf16", lambda t: t)


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max())


@pytest.mark.parametrize("C,heads,shift", [(180, 6, 4), (60, 6, 0), (244, 2, 4)])
def test_swin_attn_reference_matches_restatement(no_rounding, C, heads, shift):
    """gamma = 1 and bf16-representable weights, so the packed weights are the parameters; the rest is fp64 algebra."""
    g = torch.Generator().manual_seed(C)
    B, H, W = 2, 16, 16
    x = (torch.randn(B * H * W, C, generator=g) * 1.2 + 0.2).to(torch.bfloat16)
    qkv_w, proj_w = _bfw(3 * C, C, scale=0.08, g=g), _bfw(C, C, scale=0.08, g=g)
    qkv_b, proj_b, beta = torch.randn(3 * C, generator=g) * 0.2, torch.randn(C, generator=g) * 0.2, torch.randn(C, generator=g) * 0.1
    table = torch.randn(225, heads, generator=g) * 0.5
    pa = pack.pack_swin_attn(qkv_w, qkv_b, torch.ones(C), beta, 1e-5, proj_w, proj_b, heads)
    att, y = R.swin_attn(x, R.row_stats(x, 3), 2, pa, table, B, H, W, shift, pa.hdp <= 64)
    d = lambda t: t.double()
    att_w, y_w = _swin_attn_restated(d(x), torch.ones(C, dtype=torch.float64), d(beta), d(qkv_w), d(qkv_b), d(proj_w), d(proj_b),
                                     d(table), B, H, W, 8, shift, heads)
    assert _rel(att[:, :, :C // heads], att_w) < 1e-6               # pack folds beta into the bias in fp32
    if y is not None:
        assert _rel(y - d(x), y_w - d(x)) < 1e-6


def test_window_attention_reference_matches_restatement():
    case = R.attention_case(2, 16, 16, 4, 2, 4, 23, 5)
    q = case["qkv"].double().view(-1, 3, 4, case["hdp"])[..., :23]
    ref = R.attention_ref(case)[:, :, :23]
    # _swin_attn_restated's chain without LayerNorm and projections
    N, src = 16, O.window_source_index(16, 16, 4, 2)
    win = lambda t: t.reshape(2, 256, 4, 23)[:, src.reshape(-1)].view(2 * 16, N, 4, 23).permute(0, 2, 1, 3)
    s = win(q[:, 0]) * 23 ** -0.5 @ win(q[:, 1]).transpose(-2, -1)
    s = s + case["table"].double()[O.relative_position_index(4).reshape(-1)].view(N, N, 4).permute(2, 0, 1)
    s = (s.view(2, 16, 4, N, N) + O.attention_mask(16, 16, 4, 2).double()[None, :, None]).view(32, 4, N, N)
    o = (torch.softmax(s, -1) @ win(q[:, 2])).permute(0, 2, 1, 3).reshape(2, 256, 4, 23)
    want = torch.empty(2, 256, 4, 23, dtype=torch.float64)
    want[:, src.reshape(-1)] = o
    assert _rel(ref, want.view(512, 4, 23)) < 1e-12


@pytest.mark.parametrize("kind", ["plain", "adjust", "conv_res"])
def test_swin_mlp_reference_matches_restatement(no_rounding, kind):
    g = torch.Generator().manual_seed(7)
    M, C, H, Co = 300, 180, 360, 60
    y = (torch.randn(M, C, generator=g) * 1.5 + 0.3).to(torch.bfloat16)
    w1, w2 = _bfw(H, C, scale=0.08, g=g), _bfw(C, H, scale=0.08, g=g)
    b1, b2, beta = torch.randn(H, generator=g) * 0.2, torch.randn(C, generator=g) * 0.2, torch.randn(C, generator=g) * 0.1
    args = (w1, b1, torch.ones(C), beta, 1e-5, w2, b2)
    d = lambda t: t.double()
    z = d(y) + F.linear(F.gelu(F.linear(F.layer_norm(d(y), (C,), None, d(beta), 1e-5), d(w1), d(b1))), d(w2), d(b2))
    res = None
    if kind == "plain":
        pm, want, sc = pack.pack_swin_mlp(*args), z, d(y)
    elif kind == "adjust":
        wa, ba = _bfw(32, C, g=g), torch.randn(32, generator=g) * 0.2
        pm, want, sc = pack.pack_swin_mlp(*args, wa, ba), F.leaky_relu(F.linear(z, d(wa), d(ba)), 0.2), None
    else:
        wa, ba = _bfw(Co, C, g=g), torch.randn(Co, generator=g) * 0.2
        res = (torch.randn(M, Co, generator=g) * 2).to(torch.bfloat16)
        pm = pack.pack_swin_mlp_conv_res(*args, wa, ba, 0.25)
        want, sc = d(res) + 0.25 * F.linear(z, d(wa), d(ba)), d(res)
    got = R.swin_mlp(y, R.row_stats(y, 3), 2, pm, res=res)
    # W_adj W2 / alpha W_a W2 are formed in fp64 and stored as fp32 before the slab's bf16: bf16 when rounding is on, fp32 here
    tol = 1e-6 if kind == "plain" else 2e-3
    assert _rel(got - (0 if sc is None else sc), want - (0 if sc is None else sc)) < tol


@pytest.mark.parametrize("ln,act,rows", [(False, "gelu", False), (False, "lrelu", True), (True, "gelu", True), (True, "none", False)])
def test_gemm_reference_matches_restatement(ln, act, rows):
    g = torch.Generator().manual_seed(3)
    M, K, N = 300, 212, 424
    a = (torch.randn(M, K, generator=g) * 2.5 + 1.5 * torch.randn(M, 1, generator=g)).to(torch.bfloat16)
    w, b, beta = _bfw(N, K, g=g), torch.randn(N, generator=g), torch.randn(K, generator=g) * 0.3
    d = lambda t: t.double()
    if ln:
        pw = pack.pack_ln_gemm_weight(w, b, torch.ones(K), beta, 1e-5, rows_kernel=rows)
        want = F.linear(F.layer_norm(d(a), (K,), None, d(beta), 1e-5), d(w), d(b))
    else:
        pw = pack.pack_gemm_weight(w, b, rows_kernel=rows)
        want = F.linear(d(a), d(w), d(b))
    want = F.gelu(want) if act == "gelu" else F.leaky_relu(want, 0.2) if act == "lrelu" else want
    got = R.gemm(a, K, pw, act=act, slope=0.2, stats=R.row_stats(a, 2, split=1), slots=1)
    assert _rel(got, want) < 1e-6


# ------------------------------------------------------------------------------------------------ mutation table
# Each defect is stated on the reference, at the shape and seed of a GPU case, and must FAIL the comparator against the
# unmutated reference; the simulated kernel noise must PASS it.  The mean/std = 10 cases carry the defects that only show
# when rows have a mean (colsum), the 2^-6 shortcut cases those that hide under the shortcut's rounding (eps).
def _attn(case, fuse, **kw):
    c = dict(case)
    for k in ("pa", "stats", "table"):
        if k in kw:
            c[k] = kw.pop(k)
    att, y = R.swin_attn(c["x"], c["stats"], 2, c["pa"], c["table"], c["B"], c["H"], c["W"], c["shift"], fuse, **kw)
    return y if fuse else att


def _attn_cases():
    fused = R.swin_attn_case(3, 32, 32, 180, 6, 4, 184, shortcut_scale=2.0 ** -6)
    fused_ms = R.swin_attn_case(3, 32, 32, 180, 6, 4, 190, mean_std=10, shortcut_scale=2.0 ** -6)
    only = R.swin_attn_case(3, 32, 32, 244, 2, 4, 248)
    return {"fused": (fused, True), "fused_ms10": (fused_ms, True), "attention_only": (only, False)}


def _colsum_fp32(case):
    pa, raw = copy.copy(case["pa"]), case["raw"]
    C, heads, hd, hdp = pa.C, pa.heads, pa.hd, pa.hdp
    wg = torch.zeros(heads, 3, hdp, C)
    wg[:, :, :hd] = (raw["qkv_w"] * raw["gamma"][None]).view(3, heads, hd, C).permute(1, 0, 2, 3)
    pa.colsum_qkv = wg.sum(-1).reshape(-1)
    return pa


def _attn_defects(case):
    pa, heads, hdp, shift = case["pa"], case["pa"].heads, case["pa"].hdp, case["shift"]
    tb = case["table"].clone()
    tb[7 * 15 + 7, heads - 1] += 0.25                              # offset (0, 0): every query's own key
    eps = copy.copy(pa)
    eps.ln_eps = 1e-3
    m = O.attention_mask(case["H"], case["W"], 8, shift).clone()
    m[-1, :, 56:] = 0.0                                             # last window: keys of the wrap row ...
    m[-1, :, 7::8] = 0.0                                            # ... and of the wrap column unmasked
    rpi = O.relative_position_index(8).clone()
    rpi[13] = rpi[14]                                               # query 13 reads query 14's bias row
    vb = copy.copy(pa)
    b = pa.bias_qkv.clone().view(heads, 3, hdp)
    b[heads // 2, 2] = 0.0
    vb.bias_qkv = b.reshape(-1)
    st = case["stats"].clone()
    st[:, 1] = 0.0
    return {"bias entry +0.25": dict(table=tb), "softmax scale +1%": dict(scale=1.01 * pa.hd ** -0.5),
            "softmax scale from hdp": dict(scale=pa.hdp ** -0.5), "LayerNorm eps 1e-3": dict(pa=eps),
            "mask dropped on the wrap row / column": dict(mask=m), "neighbour's bias row": dict(rpi=rpi),
            "v bias of one head dropped": dict(pa=vb), "stats slot ignored": dict(stats=st),
            "colsum from fp32 weights": dict(pa=_colsum_fp32(case))}


ATTN_TABLE = [
    ("fused", "bias entry +0.25"), ("fused", "softmax scale +1%"), ("fused", "softmax scale from hdp"),
    ("fused", "LayerNorm eps 1e-3"), ("fused", "mask dropped on the wrap row / column"), ("fused", "neighbour's bias row"),
    ("fused", "v bias of one head dropped"), ("fused", "stats slot ignored"), ("fused_ms10", "colsum from fp32 weights"),
    ("attention_only", "bias entry +0.25"), ("attention_only", "softmax scale +1%"), ("attention_only", "softmax scale from hdp"),
    ("attention_only", "mask dropped on the wrap row / column"), ("attention_only", "neighbour's bias row"),
    ("attention_only", "v bias of one head dropped"), ("attention_only", "stats slot ignored"),
]


@pytest.fixture(scope="module")
def attn_cases():
    return _attn_cases()


def _verdict(got, ref, shortcut, kernel):
    b, rb = R.TOL[kernel]
    return R.compare(got, ref, shortcut, b=b, rms_b=rb)


@pytest.mark.parametrize("which,defect", ATTN_TABLE)
def test_swin_attn_defect_fails(attn_cases, which, defect):
    case, fuse = attn_cases[which]
    ref = _attn(case, fuse)
    got = _attn(case, fuse, **_attn_defects(case)[defect])
    sc = case["x"].double() if fuse else None
    v = _verdict(got, ref, sc, "swin_attn")
    assert not v.ok, f"{which}: '{defect}' passes the comparator: {v}"


@pytest.mark.parametrize("which", ["fused", "fused_ms10", "attention_only"])
def test_swin_attn_kernel_noise_passes(attn_cases, which):
    case, fuse = attn_cases[which]
    ref = _attn(case, fuse)
    v = _verdict(R.bf16(_attn(case, fuse, noise=True).double()), ref, case["x"].double() if fuse else None, "swin_attn")
    assert v.ok, f"{which}: simulated kernel noise fails: {v}"


@pytest.mark.parametrize("defect", ["bias entry +0.25", "softmax scale +1%", "softmax scale from hdp", "mask dropped on the wrap row / column",
                                    "neighbour's bias row"])
@pytest.mark.parametrize("ws", [8, 16])
def test_window_attention_defect_fails(ws, defect):
    case = R.attention_case(2 if ws == 8 else 1, 32 if ws == 8 else 64, 32 if ws == 8 else 64, ws, ws // 2, 6, 30, 30 + ws // 2)
    ref = R.attention_ref(case)
    n, c = ws * ws, ws - 1
    kw = {}
    if defect == "bias entry +0.25":
        tb = case["table"].clone()
        tb[c * (2 * ws - 1) + c, 0] += 0.25
        case = dict(case, table=tb)
    elif defect.startswith("softmax scale"):
        kw["scale"] = 1.01 * 30 ** -0.5 if defect.endswith("1%") else 32 ** -0.5
    elif defect.startswith("mask"):
        m = O.attention_mask(case["H"], case["W"], ws, ws // 2).clone()
        m[-1, :, n - ws:] = 0.0
        m[-1, :, ws - 1::ws] = 0.0
        kw["mask"] = m
    else:
        rpi = O.relative_position_index(ws).clone()
        rpi[n // 2 - 3] = rpi[n // 2 - 2]
        kw["rpi"] = rpi
    v = _verdict(R.attention_ref(case, **kw), ref, None, "attention")
    assert not v.ok, f"ws={ws}: '{defect}' passes the comparator: {v}"


@pytest.mark.parametrize("ws,edge", [(8, None), (16, None), (8, "masked_max"), (16, "peaked")])
def test_window_attention_kernel_noise_passes(ws, edge):
    kw = dict(masked_max=True) if edge == "masked_max" else dict(qk_scale=3.5, bias_range=8.0) if edge == "peaked" else {}
    case = R.attention_case(2 if ws == 8 else 1, 32 if ws == 8 else 64, 32 if ws == 8 else 64, ws, ws // 2, 6, 30, 30 + ws // 2, **kw)
    ref = R.attention_ref(case)
    v = _verdict(R.bf16(R.attention_ref(dict(case, qkv=case["qkv"].float()), noise=True).double()), ref, None, "attention")
    assert v.ok, f"ws={ws} {edge}: simulated kernel noise fails: {v}"


def _mlp_defect(case, defect):
    pm, raw = copy.copy(case["pm"]), case["raw"]
    kw, stats = {}, case["stats"]
    if defect == "LayerNorm eps 1e-3":
        pm.ln_eps = 1e-3
    elif defect == "stats slot ignored":
        stats = stats.clone()
        stats[:, 1] = 0.0
    elif defect == "colsum from fp32 weights":
        c1 = pm.colsum1.clone()
        c1[:raw["w1"].shape[0]] = (raw["w1"] * raw["gamma"][None]).sum(1)
        pm.colsum1 = c1
    elif defect == "tanh GELU":
        kw["gelu_kind"] = "tanh"
    elif defect == "adjust slope 0.01":
        kw["slope"] = 0.01
    return R.swin_mlp(case["y"], stats, 2, pm, res=case["res"], **kw)


def _mlp_shortcut(case):
    return case["y"].double() if case["kind"] == "plain" else case["res"].double() if case["kind"] == "conv_res" else None


MLP_CASES = {
    "plain": dict(M=677, C=180, H=360, seed=180, shortcut_scale=2.0 ** -6),
    "plain_ms10": dict(M=677, C=180, H=360, seed=10, mean_std=10, shortcut_scale=2.0 ** -6),
    "adjust": dict(M=677, C=180, H=360, seed=180, kind="adjust"),
    "conv_res": dict(M=677, C=308, H=308, seed=488, kind="conv_res", Co=180, shortcut_scale=2.0 ** -6),
    "conv_res_ms10": dict(M=677, C=308, H=308, seed=10, kind="conv_res", Co=180, mean_std=10, shortcut_scale=2.0 ** -6),
}


@pytest.mark.parametrize("which,defect", [
    ("plain", "LayerNorm eps 1e-3"), ("plain", "stats slot ignored"), ("plain_ms10", "colsum from fp32 weights"),
    ("adjust", "stats slot ignored"), ("adjust", "adjust slope 0.01"),
    ("conv_res", "LayerNorm eps 1e-3"), ("conv_res", "stats slot ignored"),
    ("conv_res_ms10", "colsum from fp32 weights"),
])
def test_swin_mlp_defect_fails(which, defect):
    kw = dict(MLP_CASES[which])
    case = R.mlp_case(kw.pop("M"), kw.pop("C"), kw.pop("H"), kw.pop("seed"), **kw)
    ref = R.swin_mlp(case["y"], case["stats"], 2, case["pm"], res=case["res"])
    v = _verdict(_mlp_defect(case, defect), ref, _mlp_shortcut(case), "swin_mlp")
    assert not v.ok, f"{which}: '{defect}' passes the comparator: {v}"


@pytest.mark.parametrize("which", ["plain", "conv_res"])
def test_tanh_gelu_is_below_bf16_resolution(which):
    """tanh-approximated GELU moves the MLP branch by about 0.005 rms(branch) at most -- inside the noise of bf16 activations
    (B200: 0.0085), so no comparator on the bf16 output can tell it apart; pinned here so the limit is a known one."""
    kw = dict(MLP_CASES[which])
    case = R.mlp_case(kw.pop("M"), kw.pop("C"), kw.pop("H"), kw.pop("seed"), **kw)
    ref = R.swin_mlp(case["y"], case["stats"], 2, case["pm"], res=case["res"])
    v = R.compare(_mlp_defect(case, "tanh GELU"), ref, _mlp_shortcut(case), b=0.0, rms_b=0.0)
    assert 0.002 < v.max_units < 0.008


@pytest.mark.parametrize("which", list(MLP_CASES))
def test_swin_mlp_kernel_noise_passes(which):
    kw = dict(MLP_CASES[which])
    case = R.mlp_case(kw.pop("M"), kw.pop("C"), kw.pop("H"), kw.pop("seed"), **kw)
    ref = R.swin_mlp(case["y"], case["stats"], 2, case["pm"], res=case["res"])
    got = R.bf16(R.swin_mlp(case["y"], case["stats"], 2, case["pm"], res=case["res"], noise=True).double())
    v = _verdict(got, ref, _mlp_shortcut(case), "swin_mlp")
    assert v.ok, f"{which}: simulated kernel noise fails: {v}"


@pytest.mark.parametrize("rows", [False, True])
@pytest.mark.parametrize("defect", ["LayerNorm eps 1e-3", "stats slot ignored", "colsum from fp32 weights"])
def test_ln_gemm_defect_fails(defect, rows):
    case = R.ln_gemm_case(128 * 20 + 37, 212, 424, 212 + 424 + 10, rows=rows, mean_std=10)
    pw, st = copy.copy(case["pw"]), case["stats"]
    if defect == "LayerNorm eps 1e-3":                              # rows of variance ~4e-3, where eps 1e-3 is not negligible
        a = (case["a"].float() * 2.0 ** -4).to(torch.bfloat16)
        st = R.row_stats(a, 4, split=1)
        st[:, 1], st[:, 2:] = 0.0, 1e9
        case = dict(case, a=a, stats=st)
        pw.ln_eps = 1e-3
    elif defect == "stats slot ignored":
        st = st.clone()
        st[:, 1] = 0.0
    else:
        cs = pw.colsum.clone()
        cs[:424] = (case["raw"]["w"] * case["raw"]["gamma"][None]).sum(1)
        pw.colsum = cs
    ref = R.gemm(case["a"], 212, case["pw"], act="gelu", stats=case["stats"], slots=2)
    v = _verdict(R.gemm(case["a"], 212, pw, act="gelu", stats=st, slots=2), ref, None, "gemm")
    assert not v.ok, f"'{defect}' passes the comparator: {v}"


@pytest.mark.parametrize("mean_std", [None, 10, 100])
def test_ln_gemm_kernel_noise_passes(mean_std):
    case = R.ln_gemm_case(128 * 20 + 37, 212, 424, 212 + 424 + (mean_std or 0), mean_std=mean_std)
    ref = R.gemm(case["a"], 212, case["pw"], act="gelu", stats=case["stats"], slots=2)
    got = R.bf16(R.gemm(case["a"], 212, case["pw"], act="gelu", stats=case["stats"], slots=2, noise=True).double())
    v = _verdict(got, ref, None, "gemm")
    assert v.ok, f"mean/std {mean_std}: simulated kernel noise fails: {v}"


def test_one_pass_variance_breaks_down_beyond_the_supported_range():
    """At mean/std = 300 the fp32 one-pass variance the kernels use fails the attention comparator: the supported range ends
    at 100 (DESIGN.md section 2)."""
    case = R.swin_attn_case(3, 32, 32, 180, 6, 4, 480, mean_std=300, shortcut_scale=2.0 ** -6)
    ref = _attn(case, True)
    v = _verdict(R.bf16(_attn(case, True, noise=True).double()), ref, case["x"].double(), "swin_attn")
    assert not v.ok


# ------------------------------------------------------------------------------------------------ convolutions and the RCAB
@pytest.mark.parametrize("cin", [3, 20, 40, 64, 72, 80, 96, 128, 180])
@pytest.mark.parametrize("cout", [16, 20, 40, 64, 80, 256])
def test_unpack_conv_inverts_pack(cin, cout):
    g = torch.Generator().manual_seed(cin * 1000 + cout)
    w = _bfw(cout, cin, 3, 3, g=g)
    pw = pack.pack_conv3x3_weight(w, None)
    assert torch.equal(R.unpack_conv(pw), w.double())
    slabs = (9 * ((cin + 15) // 16 * 16) + 63) // 64
    fits = cin <= 128 and cout <= 128 and slabs * ((cout + 15) // 16 * 16) * 128 <= 126 * 1024   # halo weights resident in smem
    assert (pw.compact is not None) == fits
    if fits:
        assert torch.equal(R.unpack_conv(pw, compact=True), w.double())


def test_conv_references_match_restatement(no_rounding):
    """Plain F.conv2d / torch restatements from the fp32 parameters (bf16-representable weights, so packing is exact)."""
    g = torch.Generator().manual_seed(11)
    B, H, W, C = 2, 12, 20, 40
    x = torch.randn(B * H * W, C, generator=g).to(torch.bfloat16)
    w, b = _bfw(C, C, 3, 3, g=g), torch.randn(C, generator=g)
    pw = pack.pack_conv3x3_weight(w, b)
    xin = x.double().view(B, H, W, C).permute(0, 3, 1, 2)
    pre = F.conv2d(xin, w.double(), b.double(), padding=1)
    rows = lambda t: t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])
    res = torch.randn(B * H * W, C, generator=g).to(torch.bfloat16)
    for compact in (False, True):
        assert torch.allclose(R.conv3x3(x, B, H, W, C, pw, act="lrelu", slope=0.2, compact=compact), rows(F.leaky_relu(pre, 0.2)),
                              rtol=0, atol=1e-12)
    assert torch.allclose(R.conv3x3(x, B, H, W, C, pw, alpha=0.5, res=res), rows(0.5 * pre) + res.double(),
                          rtol=0, atol=1e-12)
    assert torch.allclose(R.conv3x3(x, B, H, W, C, pw, ps=True), rows(F.pixel_shuffle(pre, 2)), rtol=0, atol=1e-12)
    s2 = F.conv2d(xin, w.double(), b.double(), stride=2, padding=1)
    assert torch.allclose(R.conv3x3(x, B, H, W, C, pw, stride=2), rows(s2), rtol=0, atol=1e-12)
    assert torch.allclose(R.conv_pre(xin, w, b, 2, noise=True).double(), s2, rtol=0, atol=1e-4)
    xs = torch.randn(B, 3, H, W, generator=g)
    ws, bs = torch.randn(20, 3, 3, 3, generator=g), torch.randn(20, generator=g)
    assert torch.allclose(R.conv3x3_small(xs, ws, bs), rows(F.conv2d(xs.double(), ws.double(), bs.double(), padding=1)), rtol=0, atol=1e-12)
    # the CA chain: AdaptiveAvgPool2d(1) -> 1x1 conv -> ReLU -> 1x1 conv -> sigmoid, then x + t2 * s
    t2 = torch.randn(B * H * W, C, generator=g).to(torch.bfloat16)
    mlp = (torch.randn(2, C, generator=g), torch.randn(2, generator=g), torch.randn(C, 2, generator=g), torch.randn(C, generator=g))
    t2n = t2.double().view(B, H, W, C).permute(0, 3, 1, 2)
    d = [m.double() for m in mlp]
    s = torch.sigmoid(F.conv2d(F.relu(F.conv2d(F.adaptive_avg_pool2d(t2n, 1), d[0][:, :, None, None], d[1])), d[2][:, :, None, None], d[3]))
    parts = t2.float().view(B, 4, H * W // 4, C).sum(2).reshape(B * 4, C)
    assert torch.allclose(R.channel_mean(t2, B, H * W, C), t2n.mean((2, 3)), rtol=0, atol=1e-12)
    assert torch.allclose(R.channel_mean_parts(parts, B, 4, C, H * W, mlp), s.view(B, C), rtol=0, atol=1e-6)
    assert torch.allclose(R.rcab_ca_scale(t2, x, s.view(B, C), B, H * W, C), rows(xin + t2n * s), rtol=0, atol=1e-12)


# The GPU conv cases of tests/test_gpu_gemm.py (shape, seed, epilogue) that carry a conv defect.
CONV_CASES = {
    "before_upsample": dict(B=2, H=32, W=32, Cin=180, Cout=64, seed=2, act="lrelu", slope=0.01),
    "downblock": dict(B=2, H=33, W=17, Cin=80, Cout=80, seed=33, act="lrelu", slope=0.2, stride=2),
    "tail_panel": dict(B=5, H=17, W=24, Cin=72, Cout=48, seed=72, act="lrelu", slope=0.1),
    "second_panel": dict(B=2, H=16, W=40, Cin=100, Cout=48, seed=100),
    "pixel_shuffle": dict(B=2, H=32, W=32, Cin=64, Cout=256, seed=3, ps=True),
    "res_lrelu": dict(B=2, H=24, W=24, Cin=64, Cout=64, seed=24, act="lrelu", slope=0.2, res=True),
}


def _conv_ref(case, kw, *, w=None, bias=None, xin=None, pre=None, mutate_pre=None, **over):
    kw = dict(kw, **over)
    B, H, W, cin, stride = kw["B"], kw["H"], kw["W"], kw["Cin"], kw.get("stride", 1)
    if pre is None:
        w = R.unpack_conv(case["pw"]) if w is None else w
        bias = case["pw"].bias[:kw["Cout"]] if bias is None else bias
        pre = R.conv_pre(R.conv_input(case["x"], B, H, W, cin) if xin is None else xin, w, bias, stride)
    if mutate_pre is not None:
        pre = mutate_pre(pre)
    return R.conv_epilogue(pre, act=kw.get("act", "none"), slope=kw.get("slope", 0.0), res=case["res"], ps=kw.get("ps", False))


def _conv_defect(case, kw, defect):
    B, H, W, cin = kw["B"], kw["H"], kw["W"], kw["Cin"]
    w, xin = R.unpack_conv(case["pw"]), R.conv_input(case["x"], B, H, W, cin)
    if defect == "ReLU for LeakyReLU":
        return _conv_ref(case, kw, act="relu")
    if defect == "slope 0.2 -> 0.22":
        return _conv_ref(case, kw, slope=0.22)
    if defect == "tap dropped on the last column":
        w2 = w.clone()
        w2[:, :, 1, 0] = 0.0                                      # the left neighbour: inside the image
        drop = R.conv_pre(xin, w2, case["pw"].bias[:kw["Cout"]], kw.get("stride", 1))

        def m(pre):
            pre = pre.clone()
            pre[..., -1] = drop[..., -1]
            return pre
        return _conv_ref(case, kw, mutate_pre=m)
    if defect == "replicate padding on the left border":
        xp = F.pad(xin, (1, 1, 1, 1))
        xp[..., 1:-1, 0] = xp[..., 1:-1, 1]
        pre = F.conv2d(xp, w, case["pw"].bias[:kw["Cout"]].double(), stride=kw.get("stride", 1))
        return _conv_ref(case, kw, pre=pre)
    if defect == "tail panel dropped for one tap":
        w2 = w.clone()
        w2[:, 64:80, 0, 0] = 0.0
        return _conv_ref(case, kw, w=w2)
    if defect == "last channel of the second panel dropped":
        w2 = w.clone()
        w2[:, cin - 1] = 0.0
        return _conv_ref(case, kw, w=w2)
    if defect == "bias missing on one channel":
        b = case["pw"].bias[:kw["Cout"]].clone()
        b[-1] = 0.0
        return _conv_ref(case, kw, bias=b)
    if defect == "pixel-shuffle sub-pixels transposed":
        n = kw["Cout"]
        perm = torch.arange(n).view(n // 4, 2, 2).transpose(1, 2).reshape(-1)
        return _conv_ref(case, kw, mutate_pre=lambda pre: pre[:, perm])
    if defect == "stride-2 phase off by one":
        pre = F.conv2d(F.pad(xin, (0, 1, 0, 1)), w, case["pw"].bias[:kw["Cout"]].double(), padding=1)[..., 1::2, 1::2]
        return _conv_ref(case, kw, pre=pre)
    if defect == "residual added before the activation":
        pre = R.conv_pre(xin, w, case["pw"].bias[:kw["Cout"]])
        r = case["res"][:, :kw["Cout"]].double().view(B, H, W, -1).permute(0, 3, 1, 2)
        return R.conv_epilogue(pre + r, act=kw["act"], slope=kw["slope"])
    raise KeyError(defect)


CONV_TABLE = [
    ("before_upsample", "ReLU for LeakyReLU"), ("before_upsample", "bias missing on one channel"),
    ("before_upsample", "tap dropped on the last column"), ("before_upsample", "replicate padding on the left border"),
    ("downblock", "slope 0.2 -> 0.22"), ("downblock", "stride-2 phase off by one"), ("downblock", "tap dropped on the last column"),
    ("tail_panel", "tail panel dropped for one tap"), ("tail_panel", "replicate padding on the left border"),
    ("second_panel", "last channel of the second panel dropped"), ("pixel_shuffle", "pixel-shuffle sub-pixels transposed"),
    ("res_lrelu", "residual added before the activation"), ("res_lrelu", "slope 0.2 -> 0.22"),
]


def _conv_case(which):
    kw = CONV_CASES[which]
    case = R.conv_case(kw["B"], kw["H"], kw["W"], kw["Cin"], kw["Cout"], kw["seed"], res=kw.get("res", False))
    return case, kw


def _conv_shortcut(case, kw):
    return None if case["res"] is None else case["res"][:, :kw["Cout"]]


@pytest.mark.parametrize("which,defect", CONV_TABLE)
def test_conv_defect_fails(which, defect):
    case, kw = _conv_case(which)
    ref = _conv_ref(case, kw)
    v = _verdict(_conv_defect(case, kw, defect), ref, _conv_shortcut(case, kw), "conv")
    assert not v.ok, f"{which}: '{defect}' passes the comparator: {v}"


def test_relu_for_leaky_relu_passed_the_old_bound():
    """At the conv_before_upsample shape the old bound (1.2 % of max|y|) took a ReLU for LeakyReLU(0.01)."""
    case, kw = _conv_case("before_upsample")
    ref, bad = _conv_ref(case, kw), R.bf16(_conv_defect(case, kw, "ReLU for LeakyReLU"))
    assert float((bad - ref).abs().max() / ref.abs().max()) < 0.012
    assert not _verdict(bad, ref, None, "conv").ok


@pytest.mark.parametrize("which", list(CONV_CASES))
def test_conv_kernel_noise_passes(which):
    case, kw = _conv_case(which)
    args = (case["x"], kw["B"], kw["H"], kw["W"], kw["Cin"], case["pw"])
    ep = dict(stride=kw.get("stride", 1), act=kw.get("act", "none"), slope=kw.get("slope", 0.0), res=case["res"], ps=kw.get("ps", False))
    got = R.bf16(R.conv3x3(*args, noise=True, **ep).double())
    v = _verdict(got, R.conv3x3(*args, **ep), _conv_shortcut(case, kw), "conv")
    assert v.ok, f"{which}: simulated kernel noise fails: {v}"


RCAB_CASES = {"halo_64": (4, 64, 64, 40), "halo_32": (4, 32, 32, 80), "fallback_128": (2, 128, 128, 40)}


def _rcab(which, **kw):
    B, H, W, C = RCAB_CASES[which]
    case = R.rcab_case(B, H, W, C, H + C)
    return case, R.rcab(case["x"], B, H, W, case["c1"], case["c2"], case["mlp"], **kw)


@pytest.mark.parametrize("which,defect", [(w, d) for w in RCAB_CASES for d in ("neighbour's scales", "sigmoid dropped")]
                         + [("halo_64", "pad columns pooled"), ("halo_32", "pad columns pooled")])
def test_rcab_defect_fails(which, defect):
    B, H, W, C = RCAB_CASES[which]
    case, ref = _rcab(which)
    mlp = case["mlp"]
    kw = {"neighbour's scales": dict(scale_fn=lambda m: R.ca_scale(m, *mlp).roll(1, 0)),
          "sigmoid dropped": dict(scale_fn=lambda m: torch.logit(R.ca_scale(m, *mlp))),
          "pad columns pooled": dict(pool_hw=H * (W + 2))}[defect]
    _, got = _rcab(which, **kw)
    v = _verdict(got, ref, case["x"][:, :C], "rcab")
    assert not v.ok, f"{which}: '{defect}' passes the comparator: {v}"


@pytest.mark.parametrize("which", list(RCAB_CASES))
def test_rcab_kernel_noise_passes(which):
    case, ref = _rcab(which)
    _, got = _rcab(which, noise=True)
    v = _verdict(R.bf16(got), ref, case["x"][:, :RCAB_CASES[which][3]], "rcab")
    assert v.ok, f"{which}: simulated kernel noise fails: {v}"
