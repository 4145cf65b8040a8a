"""GPU parity of the fused attention half (norm1 + qkv + shifted-window attention + proj + residual, csrc/swin_attn.cu)
against an fp32 torch restatement built on the oracle's index maps / mask / relative-position index
(src/drct.py:478-509, 271-302, 449-470)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import drct_oracle as O
from gpu_common import mod, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _want(x, gamma, beta, qkv_w, qkv_b, proj_w, proj_b, table, B, H, W, ws, shift, heads):
    """x fp32 [B*H*W, C] -> (attention rows [M, heads, hd] in token order, y = x + proj(attention))."""
    M, C = x.shape
    hd = C // heads
    N, L = ws * ws, H * W
    qkv = F.linear(F.layer_norm(x, (C,), gamma, beta, 1e-5), qkv_w, qkv_b).view(M, 3, heads, hd)
    src = O.window_source_index(H, W, ws, shift).to(x.device)           # [nW, N]
    nW = src.shape[0]

    def win(t):
        return t.reshape(B, L, heads, hd)[:, src.reshape(-1)].view(B * nW, N, heads, hd).permute(0, 2, 1, 3)

    q, k, v = win(qkv[:, 0]) * (hd ** -0.5), win(qkv[:, 1]), win(qkv[:, 2])
    attn = q @ k.transpose(-2, -1)
    rpi = O.relative_position_index(ws).to(x.device)
    attn = attn + table[rpi.reshape(-1)].view(N, N, heads).permute(2, 0, 1).unsqueeze(0)
    if shift:
        mask = O.attention_mask(H, W, ws, shift).to(x.device)
        attn = (attn.view(B, nW, heads, N, N) + mask[None, :, None]).view(B * nW, heads, N, N)
    o = (torch.softmax(attn, -1) @ v).permute(0, 2, 1, 3).reshape(B, nW * N, heads, hd)
    att = torch.empty(B, L, heads, hd, device=x.device)
    att[:, src.reshape(-1)] = o
    att = att.view(M, heads, hd)
    return att, x + F.linear(att.reshape(M, C), proj_w, proj_b)


def _case(B, H, W, C, heads, shift, fuse, seed=0):
    ops, pack = mod("ops"), mod("pack")
    torch.manual_seed(seed)
    ws, hd = 8, C // heads
    hdp = pack.head_pad(hd)
    mode = ops.swin_attn_mode(C, heads, hdp, fuse)
    assert mode == (2 if fuse else 1), f"C={C} heads={heads}: mode {mode}"
    M, ld = B * H * W, 320
    x = torch.full((M, ld), 3.0, device=DEV, dtype=torch.bfloat16)            # columns >= C hold other slab data: must be ignored
    x[:, :C] = (torch.randn(M, C, device=DEV) * 1.2 + 0.2).to(torch.bfloat16)
    xf = x[:, :C].float()
    gamma = 1.0 + 0.2 * torch.randn(C, device=DEV)
    beta = 0.1 * torch.randn(C, device=DEV)
    qkv_w = torch.randn(3 * C, C, device=DEV) * 0.08
    qkv_b = torch.randn(3 * C, device=DEV) * 0.2
    proj_w = torch.randn(C, C, device=DEV) * 0.08
    proj_b = torch.randn(C, device=DEV) * 0.2
    table = torch.randn(225, heads, device=DEV) * 0.5
    pa = pack.pack_swin_attn(qkv_w, qkv_b, gamma, beta, 1e-5, proj_w, proj_b, heads)
    stats = torch.zeros(M, 3, 2, device=DEV)
    half = C // 2
    stats[:, 0, 0], stats[:, 0, 1] = xf[:, :half].sum(1), (xf[:, :half] ** 2).sum(1)
    stats[:, 1, 0], stats[:, 1, 1] = xf[:, half:].sum(1), (xf[:, half:] ** 2).sum(1)
    stats[:, 2] = 1e9
    att_want, y_want = _want(xf, gamma, beta, qkv_w, qkv_b, proj_w, proj_b, table, B, H, W, ws, shift, heads)
    if fuse:
        out = torch.full((M, ld), -7.0, device=DEV, dtype=torch.bfloat16)
        st_out = torch.full((M, 4, 2), 1e9, device=DEV)
        ops.swin_attn(x, pa, table, out, B, H, W, shift, (stats, 2), True, stats_out=(st_out, 1))
        torch.cuda.synchronize()
        err = rel_err(out[:, :C], y_want)
        assert err < 0.012, f"C={C} heads={heads} shift={shift}: y rel err {err}"
        # the TMA store clips at the tensor-map width C rounded up to a 16-byte chunk: pad columns inside that chunk receive exact
        # zeros (zero weight rows, zero bias, zero-filled shortcut), everything beyond stays untouched
        c8 = (C + 7) // 8 * 8
        tail = out[:, C:c8].float()
        assert bool(((tail == 0.0) | (tail == -7.0)).all()), "pad columns must be zero or untouched"
        assert float((out[:, c8:].float() + 7.0).abs().max()) == 0.0, "wrote past the 16-byte chunk holding column C-1"
        yf = out[:, :C].float()
        s1, s2 = yf.sum(1), (yf ** 2).sum(1)
        assert float((st_out[:, 1, 0] - s1).abs().max() / s1.abs().max()) < 5e-3
        assert float((st_out[:, 1, 1] - s2).abs().max() / s2.abs().max()) < 5e-3
        assert float((st_out[:, 0] - 1e9).abs().max()) == 0.0 and float((st_out[:, 2:] - 1e9).abs().max()) == 0.0
    else:
        out = torch.full((M, heads * hdp), -7.0, device=DEV, dtype=torch.bfloat16)
        ops.swin_attn(x, pa, table, out, B, H, W, shift, (stats, 2), False)
        torch.cuda.synchronize()
        got = out.view(M, heads, hdp).float()
        err = float((got[:, :, :hd] - att_want).abs().max() / att_want.abs().max())
        assert err < 0.012, f"C={C} heads={heads} shift={shift}: attention rel err {err}"
        if hdp > hd:
            assert float(got[:, :, hd:].abs().max()) == 0.0, "head padding columns must be exact zeros"


@pytest.mark.parametrize("C,heads,shift", [(180, 6, 0), (212, 4, 4), (276, 6, 4), (180, 6, 4), (212, 4, 0)])
def test_swin_attn_fused_proj(C, heads, shift):
    _case(3, 32, 32, C, heads, shift, True, seed=C + shift)


@pytest.mark.parametrize("C,heads,shift", [(244, 2, 0), (308, 4, 0), (244, 2, 4), (308, 4, 4), (180, 6, 4)])
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
