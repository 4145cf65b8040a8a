"""TEST INFRASTRUCTURE ONLY -- fp64 reference of the model's hot path, built from the bytes the kernels read.

Covers the fused attention half (csrc/swin_attn.cu), the standalone window attention (csrc/attention*.cu), the fused
Swin MLP with its three epilogues (csrc/swin_mlp.cu) and the GEMM kernels with or without the folded LayerNorm
(csrc/tc_gemm*.cu), the 3x3 convs on every dispatch branch (csrc/conv_halo.cu and the implicit GEMM) and DRN's CALayer / RCAB
kernels (csrc/drn_ops.cu).

Every weight comes from the packed images (unpack_* below invert pack._swizzle_slab / pack._swizzle_tiles), so the
reference uses the kernels' own gamma fold and its bf16 rounding, colsum from the bf16 weights, GELU's 0.5 in fc2, the
W_adj W2 and alpha W_a W2 products and the head padding.  LayerNorm is taken from the same (sum, sumsq) slots the kernel
is given.  Values are rounded to bf16 wherever a kernel keeps them in bf16 between two of its stages: q | k | v after the
folded LayerNorm, the normalised attention output O, and the GELU activations fc2 reads.  Stored outputs are returned
BEFORE their final rounding: `compare` charges that rounding as half an ulp plus zero-mean noise.

What the reference cannot mirror -- P rounded to bf16 after an exp shifted by a different maximum, the fp32 accumulation
order, ex2.approx, fp32 LayerNorm arithmetic -- belongs to the error budget.  `noise=True` runs the same chain with those
roundings simulated (fp32 arithmetic, the kernels' softmax), so a host test can show that the budget covers them.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

from oracle import drct_oracle as O

F64 = torch.float64


def bf16(t: torch.Tensor) -> torch.Tensor:
    """Round to bf16 (nearest even), keep the dtype."""
    return t.to(torch.bfloat16).to(t.dtype)


def _bf16_words(img: torch.Tensor) -> torch.Tensor:
    return img.contiguous().view(torch.bfloat16)


# ------------------------------------------------------------------------------------------------ unpacking
def unswizzle_slab(img: torch.Tensor, rows: int) -> torch.Tensor:
    """Inverse of pack._swizzle_slab: uint8 image of [rows x 64] bf16 (row r at r * 128 B, 16-byte chunk c at position
    c ^ (r % 8)) -> fp64 [rows, 64]."""
    t = _bf16_words(img).view(rows, 8, 8)
    r = torch.arange(rows, device=t.device)
    pos = torch.arange(8, device=t.device)
    idx = (pos[None, :] ^ (r[:, None] % 8))[:, :, None].expand(rows, 8, 8)
    return torch.gather(t, 1, idx).reshape(rows, 64).to(F64)


def unpack_tiles(pw) -> torch.Tensor:
    """Inverse of pack._swizzle_tiles: PackedWeight.data -> fp64 [n_tiles * BN, k_stages * 64] (padding included)."""
    nt, ks, bn = pw.n_tiles, pw.k_stages, pw.BN
    t = _bf16_words(pw.data).view(nt, ks, bn, 8, 8)
    r = torch.arange(bn, device=t.device)
    pos = torch.arange(8, device=t.device)
    idx = (pos[None, :] ^ (r[:, None] % 8))[None, None, :, :, None].expand(nt, ks, bn, 8, 8)
    w = torch.gather(t, 3, idx)                                   # [tile, ks, row, chunk, elem]
    return w.permute(0, 2, 1, 3, 4).reshape(nt * bn, ks * 64).to(F64)


@dataclass
class AttnWeights:
    wqkv: torch.Tensor        # [heads, 3 * hdp, C]: q_h | k_h | v_h rows, gamma folded, bf16 values
    colsum: torch.Tensor      # [heads, 3 * hdp]
    bias: torch.Tensor        # [heads, 3 * hdp]
    wproj: torch.Tensor       # [C, heads, hdp] (None when proj is not packed)
    bias_p: torch.Tensor      # [C]


def unpack_attn(pa) -> AttnWeights:
    c, nh, hdp = pa.C, pa.heads, pa.hdp
    ks = (c + 63) // 64
    cp = (c + 15) // 16 * 16
    slab = 3 * hdp * 128
    w = torch.stack([torch.cat([unswizzle_slab(pa.w1[(h * ks + s) * slab:(h * ks + s + 1) * slab], 3 * hdp) for s in range(ks)], 1)
                     for h in range(nh)])[:, :, :c]
    wp = None
    if hdp <= 64:
        wp = torch.stack([unswizzle_slab(pa.w2[h * cp * 128:(h + 1) * cp * 128], cp)[:c, :hdp] for h in range(nh)], 1)
    return AttnWeights(w, pa.colsum_qkv.to(F64).view(nh, 3 * hdp), pa.bias_qkv.to(F64).view(nh, 3 * hdp), wp,
                       pa.bias_p.to(F64)[:c])


@dataclass
class MlpWeights:
    w1: torch.Tensor          # [nc * hc, C]: fc1 rows, gamma folded (hidden index j * hc + row of chunk j)
    w2: torch.Tensor          # [n2, nc * hc]: fc2 (0.5 of GELU folded; W_adj W2 or alpha W_a W2 when folded)
    wy: torch.Tensor          # [n2, C]: the y term of a folded wide conv (alpha W_a), else None
    wadj: torch.Tensor        # [32, C]: the y term of a folded adjust conv (W_adj), else None
    fold: int


def unpack_mlp(pm) -> MlpWeights:
    pl = pm.plan.tolist()
    ks1, nc, hc, n2 = pl[0], pl[2], pl[3], pl[4]
    pieces = pl[8:8 + pl[7]]
    widths = pl[14:14 + nc]
    fold = pl[23]
    c = pm.C
    dev = pm.w1.device
    w1 = torch.zeros(nc * hc, ks1 * 64, dtype=F64, device=dev)
    w2 = torch.zeros(n2, nc * hc, dtype=F64, device=dev)
    wy = torch.zeros(n2, ks1 * 64, dtype=F64, device=dev) if fold == 2 else None
    o1 = o2 = 0
    for j, wj in enumerate(widths):
        for s in range(ks1):
            w1[j * hc:j * hc + wj, 64 * s:64 * s + 64] = unswizzle_slab(pm.w1[o1:o1 + wj * 128], wj)
            o1 += wj * 128
        if fold == 2 and j == 0:                  # the y slabs of alpha W_a lead chunk 0, (K slab, N piece) order
            for s in range(ks1):
                d = 0
                for rows in pieces:
                    wy[d:d + rows, 64 * s:64 * s + 64] = unswizzle_slab(pm.w2[o2:o2 + rows * 128], rows)
                    o2 += rows * 128
                    d += rows
        for s in range((wj + 63) // 64):
            valid = min(64, wj - 64 * s)
            d = 0
            for rows in pieces:
                w2[d:d + rows, j * hc + 64 * s:j * hc + 64 * s + valid] = unswizzle_slab(pm.w2[o2:o2 + rows * 128], rows)[:, :valid]
                o2 += rows * 128
                d += rows
    assert o1 == pm.w1.numel() and o2 == pm.w2.numel(), "packed MLP image does not match its plan"
    wadj = None
    if fold == 1:
        wadj = torch.cat([unswizzle_slab(pm.wadj[s * 32 * 128:(s + 1) * 32 * 128], 32) for s in range(ks1)], 1)[:, :c]
    return MlpWeights(w1[:, :c], w2, wy[:, :c] if wy is not None else None, wadj, fold)


# ------------------------------------------------------------------------------------------------ building blocks
def ln_stats(stats: torch.Tensor, slots: int, c: int, eps: float, noise: bool = False):
    """(mean, rstd) [M, 1] from the first `slots` (sum, sumsq) slots of each row, the kernels' one-pass formula.
    noise=True: in fp32 as the kernels do it."""
    if noise:
        s1, s2 = stats[:, 0, 0].float(), stats[:, 0, 1].float()
        for k in range(1, slots):
            s1, s2 = s1 + stats[:, k, 0].float(), s2 + stats[:, k, 1].float()
        inv_c = torch.tensor(1.0 / c, dtype=torch.float32)
        mean = s1 * inv_c
        rstd = torch.rsqrt(torch.clamp_min(s2 * inv_c - mean * mean, 0.0) + eps)
        return mean[:, None], rstd[:, None]
    s = stats[:, :slots].to(F64).sum(1)
    mean = s[:, 0] / c
    var = torch.clamp_min(s[:, 1] / c - mean * mean, 0.0)
    return mean[:, None], (1.0 / torch.sqrt(var + eps))[:, None]


def _folded_ln(acc, mean, rstd, colsum, bias):
    """rstd * (x W^T - mean * colsum) + b: the epilogue of every LayerNorm-folded kernel."""
    return rstd * acc - (mean * rstd) * colsum + bias


def gelu(x: torch.Tensor, kind: str = "erf") -> torch.Tensor:
    if kind == "erf":
        return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))
    return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x ** 3)))


def gelu2_swin_mlp(x: torch.Tensor) -> torch.Tensor:
    """2 GELU(x) as csrc/swin_mlp.cu evaluates it (gelu2_pair: erfc from 2^(a q(a)), |error| <= 8.6e-5 after the 0.5)."""
    a = x.abs()
    q = (-0.027645503 * a - 0.48822206) * a - 1.1409364
    return a * (1.0 - torch.exp2(q * a)) + x


def window_attention(q, k, v, table, B, H, W, ws, shift, scale, *, mask=None, rpi=None, noise=False):
    """q, k, v: [B*H*W, heads, d] in token order (d may include zero head padding) -> normalised O [B*H*W, heads, d].
    Logits q k^T * scale + table[rpi] + mask (-100 between regions, the reference's mask); mask / rpi may be given to
    state a defect.  noise=True: the kernels' softmax -- maximum over all keys (masked ones included), masked keys zeroed,
    P rounded to bf16 before P V, the row sum taken from the unrounded P."""
    M, nh, d = q.shape
    N, L = ws * ws, H * W
    dev, dt = q.device, q.dtype
    src = O.window_source_index(H, W, ws, shift).to(dev)
    nW = src.shape[0]

    def win(t):
        return t.reshape(B, L, nh, d)[:, src.reshape(-1)].view(B * nW, N, nh, d).permute(0, 2, 1, 3)

    s = (win(q) @ win(k).transpose(-2, -1)) * scale
    if rpi is None:
        rpi = O.relative_position_index(ws)
    s = s + table.to(dt)[rpi.to(dev).reshape(-1)].view(N, N, nh).permute(2, 0, 1).unsqueeze(0)
    if shift or mask is not None:
        if mask is None:
            mask = O.attention_mask(H, W, ws, shift)
        mask = mask.to(dev, dt)
        s = s.view(B, nW, nh, N, N)
        if noise:
            mx = s.amax(-1, keepdim=True)
            e = torch.exp(s - mx) * (mask[None, :, None] == 0)
        else:
            s = s + mask[None, :, None]
        s = s.view(B * nW, nh, N, N)
        if noise:
            e = e.view(B * nW, nh, N, N)
    if not noise:
        p = torch.softmax(s, -1)
        o = p @ win(v)
    else:
        if not (shift or mask is not None):
            e = torch.exp(s - s.amax(-1, keepdim=True))
        o = (bf16(e) @ win(v)) / e.sum(-1, keepdim=True)
    o = o.permute(0, 2, 1, 3).reshape(B, nW * N, nh, d)
    out = torch.empty(B, L, nh, d, dtype=dt, device=dev)
    out[:, src.reshape(-1)] = o
    return out.view(M, nh, d)


# ------------------------------------------------------------------------------------------------ kernels
def swin_attn(x, stats, slots, pa, table, B, H, W, shift, fuse, *, ws=8, scale=None, mask=None, rpi=None, noise=False):
    """adsr_swin_attn_bf16.  x: bf16 [M, >= C]; stats fp32 [M, S, 2].  Returns (att, y): att = the normalised attention
    rows [M, heads, hdp] before their bf16 rounding (stored as such without fuse, the proj MMA's A operand with it);
    y = x + proj(bf16(att)) + b before its bf16 rounding (None unless fuse)."""
    dt = torch.float32 if noise else F64
    c, nh, hd, hdp = pa.C, pa.heads, pa.hd, pa.hdp
    wts = unpack_attn(pa)
    xb = x[:, :c].to(dt)
    mean, rstd = ln_stats(stats, slots, c, pa.ln_eps, noise)
    acc = torch.einsum("mc,hnc->mhn", xb, wts.wqkv.to(dt))
    qkv = bf16(_folded_ln(acc, mean[:, :, None].to(dt), rstd[:, :, None].to(dt), wts.colsum.to(dt), wts.bias.to(dt)))
    q, k, v = qkv[..., :hdp], qkv[..., hdp:2 * hdp], qkv[..., 2 * hdp:]
    att = window_attention(q, k, v, table, B, H, W, ws, shift, hd ** -0.5 if scale is None else scale, mask=mask, rpi=rpi,
                           noise=noise)
    if not fuse:
        return att, None
    y = xb + bf16(att).reshape(-1, nh * hdp) @ wts.wproj.to(dt).reshape(c, nh * hdp).t() + wts.bias_p.to(dt)
    return att, y


def swin_mlp(y, stats, slots, pm, *, res=None, slope=0.2, gelu_kind="erf", noise=False):
    """adsr_swin_mlp_bf16 (z = y + fc2(GELU(fc1(LN(y))))), _adjust_bf16 (LReLU_slope(W_adj z + b), 32 columns) and
    _conv_res_bf16 (res + alpha (W_a z + b_a), conv_out columns), chosen by the plan's fold; the output before its bf16
    rounding."""
    dt = torch.float32 if noise else F64
    c = pm.C
    wts = unpack_mlp(pm)
    yb = y[:, :c].to(dt)
    mean, rstd = ln_stats(stats, slots, c, pm.ln_eps, noise)
    h = _folded_ln(yb @ wts.w1.to(dt).t(), mean.to(dt), rstd.to(dt), pm.colsum1.to(dt), pm.bias1.to(dt))
    g = bf16(gelu2_swin_mlp(h) if noise else 2.0 * gelu(h, gelu_kind))      # the 0.5 of GELU lives in the packed fc2
    f2 = g @ wts.w2.to(dt).t()
    if wts.fold == 0:
        return yb + f2[:, :c] + pm.bias2.to(dt)[:c]
    if wts.fold == 1:
        a = yb @ wts.wadj.to(dt).t() + f2 + pm.bias_adj.to(dt)
        return torch.where(a > 0, a, a * slope)
    co = pm.conv_out
    return res[:, :co].to(dt) + (yb @ wts.wy.to(dt).t() + f2 + pm.bias2.to(dt))[:, :co]


def gemm(a, k, pw, *, act="none", slope=0.0, alpha=1.0, res=None, stats=None, slots=0, gelu_kind="erf", noise=False):
    """tc_gemm: alpha * act(a[:, :k] W^T + b) (+ res[:, :N]); with pw.colsum (pack_ln_gemm_weight) LayerNorm(a) is folded
    in from the (sum, sumsq) slots.  Before the bf16 rounding of the output."""
    dt = torch.float32 if noise else F64
    n = pw.N
    w = unpack_tiles(pw)[:n, :k].to(dt)
    v = a[:, :k].to(dt) @ w.t()
    bias = pw.bias.to(dt)[:n]
    if pw.colsum is not None:
        mean, rstd = ln_stats(stats, slots, k, pw.ln_eps, noise)
        v = _folded_ln(v, mean.to(dt), rstd.to(dt), pw.colsum.to(dt)[:n], bias)
    else:
        v = v + bias
    if act == "gelu":
        v = gelu(v, gelu_kind)
    elif act == "lrelu":
        v = torch.where(v > 0, v, v * slope)
    elif act == "relu":
        v = torch.clamp_min(v, 0.0)
    v = v * alpha
    if res is not None:
        v = v + res[:, :n].to(dt)
    return v


# ------------------------------------------------------------------------------------------------ convolutions (DRCT, DRN)
def unpack_conv(pw, compact: bool = False) -> torch.Tensor:
    """Inverse of pack.pack_conv3x3_weight -> fp64 [Cout, Cin, 3, 3].  The tiled implicit-GEMM image has K = tap * round64(Cin) + c;
    the `compact` halo twin (csrc/conv_halo.cu) K = tap * round16(Cin) + c in one N tile of round16(Cout) rows."""
    cout, cin = pw.N, pw.K
    src = pw.compact if compact else pw
    step = (cin + 15) // 16 * 16 if compact else (cin + 63) // 64 * 64
    w = unpack_tiles(src)[:cout, :9 * step].reshape(cout, 9, step)[:, :, :cin]
    return w.permute(0, 2, 1).reshape(cout, cin, 3, 3)


def conv_input(x: torch.Tensor, B: int, H: int, W: int, cin: int, dt=F64) -> torch.Tensor:
    """NHWC rows [B*H*W, >= cin] -> NCHW."""
    return x[:, :cin].to(dt).reshape(B, H, W, cin).permute(0, 3, 1, 2)


def rows_of(t: torch.Tensor) -> torch.Tensor:
    """NCHW -> NHWC rows [B*H*W, C]."""
    return t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])


def act_fn(v: torch.Tensor, act: str, slope: float) -> torch.Tensor:
    if act == "relu":
        return torch.clamp_min(v, 0.0)
    if act == "lrelu":
        return torch.where(v > 0, v, v * slope)
    return v


def conv_pre(xin: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, stride: int = 1, noise: bool = False) -> torch.Tensor:
    """conv + bias, zero padding 1, NCHW.  noise=True: fp32, accumulated tap by tap (tap-major, then channel) like the kernels."""
    if not noise:
        return torch.nn.functional.conv2d(xin.to(F64), w.to(F64), bias.to(F64), stride=stride, padding=1)
    xp = torch.nn.functional.pad(xin.float(), (1, 1, 1, 1))
    B, _, H, W = xin.shape
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    acc = torch.zeros(B, w.shape[0], Ho, Wo)
    for ky in range(3):
        for kx in range(3):
            tap = xp[:, :, ky:ky + stride * (Ho - 1) + 1:stride, kx:kx + stride * (Wo - 1) + 1:stride]
            acc = acc + torch.einsum("bchw,oc->bohw", tap, w[:, :, ky, kx].float())
    return acc + bias.float()[None, :, None, None]


def conv_epilogue(pre, *, act="none", slope=0.0, alpha=1.0, res=None, ps=False) -> torch.Tensor:
    """alpha * act(pre) (+ res rows) -> output rows; `ps`: PixelShuffle(2) rows [B*2Ho*2Wo, N/4].  The manual epilogue
    (tc_gemm_manual.cu) rounds alpha * act(.) to bf16 before it adds the residual, the TMA epilogue (tc_gemm.cu) adds it in fp32:
    `compare(..., rounded_branch=True)` charges the first rounding."""
    v = act_fn(pre, act, slope) * alpha
    if ps:
        return rows_of(torch.nn.functional.pixel_shuffle(v, 2))
    v = rows_of(v)
    if res is not None:
        v = v + res[:, :v.shape[1]].to(v.dtype)
    return v


def conv3x3(x, B, H, W, cin, pw, *, stride=1, act="none", slope=0.0, alpha=1.0, res=None, ps=False, compact=False,
            noise=False) -> torch.Tensor:
    """adsr_conv3x3_igemm_bf16 / adsr_conv3x3_halo_bf16 from the packed image: alpha * act(conv(x) + b) (+ res), fp64 (noise:
    fp32 tap-major accumulation), output rows before their bf16 rounding."""
    w = unpack_conv(pw, compact).to(x.device)
    bias = (pw.compact if compact else pw).bias[:pw.N].to(x.device)
    pre = conv_pre(conv_input(x, B, H, W, cin, torch.float32 if noise else F64), w, bias, stride, noise)
    return conv_epilogue(pre, act=act, slope=slope, alpha=alpha, res=res, ps=ps)


def conv3x3_small(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """adsr_conv3x3_small (DRN head): fp32 NCHW input and weights -> rows [B*H*W, C] before the bf16 rounding."""
    return rows_of(conv_pre(x, w, b))


def channel_mean(t: torch.Tensor, B: int, HW: int, C: int) -> torch.Tensor:
    """AdaptiveAvgPool2d(1) of NHWC rows [B*HW, >= C] -> fp64 [B, C]."""
    return t[:, :C].to(F64).reshape(B, HW, C).mean(1)


def ca_scale(mean: torch.Tensor, w1, b1, w2, b2) -> torch.Tensor:
    """CALayer's squeeze-excite: sigmoid(W2 relu(W1 mean + b1) + b2), fp64 [B, C]."""
    h = torch.clamp_min(mean.to(F64) @ w1.to(F64).t() + b1.to(F64), 0.0)
    return torch.sigmoid(h @ w2.to(F64).t() + b2.to(F64))


def channel_mean_parts(part: torch.Tensor, B: int, parts: int, C: int, HW: int, mlp=None) -> torch.Tensor:
    """adsr_channel_mean_parts: [B*parts, >= C] fp32 partial sums -> the means, or with mlp = (w1, b1, w2, b2) the CA scales."""
    mean = part[:, :C].to(F64).reshape(B, parts, C).sum(1) / HW
    return mean if mlp is None else ca_scale(mean, *mlp)


def rcab_ca_scale(t2: torch.Tensor, x: torch.Tensor, scale: torch.Tensor, B: int, HW: int, C: int) -> torch.Tensor:
    """adsr_rcab_ca_scale: x + t2 * s per image, rows before the bf16 rounding."""
    t = t2[:, :C].to(F64).reshape(B, HW, C)
    return (x[:, :C].to(F64).reshape(B, HW, C) + t * scale.to(F64)[:, None, :]).reshape(B * HW, C)


def rcab(x, B, H, W, c1, c2, mlp, *, noise=False, pool_hw=None, scale_fn=None):
    """One RCAB of DRN: t1 = bf16(ReLU(c1 x)), t2 = bf16(c2 t1), s = CA(mean(t2)), x + t2 * s before the bf16 rounding.
    The pooled mean is taken from t2 before its rounding (the halo epilogue's partial sums); the fallback pools the bf16 t2,
    the same to ~ulp / sqrt(HW).  pool_hw / scale_fn state CA defects: the mean's divisor and the map from means to scales."""
    C = c1.N
    t1 = bf16(conv3x3(x, B, H, W, C, c1, act="relu", noise=noise))
    t2p = conv3x3(t1, B, H, W, C, c2, noise=noise)
    t2 = bf16(t2p)
    mean = t2p.to(F64).reshape(B, H * W, C).sum(1) / (H * W if pool_hw is None else pool_hw)
    s = ca_scale(mean, *mlp) if scale_fn is None else scale_fn(mean)
    if noise:
        s = s.float().double()
    return rcab_ca_scale(t2, x, s, B, H * W, C)


# ------------------------------------------------------------------------------------------------ comparator
def ulp_bf16(t: torch.Tensor) -> torch.Tensor:
    """Spacing of bf16 numbers at |t| (8 significant bits); 0 at 0."""
    t = t.to(F64)
    _, e = torch.frexp(t)
    return torch.where(t == 0, torch.zeros_like(t), torch.ldexp(torch.ones_like(t), e - 8))


@dataclass
class Verdict:
    max_units: float          # max over elements of (|got - ref| - a ulp_bf16(ref)) / rms(branch)
    rms_units: float          # sqrt(max(mean (got - ref)^2 - mean ulp_bf16(ref)^2 / 12, 0)) / rms(branch)
    b: float
    rms_b: float

    @property
    def ok(self) -> bool:
        return self.max_units <= self.b and self.rms_units <= self.rms_b

    def __str__(self) -> str:
        return (f"max {self.max_units:.4g} (limit {self.b:.3g}) rms {self.rms_units:.4g} (limit {self.rms_b:.3g}) "
                f"in units of rms(branch)")


def compare(got, ref, shortcut=None, *, b, rms_b, a=1.0, rounded_branch=False) -> Verdict:
    """Per element |got - ref| <= a ulp_bf16(ref) + b rms(branch), branch = ref - shortcut (the whole output without a
    shortcut), and the RMS error net of the output rounding's mean square ulp^2 / 12 <= rms_b rms(branch).  `ref` is the
    output before its bf16 rounding; `got` what the kernel stored.  rounded_branch: the kernel rounded the branch to bf16
    before it added the shortcut, charged like the output rounding (half an ulp of the branch, mean square ulp^2 / 12)."""
    ref = ref.to(F64)
    err = got.to(F64) - ref
    branch = ref if shortcut is None else ref - shortcut.to(F64)
    scale = float(branch.square().mean().sqrt().clamp_min(1e-30))
    ulp = ulp_bf16(ref)
    ulp_b = ulp_bf16(branch) if rounded_branch else torch.zeros_like(ulp)
    mx = float((err.abs() - a * ulp - 0.5 * ulp_b).max()) / scale
    ms = float(err.square().mean() - ulp.square().mean() / 12.0 - ulp_b.square().mean() / 12.0)
    return Verdict(mx, math.sqrt(max(ms, 0.0)) / scale, b, rms_b)


def stats_bound_check(st: torch.Tensor, out_bf16: torch.Tensor, slack: float = 4.0):
    """(sum, sumsq) [M, 2] the epilogue summed from its fp32 values v, against the stored bf16 rows o = round(v): |v - o| is at
    most half an ulp, so |sum v - sum o| <= sum ulp / 2 and |sum v^2 - sum o^2| <= sum (|o| ulp + ulp^2 / 4), plus fp32
    summation error.  Returns the largest excess over that bound in units of the bound (<= 1 passes)."""
    o = out_bf16.to(F64)
    u = ulp_bf16(o)
    n = o.shape[1]
    eps32 = 2.0 ** -24
    s1, s2 = o.sum(1), o.square().sum(1)
    b1 = 0.5 * u.sum(1) + slack * n * eps32 * o.abs().sum(1)
    b2 = (o.abs() * u + 0.25 * u * u).sum(1) + slack * n * eps32 * s2
    r1 = ((st[:, 0].to(F64) - s1).abs() / b1).max()
    r2 = ((st[:, 1].to(F64) - s2).abs() / b2).max()
    return float(max(r1, r2))


# ------------------------------------------------------------------------------------------------ seeded cases
# Built on the host from a seeded generator, so the GPU tests and the host tests (mutation table, kernel-noise check) see
# the same bytes.  `shortcut_scale` multiplies the bf16 shortcut by a power of two (exact); `mean_std` gives every row a
# mean of that many standard deviations; `qk_gain` sharpens the logits; `bias_range` draws the bias table from
# U(-range, range); `masked_max` raises the bias of every offset that crosses a shift region boundary in the last
# window row / column by 10, so that rows of the wrap windows take their largest logit from a masked key.
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _rows(g, M, C, mean_std, base_std, base_mean):
    if mean_std is None:
        return (torch.randn(M, C, generator=g) * base_std + base_mean).to(torch.bfloat16)
    sign = torch.where(torch.rand(M, 1, generator=g) < 0.5, -1.0, 1.0)
    return (torch.randn(M, C, generator=g) + sign * mean_std * (1.0 + 0.25 * torch.rand(M, 1, generator=g))).to(torch.bfloat16)


def row_stats(t: torch.Tensor, slots: int, split: int = 2) -> torch.Tensor:
    """fp32 [M, slots, 2]: the row's (sum, sumsq) in fp64 over `split` column ranges, rounded to fp32 (what a producing
    epilogue leaves behind); the remaining slots hold 1e9 and must be ignored."""
    tf = t.to(F64)
    st = torch.full((t.shape[0], slots, 2), 1e9, dtype=torch.float32)
    edges = [t.shape[1] * i // split for i in range(split + 1)]
    for i in range(split):
        p = tf[:, edges[i]:edges[i + 1]]
        st[:, i, 0], st[:, i, 1] = p.sum(1).float(), p.square().sum(1).float()
    return st


def bias_table(g, ws, heads, bias_range=None, masked_max=False, shift=0):
    assert shift or not masked_max
    nt = (2 * ws - 1) ** 2
    t = (torch.rand(nt, heads, generator=g) * 2 - 1) * bias_range if bias_range else torch.randn(nt, heads, generator=g) * 0.5
    if masked_max:
        d = torch.arange(nt)
        dy, dx = d // (2 * ws - 1) - (ws - 1), d % (2 * ws - 1) - (ws - 1)
        h = max(shift, ws - shift)                  # an offset this long crosses the region boundary of a wrap window
        t[(dy.abs() >= h) | (dx.abs() >= h)] += 10.0
    return t


def swin_attn_case(B, H, W, C, heads, shift, seed, *, shortcut_scale=1.0, mean_std=None, qk_gain=1.0, bias_range=None,
                   masked_max=False):
    from importlib import import_module
    pack = import_module("anomaly-detection-super-resolution_b200.pack")
    g = _gen(seed)
    M = B * H * W
    x = _rows(g, M, C, mean_std, 1.2, 0.2)
    if shortcut_scale != 1.0:
        x = (x.float() * shortcut_scale).to(torch.bfloat16)
    gamma = 1.0 + 0.2 * torch.randn(C, generator=g)
    beta = 0.1 * torch.randn(C, generator=g)
    qkv_w = torch.randn(3 * C, C, generator=g) * 0.08
    qkv_w[:2 * C] *= qk_gain
    qkv_b = torch.randn(3 * C, generator=g) * 0.2
    proj_w = torch.randn(C, C, generator=g) * 0.08
    proj_b = torch.randn(C, generator=g) * 0.2
    table = bias_table(g, 8, heads, bias_range, masked_max, shift)
    pa = pack.pack_swin_attn(qkv_w, qkv_b, gamma, beta, 1e-5, proj_w, proj_b, heads)
    return dict(x=x, stats=row_stats(x, 3), table=table, pa=pa, B=B, H=H, W=W, shift=shift,
                raw=dict(qkv_w=qkv_w, gamma=gamma, beta=beta, qkv_b=qkv_b, proj_w=proj_w, proj_b=proj_b))


def attention_case(B, H, W, ws, shift, heads, hd, seed, *, qk_scale=1.0, bias_range=None, masked_max=False):
    """Standalone window attention: bf16 q | k | v in the head-padded layout [M, 3, heads, hdp]."""
    g = _gen(seed)
    M = B * H * W
    hdp = (hd + 15) // 16 * 16
    qkv = torch.zeros(M, 3, heads, hdp, dtype=torch.bfloat16)
    for i in range(3):
        qkv[:, i, :, :hd] = (torch.randn(M, heads, hd, generator=g) * (qk_scale if i < 2 else 1.0)).to(torch.bfloat16)
    table = bias_table(g, ws, heads, bias_range, masked_max, shift)
    return dict(qkv=qkv.view(M, 3 * heads * hdp), table=table, B=B, H=H, W=W, ws=ws, shift=shift, heads=heads, hd=hd, hdp=hdp)


def attention_ref(case, **kw):
    qkv = case["qkv"].to(F64).view(-1, 3, case["heads"], case["hdp"])
    return window_attention(qkv[:, 0], qkv[:, 1], qkv[:, 2], case["table"], case["B"], case["H"], case["W"], case["ws"],
                            case["shift"], kw.pop("scale", case["hd"] ** -0.5), **kw)


def mlp_case(M, C, H, seed, *, kind="plain", Co=0, shortcut_scale=1.0, mean_std=None):
    """kind: plain (z = y + MLP), adjust (32 folded adjust columns), conv_res (alpha W_a z + residual, Co columns)."""
    from importlib import import_module
    pack = import_module("anomaly-detection-super-resolution_b200.pack")
    g = _gen(seed)
    y = _rows(g, M, C, mean_std, 1.5, 0.3)
    if shortcut_scale != 1.0:
        y = (y.float() * shortcut_scale).to(torch.bfloat16)
    w1, b1 = torch.randn(H, C, generator=g) * 0.08, torch.randn(H, generator=g) * 0.2
    w2, b2 = torch.randn(C, H, generator=g) * 0.08, torch.randn(C, generator=g) * 0.2
    gamma, beta = 1.0 + 0.2 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    res = None
    raw = dict(w1=w1, b1=b1, w2=w2, b2=b2, gamma=gamma, beta=beta)
    if kind == "plain":
        pm = pack.pack_swin_mlp(w1, b1, gamma, beta, 1e-5, w2, b2)
    elif kind == "adjust":
        wa, ba = torch.randn(32, C, 1, 1, generator=g) * 0.1, torch.randn(32, generator=g) * 0.2
        pm = pack.pack_swin_mlp(w1, b1, gamma, beta, 1e-5, w2, b2, wa, ba)
        raw.update(wa=wa, ba=ba)
    else:
        wa, ba = torch.randn(Co, C, 1, 1, generator=g) * 0.1, torch.randn(Co, generator=g) * 0.2
        pm = pack.pack_swin_mlp_conv_res(w1, b1, gamma, beta, 1e-5, w2, b2, wa, ba, 0.2)
        res = (torch.randn(M, Co, generator=g) * 2.0 * shortcut_scale).to(torch.bfloat16)
        raw.update(wa=wa, ba=ba)
    return dict(y=y, stats=row_stats(y, 3), pm=pm, res=res, kind=kind, raw=raw)


def ln_gemm_case(M, K, N, seed, *, rows=False, mean_std=None):
    from importlib import import_module
    pack = import_module("anomaly-detection-super-resolution_b200.pack")
    g = _gen(seed)
    if mean_std is None:
        a = (torch.randn(M, K, generator=g) * 2.5 + 1.5 * torch.randn(M, 1, generator=g)).to(torch.bfloat16)
    else:
        a = _rows(g, M, K, mean_std, 1.0, 0.0)
    w, b = torch.randn(N, K, generator=g) * 0.1, torch.randn(N, generator=g)
    gm, bt = torch.rand(K, generator=g) + 0.5, torch.randn(K, generator=g) * 0.3
    pw = pack.pack_ln_gemm_weight(w, b, gm, bt, 1e-5, rows_kernel=rows)
    st = row_stats(a, 4, split=1)
    st[:, 1] = st[:, 0] * 0.25                     # statistics split over two slots
    st[:, 0] = st[:, 0] * 0.75
    st[:, 2:] = 1e9
    return dict(a=a, stats=st, pw=pw, raw=dict(w=w, b=b, gamma=gm, beta=bt))


def conv_case(B, H, W, Cin, Cout, seed, *, res=False, ld=None, fill=0.0):
    """bf16 NHWC rows [B*H*W, ld] (columns >= Cin hold `fill`, the 8-channel K tail zeros), weights ~ N(0, 0.05^2), bias ~ N(0, 1),
    and for `res` bf16 residual rows; Ho, Wo at stride 1 (the caller sizes a stride-2 residual itself)."""
    from importlib import import_module
    pack = import_module("anomaly-detection-super-resolution_b200.pack")
    g = _gen(seed)
    ld = (Cin + 15) // 16 * 16 if ld is None else ld
    x = torch.full((B * H * W, ld), fill, dtype=torch.bfloat16)
    x[:, :Cin] = torch.randn(B * H * W, Cin, generator=g).to(torch.bfloat16)
    x[:, Cin:(Cin + 7) // 8 * 8] = 0
    w = torch.randn(Cout, Cin, 3, 3, generator=g) * 0.05
    bias = torch.randn(Cout, generator=g)
    r = (torch.randn(B * H * W, (Cout + 15) // 16 * 16, generator=g)).to(torch.bfloat16) if res else None
    return dict(x=x, w=w, bias=bias, pw=pack.pack_conv3x3_weight(w, bias), res=r)


def rcab_case(B, H, W, C, seed):
    """One RCAB's inputs: bf16 x rows [B*H*W, round16(C)], c1 / c2 packed with DRN's init scale, CALayer weights (C // 16 hidden)."""
    from importlib import import_module
    pack = import_module("anomaly-detection-super-resolution_b200.pack")
    g = _gen(seed)
    ld = (C + 15) // 16 * 16
    x = torch.zeros(B * H * W, ld, dtype=torch.bfloat16)
    off = torch.randn(B, 1, C, generator=g) * 1.5                 # per-image channel offsets: images differ in their CA scales
    x[:, :C] = (torch.randn(B, H * W, C, generator=g) * 2.0 + off).reshape(-1, C).to(torch.bfloat16)
    s = (9 * C) ** -0.5
    c1 = pack.pack_conv3x3_weight(torch.randn(C, C, 3, 3, generator=g) * s, torch.randn(C, generator=g) * 0.2)
    c2 = pack.pack_conv3x3_weight(torch.randn(C, C, 3, 3, generator=g) * s, torch.randn(C, generator=g) * 0.5)
    cr = C // 16
    mlp = (torch.randn(cr, C, generator=g), torch.randn(cr, generator=g) * 0.1,
           torch.randn(C, cr, generator=g), torch.randn(C, generator=g) * 0.1)
    return dict(x=x, c1=c1, c2=c2, mlp=mlp, B=B, H=H, W=W, C=C)


# ------------------------------------------------------------------------------------------------ tolerances
# (b, rms_b) of `compare` per kernel, in units of rms(branch); a = 1 ulp everywhere.  Bounded from below by the largest
# error measured on a B200 (1000 W power limit) over the seeded GPU cases and by the simulated kernel noise (`noise=True`),
# from above by the smallest defect of the mutation table in tests/test_hotpath_oracle_host.py:
#   swin_attn  measured max 0.032 / rms 0.0031 (attention only at mean/std 100); softmax scale +1 % gives rms 0.0070
#   attention  measured max 0.017 / rms 0.0017;                                   softmax scale +1 % gives rms 0.0098
#   swin_mlp   measured max 0.0085 / rms 0.0016 (mean/std 100);                  colsum from fp32 weights gives 0.079
#   gemm       measured max 0.0016 / rms 0.00032;                                 LayerNorm eps 1e-3 gives > 0.01
#   conv       measured within 1 ulp, rms <= 0.00094 (double-rounded residual);   ReLU for LeakyReLU(0.01) gives 0.067 / 0.011
#   rcab       measured max 0.0137 / rms 0.00029;                                 pad columns pooled gives 0.046 / 0.0045 (64 px)
TOL = {
    "swin_attn": (0.045, 0.005),      # q | k | v and O are bf16 operands: their rounding flips are the noise floor
    "attention": (0.03, 0.004),
    "swin_mlp": (0.012, 0.003),       # one bf16 intermediate: the GELU activations, from a GELU approximation good to 8.6e-5
    "gemm": (0.003, 0.0008),          # fp32 accumulation only
    "conv": (0.003, 0.0008),          # exact bf16 inputs and weights: fp32 accumulation order only
    "rcab": (0.02, 0.003),            # bf16 t1 and t2 between the stages: a rounding flip of t2 shows as ulp(t2) * s
}
# Logits about 10 apart: where two keys nearly tie, O moves by p (1 - p) |v1 - v2| per unit of logit error, so the fp32
# logits' rounding shows in single elements (simulated noise 0.035, B200 0.074 on C = 244); the RMS limit is unchanged.
PEAKED_B = 0.15
