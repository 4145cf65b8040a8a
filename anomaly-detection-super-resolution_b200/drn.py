"""B200-native DRN (dual regression network, "DRN-L"): same constructor, state_dict and forward contract as the
reference's `src.drn.DRN` (/root/reference/src/drn.py:160-270), executed by the sm_100a kernels.

The module tree only holds parameters under the reference's names (sub_mean, add_mean, head,
down.{p}.dual_module.{0.0,1}, up_blocks.{i}.{j}.body.{0,2,3.conv_du.{0,2}}, up_blocks.{i}.{n}.0, up_blocks.{i}.{n+1},
tail.{i}); `forward` returns the reference's list [sr_x1, sr_x2, ..., sr_xS] (low -> high resolution).

Data flow (NHWC bf16 rows; every 3x3 conv is the tcgen05 implicit GEMM):
  bicubic xS + sub_mean (one kernel, fp32) -> head conv -> stride-2 DownBlocks (skip copies are written straight
  into the channel slice of the later torch.cat buffer) -> per level: n_blocks x RCAB [conv+ReLU, conv, channel
  mean, channel-attention scale + residual] -> conv + fused PixelShuffle(2) -> 1x1 conv into the cat buffer ->
  tail conv (+ add_mean folded into its weights) -> SR image (fp32 NCHW, last level optionally uint8).
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import torch
import torch.nn as nn

from . import ops, pack
from .pack import round_up


class _MeanShift(nn.Conv2d):
    def __init__(self, rgb_range, mean, std, sign=-1, n_channels=3):
        super().__init__(n_channels, n_channels, kernel_size=1)
        std_t = torch.Tensor(std)
        self.weight.data = torch.eye(n_channels).view(n_channels, n_channels, 1, 1) / std_t.view(n_channels, 1, 1, 1)
        self.bias.data = sign * rgb_range * torch.Tensor(mean) / std_t
        self.requires_grad = False          # (an attribute, exactly like the reference: it does not freeze anything)


class _DownBlock(nn.Module):
    def __init__(self, negval, n_feat, cin, cout):
        super().__init__()
        self.dual_module = nn.Sequential(
            nn.Sequential(nn.Conv2d(cin, n_feat, 3, stride=2, padding=1, bias=False), nn.LeakyReLU(negval, inplace=True)),
            nn.Conv2d(n_feat, cout, 3, stride=1, padding=1, bias=False))


class _CALayer(nn.Module):
    def __init__(self, channel, reduction=16):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.conv_du = nn.Sequential(nn.Conv2d(channel, channel // reduction, 1), nn.ReLU(inplace=True),
                                     nn.Conv2d(channel // reduction, channel, 1), nn.Sigmoid())


class _RCAB(nn.Module):
    def __init__(self, n_feat):
        super().__init__()
        self.body = nn.Sequential(nn.Conv2d(n_feat, n_feat, 3, padding=1), nn.ReLU(True),
                                  nn.Conv2d(n_feat, n_feat, 3, padding=1), _CALayer(n_feat))
        self.res_scale = 1                  # stored, never applied (src/drn.py:153-158)


class DRN(nn.Module):
    """Drop-in for `src.drn.DRN(opt)`: reads opt.{scale(list), n_blocks, n_feats, n_colors, rgb_range, negval}."""

    def __init__(self, opt, conv=None):
        super().__init__()
        self.opt = opt
        self.scale = list(opt.scale)
        self.phase = len(self.scale)
        nb, nf, nc = opt.n_blocks, opt.n_feats, opt.n_colors
        if nf % 4:
            # the skip copies live in channel slices [c, 2c) of the later torch.cat buffers; the tensor-core loaders need 16-byte aligned
            # slices, i.e. 2 * n_feats a multiple of 8 (DRN-L x4: n_feats = 20 is; the reference's x8 setting n_feats = 10 is not)
            raise ValueError(f"n_feats={nf} is not supported by the B200 build: channel slices must be 16-byte aligned (n_feats % 4 == 0); "
                             "the reference's scale-8 configuration (n_feats=10) needs padded slices, which are not implemented")
        self.n_blocks, self.n_feats, self.n_colors = nb, nf, nc
        self.rgb_range, self.negval = float(opt.rgb_range), float(opt.negval)
        self.upsample = nn.Upsample(scale_factor=max(self.scale), mode='bicubic', align_corners=False)
        if nc == 1:
            mean, std = (0.4440,), (1.0,)
        else:
            mean, std = (0.4488, 0.4371, 0.4040), (1.0, 1.0, 1.0)
        self.sub_mean = _MeanShift(opt.rgb_range, mean, std, n_channels=nc)
        self.add_mean = _MeanShift(opt.rgb_range, mean, std, 1, n_channels=nc)
        self.head = nn.Conv2d(nc, nf, 3, padding=1)
        ph = self.phase
        self.down = nn.ModuleList([_DownBlock(opt.negval, nf * 2 ** p, nf * 2 ** p, nf * 2 ** (p + 1)) for p in range(ph)])
        ups = []
        for idx in range(ph):
            c = nf * 2 ** ph if idx == 0 else 2 * nf * 2 ** (ph - idx)
            blocks = [_RCAB(c) for _ in range(nb)]
            upsampler = nn.Sequential(nn.Conv2d(c, 4 * c, 3, padding=1), nn.PixelShuffle(2))
            ups.append(nn.Sequential(*blocks, upsampler, nn.Conv2d(c, nf * 2 ** (ph - idx - 1), 1)))
        self.up_blocks = nn.ModuleList(ups)
        tail = [nn.Conv2d(nf * 2 ** ph, nc, 3, padding=1)]
        for p in range(ph, 0, -1):
            tail.append(nn.Conv2d(nf * 2 ** p, nc, 3, padding=1))
        self.tail = nn.ModuleList(tail)
        self._packed = None
        self._packed_key = None

    # ------------------------------------------------------------------ packing
    def _apply(self, fn, *a, **k):
        self._packed = None
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._packed = None
        return super().load_state_dict(*a, **k)

    def _pack(self) -> dict:
        key = tuple((p.data_ptr(), p._version) for p in self.parameters())
        if self._packed is not None and self._packed_key == key:
            return self._packed
        dev = self.head.weight.device
        if dev.type != "cuda":
            raise RuntimeError("DRN parameters must live on a CUDA device (no CPU fallback); call .cuda()")
        f32 = lambda t: t.detach().float().contiguous()
        # packed on the HOST from CPU copies of the parameters, uploaded with one copy per buffer (pack.to_device)
        cpu = lambda t: None if t is None else t.detach().float().cpu()
        up = lambda o: pack.to_device(o, dev)
        pconv = lambda w, b: up(pack.pack_conv3x3_weight(cpu(w), cpu(b)))
        nc = self.n_colors
        P = {"sub_w": f32(self.sub_mean.weight).view(nc, nc).contiguous(), "sub_b": f32(self.sub_mean.bias),
             "head_w": f32(self.head.weight), "head_b": f32(self.head.bias), "down": [], "levels": [], "tails": []}
        for d in self.down:
            P["down"].append((pconv(d.dual_module[0][0].weight, None), pconv(d.dual_module[1].weight, None)))
        for seq in self.up_blocks:
            mods = list(seq)
            rcabs = []
            for m in mods[:self.n_blocks]:
                ca = m.body[3].conv_du
                c, cr = ca[0].in_channels, ca[0].out_channels
                rcabs.append(dict(c1=pconv(m.body[0].weight, m.body[0].bias), c2=pconv(m.body[2].weight, m.body[2].bias),
                                  w1=f32(ca[0].weight).view(cr, c).contiguous(), b1=f32(ca[0].bias),
                                  w2=f32(ca[2].weight).view(c, cr).contiguous(), b2=f32(ca[2].bias), c=c, cr=cr))
            up_conv, conv1 = mods[self.n_blocks][0], mods[self.n_blocks + 1]
            P["levels"].append(dict(rcabs=rcabs, up=pconv(up_conv.weight, up_conv.bias),
                                    c1x1=up(pack.pack_gemm_weight(cpu(conv1.weight), cpu(conv1.bias))), c=up_conv.in_channels,
                                    cout=conv1.out_channels))
        # add_mean (a 1x1 conv) is folded into each tail conv: W' = A W, b' = A b + a   (exact)
        A, a = cpu(self.add_mean.weight).view(nc, nc), cpu(self.add_mean.bias)
        for t in self.tail:
            w = torch.einsum("oc,cikl->oikl", A, cpu(t.weight)).contiguous()
            P["tails"].append((w.to(dev), (A @ cpu(t.bias) + a).contiguous().to(dev), t.in_channels))
        P["zero_mean"] = torch.zeros(nc, dtype=torch.float32).to(dev)
        self._packed, self._packed_key = P, key
        return P

    # ------------------------------------------------------------------ forward
    def forward(self, x: torch.Tensor) -> List[torch.Tensor]:
        outs, _ = self.run(x, want_u8=False)
        return outs

    @torch.no_grad()
    def run(self, x: torch.Tensor, want_float: bool = True, want_u8: bool = False,
            out_u8: Optional[torch.Tensor] = None) -> Tuple[Optional[List[torch.Tensor]], Optional[torch.Tensor]]:
        """Returns ([sr_x1, .., sr_xS] fp32 NCHW or None, uint8 NHWC truncation of the LAST output or None)."""
        if not x.is_cuda:
            raise RuntimeError("input must be a CUDA tensor: this package has no CPU fallback")
        P = self._pack()
        x = x.contiguous().float()
        B, nc, h, w = x.shape
        if nc != self.n_colors:
            raise ValueError(f"expected {self.n_colors} input channels, got {nc}")
        ph, nf, S = self.phase, self.n_feats, max(self.scale)
        if (h * S) % (2 ** ph) or (w * S) % (2 ** ph):
            raise ValueError("input size must keep every pyramid level integral")
        dev = x.device
        bf = dict(dtype=torch.bfloat16, device=dev)
        H, W = h * S, w * S
        res = [(H >> p, W >> p) for p in range(ph + 1)]                     # level p: HR / 2^p
        rows = [B * r[0] * r[1] for r in res]

        up = torch.empty(B, nc, H, W, dtype=torch.float32, device=dev)
        ops.bicubic_affine(x, S, P["sub_w"], P["sub_b"], up)
        # cat buffers: level p < ph holds  [ up-path features | skip copy ]  = 2 * nf * 2^p channels
        cat = [torch.zeros(rows[p], round_up(2 * nf * 2 ** p, 16), **bf) for p in range(ph)]
        feat = torch.zeros(rows[0], round_up(nf, 16), **bf)
        ops.conv3x3_small(up, P["head_w"], P["head_b"], nf, feat, cat[0], nf)
        cur, cur_c = feat, nf                                                 # down path input (first nf columns)
        for p in range(ph):
            c = nf * 2 ** p
            d_a, d_b = P["down"][p]
            mid = torch.zeros(rows[p + 1], round_up(c, 16), **bf)
            ops.conv3x3(cur, B, res[p][0], res[p][1], c, d_a, mid, stride=2, act=ops.ACT_LRELU, slope=self.negval)
            if p + 1 < ph:                                                   # next skip copy: right half of cat[p+1]
                ops.conv3x3(mid, B, res[p + 1][0], res[p + 1][1], c, d_b, cat[p + 1], ocol0=2 * c, n_store=2 * c)
                cur = cat[p + 1][:, 2 * c:]                                  # view: same rows, offset base pointer
            else:
                bottom = torch.zeros(rows[ph], round_up(2 * c, 16), **bf)
                ops.conv3x3(mid, B, res[ph][0], res[ph][1], c, d_b, bottom)
                cur = bottom
        outs: List[Optional[torch.Tensor]] = []

        def tail(i, src, hh, ww, last):
            wt, bt, cin = P["tails"][i]
            o = torch.empty(B, nc, hh, ww, dtype=torch.float32, device=dev) if want_float else None
            u8 = None
            if last and want_u8:
                u8 = out_u8 if out_u8 is not None else torch.empty(B, hh, ww, nc, dtype=torch.uint8, device=dev)
            if o is not None or u8 is not None:
                ops.conv_last_quant(src, B, hh, ww, cin, wt, bt, nc, P["zero_mean"], 1.0, self.rgb_range, o, u8)
            outs.append(o)
            return u8

        tail(0, cur, res[ph][0], res[ph][1], False)
        u8 = None
        xbuf = cur
        for idx in range(ph):
            lvl = P["levels"][idx]
            p = ph - idx                                                     # resolution level of this stage
            c, hw = lvl["c"], res[p][0] * res[p][1]
            t1 = torch.empty(rows[p], round_up(c, 16), **bf)
            t2 = torch.empty(rows[p], round_up(c, 16), **bf)
            gap = torch.empty(B, c, dtype=torch.float32, device=dev)
            n_parts = ops.halo_parts(res[p][0], res[p][1])                   # >= channel_mean_slices(hw)
            parts = torch.empty(B * n_parts, round_up(c, 16), dtype=torch.float32, device=dev)
            for r in lvl["rcabs"]:
                ops.conv3x3(xbuf, B, res[p][0], res[p][1], c, r["c1"], t1, act=ops.ACT_RELU)
                # CALayer's pooled mean leaves the second conv's epilogue as per-tile partial sums when the halo kernel covers it,
                # else channel_mean writes per-slice sums in the same layout: both reduced in a fixed order
                n = n_parts
                if not ops.conv3x3(t1, B, res[p][0], res[p][1], c, r["c2"], t2, chan_part=parts):
                    n = ops.channel_mean_slices(hw)
                    ops.channel_sums(t2, B, hw, c, parts)
                ops.channel_mean_parts(parts, B, n, c, hw, gap, r["w1"], r["b1"], r["w2"], r["b2"], r["cr"])
                ops.rcab_ca_scale(t2, xbuf, xbuf, gap, r["w1"], r["b1"], r["w2"], r["b2"], B, hw, c, 0)     # gap = the scales
            shuf = torch.empty(rows[p - 1], round_up(c, 16), **bf)
            ops.conv3x3(xbuf, B, res[p][0], res[p][1], c, lvl["up"], shuf, out_mode=ops.OUT_PIXEL_SHUFFLE2)
            ops.tc_gemm(shuf, c, lvl["c1x1"], cat[p - 1], n_store=lvl["cout"])
            xbuf = cat[p - 1]
            u8 = tail(idx + 1, xbuf, res[p - 1][0], res[p - 1][1], idx == ph - 1)
        return (outs if want_float else None), u8
