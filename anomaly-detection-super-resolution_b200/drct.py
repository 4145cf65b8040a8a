"""B200-native DRCT: same constructor, state_dict and forward contract as the reference's
`src.drct.DRCT` (/root/reference/src/drct.py:716-899), executed by hand-written sm_100a kernels.

The nn.Module tree below only *holds parameters* with the reference's names and shapes
(conv_first, patch_embed.norm, layers.{i}.swin{k}.{norm1,attn.{relative_position_bias_table,
relative_position_index,qkv,proj},norm2,mlp.{fc1,fc2},attn_mask}, layers.{i}.adjust{k}, norm,
conv_after_body, conv_before_upsample.0, upsample.{0,2,..}, conv_last) so reference checkpoints load
with zero missing / unexpected keys.  `forward` never runs a torch op on activations: it packs the
weights once into tensor-core images (pack.py) and enqueues kernels through the C ABI (ops.py).

Data layout in HBM (all bf16, token-major = NHWC, row m = (b*H + y)*W + x):
  slab [M, 320]   one RDG's dense feature slab  x | x1 | x2 | x3 | x4  at columns 0/180/212/244/276
                  (torch.cat of src/drct.py:389-393 disappears: adjust_k writes its 32-wide slice)
  ln/qkv/att/y/h/z  per-block scratch rows (LayerNorm out, head-padded q|k|v, attention out,
                  post-attention residual, MLP hidden, post-MLP residual)
Evaluation semantics only (DropPath = identity, as `model.eval()`); see DESIGN.md.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import ops, pack
from .pack import PackedWeight, round_up

RGB_MEAN = (0.4488, 0.4371, 0.4040)   # src/drct.py:774


def _heads_for(dim: int, k: int, nh: int) -> int:
    """Head count of the k-th Swin block of an RDG (src/drct.py:326-367)."""
    return nh if k == 0 else nh - (dim % nh)


class _Mlp(nn.Module):
    def __init__(self, dim: int, hidden: int):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _WindowAttention(nn.Module):
    def __init__(self, dim: int, ws: int, heads: int):
        super().__init__()
        self.dim, self.window_size, self.num_heads = dim, (ws, ws), heads
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * ws - 1) * (2 * ws - 1), heads))
        n = torch.arange(ws * ws)
        y, x = n // ws, n % ws
        rpi = (y[:, None] - y[None, :] + ws - 1) * (2 * ws - 1) + (x[:, None] - x[None, :] + ws - 1)
        self.register_buffer("relative_position_index", rpi)
        self.qkv = nn.Linear(dim, dim * 3)
        self.proj = nn.Linear(dim, dim)
        nn.init.trunc_normal_(self.relative_position_bias_table, std=0.02)


def _attn_mask(h: int, w: int, ws: int, shift: int) -> torch.Tensor:
    """Buffer kept only for state_dict parity (src/drct.py:449-470); the kernels derive it in registers."""
    nwx = w // ws
    win = torch.arange((h // ws) * nwx).view(-1, 1)
    n = torch.arange(ws * ws).view(1, -1)
    ys, xs = (win // nwx) * ws + n // ws, (win % nwx) * ws + n % ws

    def r(t, length):
        return (t >= length - ws).long() + (t >= length - shift).long()

    ids = 3 * r(ys, h) + r(xs, w)
    neq = ids[:, None, :] != ids[:, :, None]
    return torch.where(neq, torch.tensor(-100.0), torch.tensor(0.0))


class _SwinBlock(nn.Module):
    def __init__(self, dim: int, res: Tuple[int, int], heads: int, ws: int, shift: int, mlp_ratio: float):
        super().__init__()
        if min(res) <= ws:                       # src/drct.py:425-428
            shift, ws = 0, min(res)
        self.dim, self.num_heads, self.window_size, self.shift_size = dim, heads, ws, shift
        self.hidden = int(dim * mlp_ratio)
        self.norm1 = nn.LayerNorm(dim)
        self.attn = _WindowAttention(dim, ws, heads)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = _Mlp(dim, self.hidden)
        self.register_buffer("attn_mask", _attn_mask(res[0], res[1], ws, shift) if shift > 0 else None)


class _RDG(nn.Module):
    def __init__(self, dim: int, res: Tuple[int, int], heads: int, ws: int, mlp_ratio: float, gc: int):
        super().__init__()
        ratios = (mlp_ratio, mlp_ratio, mlp_ratio, 1, 1)
        for k in range(5):
            d = dim + k * gc
            setattr(self, f"swin{k + 1}", _SwinBlock(d, res, _heads_for(d, k, heads), ws, (ws // 2) if k in (1, 3) else 0,
                                                     ratios[k]))
            setattr(self, f"adjust{k + 1}", nn.Conv2d(d, gc if k < 4 else dim, 1))


class _PatchNorm(nn.Module):
    def __init__(self, dim: int):
        super().__init__()
        self.norm = nn.LayerNorm(dim)


class _Block:
    """Packed weights + geometry of one Swin block and its adjust conv."""
    __slots__ = ("dim", "heads", "hd", "hdp", "shift", "ws", "hidden", "adjust_out", "n1w", "n1b", "n2w", "n2b", "table",
                 "qkv", "proj", "mlp", "mlp_res", "adjust", "last", "attn", "attn_mode")


class DRCT(nn.Module):
    """Drop-in for `src.drct.DRCT(opt)`: reads the same `opt` fields (src/drct.py:748-762)."""

    def __init__(self, opt, gc: int = 32, **kwargs):
        super().__init__()
        img_size, in_chans = opt.img_size, opt.n_colors
        embed_dim, depths, num_heads = opt.embed_dim, opt.depths, opt.num_heads
        ws, mlp_ratio, upscale = opt.window_size, opt.mlp_ratio, opt.upscale
        if getattr(opt, "upsampler", "pixelshuffle") != "pixelshuffle":
            raise ValueError("only the 'pixelshuffle' upsampler path of the reference is implemented")
        if getattr(opt, "resi_connection", "1conv") != "1conv":
            raise ValueError("only resi_connection='1conv' is implemented")
        if upscale & (upscale - 1):
            raise ValueError(f"scale {upscale} is not supported. Supported scales: 2^n")
        self.window_size, self.shift_size = ws, ws // 2
        self.img_range, self.upscale, self.upsampler = opt.img_range, upscale, "pixelshuffle"
        self.embed_dim, self.num_layers, self.mlp_ratio, self.gc = embed_dim, len(depths), mlp_ratio, gc
        self.n_colors, self.num_feat = in_chans, 64
        self.rgb_range = float(getattr(opt, "rgb_range", 255))
        self.mean = torch.Tensor(RGB_MEAN).view(1, 3, 1, 1) if in_chans == 3 else torch.zeros(1, 1, 1, 1)
        res = (img_size, img_size)

        self.conv_first = nn.Conv2d(in_chans, embed_dim, 3, 1, 1)
        self.patch_embed = _PatchNorm(embed_dim)
        self.layers = nn.ModuleList([_RDG(embed_dim, res, num_heads[i], ws, mlp_ratio, gc) for i in range(self.num_layers)])
        self.norm = nn.LayerNorm(embed_dim)
        self.conv_after_body = nn.Conv2d(embed_dim, embed_dim, 3, 1, 1)
        self.conv_before_upsample = nn.Sequential(nn.Conv2d(embed_dim, 64, 3, 1, 1), nn.LeakyReLU(inplace=True))
        ups: List[nn.Module] = []
        for _ in range(int(math.log2(upscale))):
            ups += [nn.Conv2d(64, 256, 3, 1, 1), nn.PixelShuffle(2)]
        self.upsample = nn.Sequential(*ups)
        self.conv_last = nn.Conv2d(64, in_chans, 3, 1, 1)
        self.apply(self._init_weights)

        self._packed: Optional[dict] = None
        self._packed_key = None
        self._ws_cache: Dict[tuple, dict] = {}

    @staticmethod
    def _init_weights(m):                       # src/drct.py:851-858
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=0.02)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)

    # ------------------------------------------------------------------ packing
    def _param_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def invalidate_packed(self) -> None:
        self._packed = None

    def _pack(self) -> dict:
        key = self._param_key()
        if self._packed is not None and self._packed_key == key:
            return self._packed
        dev = self.conv_first.weight.device
        if dev.type != "cuda":
            raise RuntimeError("DRCT parameters must live on a CUDA device (no CPU fallback); call .cuda()")
        f32 = lambda t: t.detach().float().contiguous()
        # tensor-core images are packed on the HOST from CPU copies of the parameters and uploaded with one copy per buffer
        # (pack.to_device): loading a model launches no device kernel
        cpu = lambda t: None if t is None else t.detach().float().cpu()
        up = lambda o: pack.to_device(o, dev)
        P: dict = {"blocks": []}
        P["mean"] = self.mean.to(dev).float().reshape(-1).contiguous()
        P["cf_w"], P["cf_b"] = f32(self.conv_first.weight), f32(self.conv_first.bias)
        P["pe_w"], P["pe_b"] = f32(self.patch_embed.norm.weight), f32(self.patch_embed.norm.bias)
        for layer in self.layers:
            blocks = []
            for k in range(5):
                sw, adj = getattr(layer, f"swin{k + 1}"), getattr(layer, f"adjust{k + 1}")
                b = _Block()
                b.dim, b.heads, b.ws, b.shift, b.hidden = sw.dim, sw.num_heads, sw.window_size, sw.shift_size, sw.hidden
                b.hd = b.dim // b.heads
                b.hdp = pack.head_pad(b.hd)
                b.adjust_out, b.last = adj.out_channels, k == 4
                b.n1w, b.n1b, b.n2w, b.n2b = f32(sw.norm1.weight), f32(sw.norm1.bias), f32(sw.norm2.weight), f32(sw.norm2.bias)
                b.table = f32(sw.attn.relative_position_bias_table)
                qkv_w, qkv_b, n1w, n1b = cpu(sw.attn.qkv.weight), cpu(sw.attn.qkv.bias), cpu(sw.norm1.weight), cpu(sw.norm1.bias)
                proj_w, proj_b = cpu(sw.attn.proj.weight), cpu(sw.attn.proj.bias)
                fc1_w, fc1_b, fc2_w, fc2_b = cpu(sw.mlp.fc1.weight), cpu(sw.mlp.fc1.bias), cpu(sw.mlp.fc2.weight), cpu(sw.mlp.fc2.bias)
                n2w, n2b, adj_w, adj_b = cpu(sw.norm2.weight), cpu(sw.norm2.bias), cpu(adj.weight), cpu(adj.bias)
                b.qkv = up(pack.pack_qkv_weight(qkv_w, qkv_b, b.heads, n1w, n1b, sw.norm1.eps))
                b.proj = up(pack.pack_proj_weight(proj_w, proj_b, b.heads))
                # fused attention half (csrc/swin_attn.cu): 2 = qkv + attention + proj + residual in one kernel,
                # 1 = qkv + attention (proj stays a row-tile GEMM), 0 = shape not covered (separate kernels)
                b.attn_mode = ops.swin_attn_mode(b.dim, b.heads, b.hdp) if b.ws == 8 else 0
                b.attn = up(pack.pack_swin_attn(qkv_w, qkv_b, n1w, n1b, sw.norm1.eps, proj_w, proj_b, b.heads)) if b.attn_mode else None
                # the 32-channel adjust convs ride in the MLP kernel's last epilogue where its tiling leaves room (z is then never
                # written); otherwise (and for adjust5) the adjust conv stays a GEMM of its own
                b.mlp = None
                if k < 4 and adj.out_channels == 32:
                    try:
                        b.mlp = up(pack.pack_swin_mlp(fc1_w, fc1_b, n2w, n2b, sw.norm2.eps, fc2_w, fc2_b, adj_w, adj_b))
                    except ValueError:
                        b.mlp = None
                if b.mlp is None:
                    b.mlp = up(pack.pack_swin_mlp(fc1_w, fc1_b, n2w, n2b, sw.norm2.eps, fc2_w, fc2_b))
                # adjust5 and the group's residual (`x5 * 0.2 + x`, src/drct.py:394-396) fold into the last block's MLP kernel the same way
                b.mlp_res = None
                if k == 4:
                    try:
                        b.mlp_res = up(pack.pack_swin_mlp_conv_res(fc1_w, fc1_b, n2w, n2b, sw.norm2.eps, fc2_w, fc2_b, adj_w, adj_b, 0.2))
                    except ValueError:
                        b.mlp_res = None
                b.adjust = up(pack.pack_gemm_weight(adj_w, adj_b, rows_kernel=(k == 4)))
                blocks.append(b)
            P["blocks"].append(blocks)
        P["norm_w"], P["norm_b"] = f32(self.norm.weight), f32(self.norm.bias)
        P["cab"] = up(pack.pack_conv3x3_weight(cpu(self.conv_after_body.weight), cpu(self.conv_after_body.bias)))
        P["cbu"] = up(pack.pack_conv3x3_weight(cpu(self.conv_before_upsample[0].weight), cpu(self.conv_before_upsample[0].bias)))
        P["ups"] = [up(pack.pack_conv3x3_weight(cpu(m.weight), cpu(m.bias))) for m in self.upsample if isinstance(m, nn.Conv2d)]
        P["cl_w"], P["cl_b"] = f32(self.conv_last.weight), f32(self.conv_last.bias)
        self._packed, self._packed_key = P, key
        return P

    def _apply(self, fn, *a, **k):              # .to()/.cuda()/.half() move parameters -> repack lazily
        self._packed = None
        self._ws_cache = {}
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._packed = None
        return super().load_state_dict(*a, **k)

    # ------------------------------------------------------------------ workspaces
    def _workspace(self, B: int, H: int, W: int, dev) -> dict:
        key = (B, H, W, str(dev))
        ws = self._ws_cache.get(key)
        if ws is not None:
            return ws
        M = B * H * W
        max_dim = self.embed_dim + 4 * self.gc
        pitch = round_up(max_dim, 64)
        blocks = self._pack()["blocks"][0]
        qkv_w = max(3 * b.heads * b.hdp for b in blocks)
        att_w = max(round_up(b.heads * b.hdp, 16) for b in blocks)
        hid_w = max(round_up(b.hidden, 16) for b in blocks)
        e16 = round_up(self.embed_dim, 16)
        bf = dict(dtype=torch.bfloat16, device=dev)
        ws = {
            "slab": torch.zeros(M, pitch, **bf), "ln": torch.zeros(M, pitch, **bf), "y": torch.zeros(M, pitch, **bf),
            "z": torch.zeros(M, pitch, **bf), "qkv": torch.zeros(M, qkv_w, **bf), "att": torch.zeros(M, att_w, **bf),
            "h": torch.zeros(M, hid_w, **bf), "x0": torch.zeros(M, e16, **bf), "body": torch.zeros(M, e16, **bf),
            "f": torch.zeros(M, 64, **bf),
            # per-row (sum, sumsq) partials for the folded LayerNorms: slab = x (2 slots) + x1..x4 (2 slots each); y = proj
            "st_slab": torch.zeros(M, 12, 2, dtype=torch.float32, device=dev),
            "st_y": torch.zeros(M, 8, 2, dtype=torch.float32, device=dev),
        }
        ups, m = [], M
        for _ in range(int(math.log2(self.upscale))):
            m *= 4
            ups.append(torch.zeros(m, 64, **bf))
        ws["ups"] = ups
        if len(self._ws_cache) > 4:
            self._ws_cache.clear()
        self._ws_cache[key] = ws
        return ws

    # ------------------------------------------------------------------ forward
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """[B, nc, h, w] float in [0, rgb_range] -> fp32 [B, nc, h*s, w*s]  (src/drct.py:886-899)."""
        sr, _ = self.run(x, want_float=True, want_u8=False)
        return sr

    @torch.no_grad()
    def run(self, x: torch.Tensor, want_float: bool = True, want_u8: bool = False,
            out_u8: Optional[torch.Tensor] = None) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
        """Forward with the evaluator's uint8 truncation (src/evaluate.py:214) fused into the last kernel.
        Returns (sr fp32 NCHW or None, sr uint8 NHWC or None)."""
        if not x.is_cuda:
            raise RuntimeError("input must be a CUDA tensor: this package has no CPU fallback")
        P = self._pack()
        x = x.contiguous().float()
        B, nc, H, W = x.shape
        if nc != self.n_colors:
            raise ValueError(f"expected {self.n_colors} input channels, got {nc}")
        wsz = self.window_size
        if H % wsz or W % wsz:
            raise ValueError(f"input size {H}x{W} must be a multiple of the window size {wsz}")
        dev = x.device
        ws = self._workspace(B, H, W, dev)
        slab, ln, y, z, qkv, att, hb = ws["slab"], ws["ln"], ws["y"], ws["z"], ws["qkv"], ws["att"], ws["h"]
        D = self.embed_dim

        # (x - mean)*img_range -> conv_first -> x0 ; patch_embed.norm(x0) -> slab[:, :D]
        st_slab, st_y = ws["st_slab"], ws["st_y"]
        ops.drct_head(x, P["cf_w"], P["cf_b"], P["mean"], float(self.img_range), P["pe_w"], P["pe_b"], D, ws["x0"], slab,
                      stats_out=st_slab)

        # Tile order: the persistent row-tile kernels (proj / adjust GEMMs, fused MLP) walk their 128-row tiles in either direction.  A
        # batch-256 activation (94 - 168 MB) does not fit the 126 MB L2 next to everything else, but the rows its producer wrote LAST are
        # still there: each of these kernels runs opposite to the kernel that produced its input (the attention kernels always run forward).
        slab_fwd = True                                   # direction in which the current slab contents were written
        for blocks in P["blocks"]:
            # st_slab: x owns the first xs slots (written by adjust5: four partial slots from the folded kernel), each x_j two more
            xs = 4 if blocks[-1].mlp_res is not None else 2 * blocks[-1].adjust.n_tiles
            for k, b in enumerate(blocks):
                C = b.dim
                # ---- W-MSA / SW-MSA half (src/drct.py:478-509); norm1 is folded into the qkv GEMM, its row statistics
                #      are the partial sums the producing epilogues left in st_slab
                fused = b.attn_mode if (H % 8 == 0 and W % 8 == 0 and (B * (H // 8) * (W // 8)) % 2 == 0) else 0
                y_slots = 2 * b.proj.n_tiles
                if fused == 2:
                    ops.swin_attn(slab, b.attn, b.table, y, B, H, W, b.shift, (st_slab, xs + 2 * k), True, stats_out=(st_y, 0))
                    y_slots = 1
                    y_fwd = True
                elif fused == 1:
                    ops.swin_attn(slab, b.attn, b.table, att, B, H, W, b.shift, (st_slab, xs + 2 * k), False)
                    ops.tc_gemm(att, b.heads * b.hdp, b.proj, y, res=slab, stats_out=(st_y, 0), reverse=True)
                    y_fwd = False
                else:
                    ops.tc_gemm(slab, C, b.qkv, qkv, stats_in=(st_slab, xs + 2 * k), reverse=slab_fwd)
                    ops.window_attention(qkv, att, b.table, B, H, W, b.ws, b.shift, b.heads, b.hd, b.hdp)
                    ops.tc_gemm(att, b.heads * b.hdp, b.proj, y, res=slab, stats_out=(st_y, 0), reverse=True)
                    y_fwd = False
                # ---- MLP half (src/drct.py:510, 185-189): norm2 + fc1 + GELU + fc2 + residual in ONE kernel, the hidden
                #      activations never leave the SM
                mlp_rev = y_fwd
                if b.mlp.wadj is not None:
                    # ... and the adjust 1x1 conv (+LeakyReLU 0.2) into the slab slice (src/drct.py:389-393) in the same kernel
                    ops.swin_mlp_adjust(y, C, b.mlp, slab, C, stats_in=(st_y, y_slots), stats_out=(st_slab, xs + 2 * k), reverse=mlp_rev)
                    slab_fwd = not mlp_rev
                    continue
                if b.last and b.mlp_res is not None:
                    # ... and adjust5 + the group's residual: slab[:, :D] = slab[:, :D] + 0.2 adjust5(z), in place, in the same kernel
                    ops.swin_mlp_conv_res(y, C, b.mlp_res, slab, slab, stats_in=(st_y, y_slots), stats_out=(st_slab, 0), reverse=mlp_rev)
                    slab_fwd = not mlp_rev
                    continue
                ops.swin_mlp(y, C, b.mlp, z, stats_in=(st_y, y_slots), reverse=mlp_rev)
                # ---- adjust 1x1 conv (+LeakyReLU 0.2) into the slab slice / 0.2*x5 + x  (src/drct.py:389-396)
                adj_rev = not mlp_rev
                if not b.last:
                    ops.tc_gemm(z, C, b.adjust, slab, act=ops.ACT_LRELU, slope=0.2, ocol0=C, n_store=b.adjust_out,
                                stats_out=(st_slab, xs + 2 * k), reverse=adj_rev)
                else:
                    ops.tc_gemm(z, C, b.adjust, slab, alpha=0.2, res=slab, stats_out=(st_slab, 0), reverse=adj_rev)
                slab_fwd = not adj_rev

        # final norm -> conv_after_body + x0 -> conv_before_upsample + LeakyReLU(0.01) -> upsample -> conv_last
        ops.layernorm_rows(slab, ln, P["norm_w"], P["norm_b"], D)
        ops.conv3x3(ln, B, H, W, D, P["cab"], ws["body"], res=ws["x0"])
        ops.conv3x3(ws["body"], B, H, W, D, P["cbu"], ws["f"], act=ops.ACT_LRELU, slope=0.01)
        cur, ch, cw = ws["f"], H, W
        for pw, dst in zip(P["ups"], ws["ups"]):
            ops.conv3x3(cur, B, ch, cw, 64, pw, dst, out_mode=ops.OUT_PIXEL_SHUFFLE2)
            cur, ch, cw = dst, ch * 2, cw * 2
        sr = torch.empty(B, nc, ch, cw, dtype=torch.float32, device=dev) if want_float else None
        if want_u8 and out_u8 is None:
            out_u8 = torch.empty(B, ch, cw, nc, dtype=torch.uint8, device=dev)
        ops.conv_last_quant(cur, B, ch, cw, 64, P["cl_w"], P["cl_b"], nc, P["mean"], float(self.img_range), self.rgb_range,
                            sr, out_u8 if want_u8 else None)
        return sr, (out_u8 if want_u8 else None)

    # reference API parity helpers
    def no_weight_decay(self):
        return {"absolute_pos_embed"}

    def no_weight_decay_keywords(self):
        return {"relative_position_bias_table"}
