"""Thin torch-tensor wrappers over the C ABI (one Python function per entry point).

Tensors are only carriers of device memory; every function enqueues exactly one kernel on the
current CUDA stream and returns immediately.  `LAUNCHES` counts kernels launched through this
module (bench.py reports it as `gpu_launches`).
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import torch

from . import _abi
from ._abi import ACT_GELU, ACT_LRELU, ACT_NONE, ACT_RELU, OUT_PIXEL_SHUFFLE2, OUT_ROWS, check, lib, ptr, stream_ptr
from .pack import PackedWeight

LAUNCHES = 0
_HALO_CONV = True   # narrow 3x3 convs through csrc/conv_halo.cu; tests and tools/conv_bench.py clear it to run the implicit GEMM instead
PROFILE = None      # set to a list to collect (kind, algorithmic_flops, start_event, end_event) per launch (bench.py)


def _count(kind: str = "", flops: float = 0.0, start=None) -> None:
    global LAUNCHES
    LAUNCHES += 1
    if start is not None:
        end = torch.cuda.Event(enable_timing=True)
        end.record()
        PROFILE.append((kind, flops, start, end))


def _begin():
    if PROFILE is None:
        return None
    ev = torch.cuda.Event(enable_timing=True)
    ev.record()
    return ev


def _cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: this package has no CPU fallback")


def tc_gemm(a: torch.Tensor, k: int, w: PackedWeight, out: torch.Tensor, *, act: int = ACT_NONE, slope: float = 0.0,
            alpha: float = 1.0, res: Optional[torch.Tensor] = None, ocol0: int = 0, n_store: Optional[int] = None,
            m: Optional[int] = None, stats_in: Optional[tuple] = None, stats_out: Optional[tuple] = None, reverse: bool = False) -> None:
    """out[:, ocol0:ocol0+n_store] = alpha * act(a[:, :k] @ W^T + b) (+ res[:, :N]).

    If `w` was packed with pack_ln_gemm_weight the rows of `a` are layer-normalised over their first k columns on the fly;
    their (sum, sumsq) come from stats_in = (fp32 tensor [M, S, 2], number of leading slots to add up).
    stats_out = (fp32 tensor [M, S, 2], first slot) makes this call write such partials for ITS output rows
    (slots first .. first + 2*n_tiles - 1).
    reverse: the row-tile kernel walks its 128-row tiles from the last one down (the rows the producer of `a` wrote last are in L2)."""
    _cuda(a, "a")
    m = a.shape[0] if m is None else m
    n_store = (w.N + 15) // 16 * 16 if n_store is None else n_store
    if (w.colsum is not None) != (stats_in is not None):
        raise ValueError("LayerNorm-folded weights need stats_in (and only they do)")
    si_t, si_n = stats_in if stats_in is not None else (None, 0)
    so_t, so_0 = stats_out if stats_out is not None else (None, 0)
    _t = _begin()
    check(lib().adsr_tc_gemm_bf16(ptr(a), a.stride(0), m, k, ptr(w.data), ptr(w.bias), w.N, w.BN, w.n_tiles, act, slope,
                                  alpha, ptr(res), res.stride(0) if res is not None else 0, ptr(out), out.stride(0), ocol0,
                                  n_store, ptr(w.colsum), w.ln_eps, ptr(si_t), si_n, si_t.shape[1] if si_t is not None else 0,
                                  ptr(so_t), so_0, so_t.shape[1] if so_t is not None else 0, int(reverse), _abi.num_sms(), stream_ptr()),
          "adsr_tc_gemm_bf16")
    _count("tc_gemm", 2.0 * m * k * w.N, _t)


def swin_mlp(y: torch.Tensor, c: int, pm, z: torch.Tensor, stats_in: tuple, m: Optional[int] = None, reverse: bool = False) -> None:
    """z[:, :c] = y + fc2(GELU(fc1(LayerNorm(y[:, :c]))))  -- one fused kernel (csrc/swin_mlp.cu); `pm` from
    pack.pack_swin_mlp, stats_in = (fp32 [M, S, 2] partial (sum, sumsq) of the rows of y, slots to add up)."""
    _cuda(y, "y")
    _cuda(z, "z")
    if y.data_ptr() == z.data_ptr():
        raise ValueError("swin_mlp: y and z must not alias")
    m = y.shape[0] if m is None else m
    si_t, si_n = stats_in
    _t = _begin()
    check(lib().adsr_swin_mlp_bf16(ptr(y), y.stride(0), m, c, ptr(pm.w1), ptr(pm.w2), ptr(pm.bias1), ptr(pm.colsum1), ptr(pm.bias2),
                                   pm.plan.data_ptr(), pm.plan.numel(), pm.ln_eps, ptr(si_t), si_n, si_t.shape[1],
                                   ptr(z), z.stride(0), int(reverse), _abi.num_sms(), stream_ptr()), "adsr_swin_mlp_bf16")
    _count("swin_mlp", 4.0 * m * pm.C * pm.H, _t)


def swin_mlp_adjust(y: torch.Tensor, c: int, pm, out: torch.Tensor, ocol0: int, stats_in: tuple, stats_out: Optional[tuple] = None,
                    slope: float = 0.2, m: Optional[int] = None, reverse: bool = False) -> None:
    """out[:, ocol0:ocol0+32] = LReLU_slope(adjust(z)),  z = y + fc2(GELU(fc1(LayerNorm(y[:, :c]))))  -- the fused MLP kernel with
    the RDG's adjust 1x1 conv in its last epilogue; z is never written.  `pm` from pack.pack_swin_mlp(..., adjust_w, adjust_b)."""
    _cuda(y, "y")
    _cuda(out, "out")
    if pm.wadj is None:
        raise ValueError("swin_mlp_adjust: weights were packed without the adjust conv")
    m = y.shape[0] if m is None else m
    si_t, si_n = stats_in
    so_t, so_0 = stats_out if stats_out is not None else (None, 0)
    _t = _begin()
    check(lib().adsr_swin_mlp_adjust_bf16(ptr(y), y.stride(0), m, c, ptr(pm.w1), ptr(pm.w2), ptr(pm.bias1), ptr(pm.colsum1), ptr(pm.bias2),
                                          pm.plan.data_ptr(), pm.plan.numel(), pm.ln_eps, ptr(si_t), si_n, si_t.shape[1],
                                          ptr(pm.wadj), ptr(pm.bias_adj), slope, ptr(out), out.stride(0), ocol0, ptr(so_t), so_0,
                                          so_t.shape[1] if so_t is not None else 0, int(reverse), _abi.num_sms(), stream_ptr()),
          "adsr_swin_mlp_adjust_bf16")
    _count("swin_mlp", 4.0 * m * pm.C * pm.H + 2.0 * m * pm.C * 32, _t)


def swin_mlp_conv_res(y: torch.Tensor, c: int, pm, res: torch.Tensor, out: torch.Tensor, stats_in: tuple,
                      stats_out: Optional[tuple] = None, m: Optional[int] = None, reverse: bool = False) -> None:
    """out[:, :c_out] = res[:, :c_out] + alpha * conv(z),  z = y + fc2(GELU(fc1(LayerNorm(y[:, :c]))))  -- the fused MLP kernel with a
    wide 1x1 conv (adjust5 of the RDG) and the residual folded in; z is never written, out may alias res.  `pm` from
    pack.pack_swin_mlp_conv_res(...); stats_out receives the row's (sum, sumsq) of the c_out output columns as four partial slots."""
    _cuda(y, "y")
    _cuda(res, "res")
    _cuda(out, "out")
    if not getattr(pm, "conv_out", 0):
        raise ValueError("swin_mlp_conv_res: weights were not packed by pack_swin_mlp_conv_res")
    m = y.shape[0] if m is None else m
    si_t, si_n = stats_in
    so_t, so_0 = stats_out if stats_out is not None else (None, 0)
    _t = _begin()
    check(lib().adsr_swin_mlp_conv_res_bf16(ptr(y), y.stride(0), m, c, ptr(pm.w1), ptr(pm.w2), ptr(pm.bias1), ptr(pm.colsum1), ptr(pm.bias2),
                                            pm.plan.data_ptr(), pm.plan.numel(), pm.ln_eps, ptr(si_t), si_n, si_t.shape[1],
                                            ptr(res), res.stride(0), ptr(out), out.stride(0), pm.conv_out, ptr(so_t), so_0,
                                            so_t.shape[1] if so_t is not None else 0, int(reverse), _abi.num_sms(), stream_ptr()),
          "adsr_swin_mlp_conv_res_bf16")
    _count("swin_mlp", 2.0 * m * pm.C * pm.H + 2.0 * m * pm.H * pm.conv_out + 2.0 * m * pm.C * pm.conv_out, _t)


def swin_attn_mode(c: int, heads: int, hdp: int, allow_proj: bool = True) -> int:
    """What adsr_swin_attn_bf16 covers for this block shape: 2 = whole attention half, 1 = qkv + attention, 0 = nothing."""
    return int(lib().adsr_swin_attn_mode(c, heads, hdp, int(allow_proj)))


def swin_attn(x: torch.Tensor, pa, table: torch.Tensor, out: torch.Tensor, b: int, h: int, w: int, shift: int, stats_in: tuple,
              fuse_proj: bool, stats_out: Optional[tuple] = None) -> None:
    """fuse_proj: out[:, :C] = x + proj(W-MSA(LayerNorm(x[:, :C])))  else  out = attention rows [M, heads*hdp]
    -- one fused kernel (csrc/swin_attn.cu); `pa` from pack.pack_swin_attn, stats as in tc_gemm (stats_out: ONE slot)."""
    _cuda(x, "x")
    _cuda(out, "out")
    if x.data_ptr() == out.data_ptr():
        raise ValueError("swin_attn: x and out must not alias")
    si_t, si_n = stats_in
    so_t, so_0 = stats_out if stats_out is not None else (None, 0)
    m = b * h * w
    _t = _begin()
    check(lib().adsr_swin_attn_bf16(ptr(x), x.stride(0), b, h, w, pa.C, shift, pa.heads, pa.hd, pa.hdp, ptr(pa.w1), ptr(pa.w2),
                                    ptr(pa.bias_qkv), ptr(pa.colsum_qkv), ptr(pa.bias_p), ptr(table), pa.ln_eps, ptr(si_t), si_n,
                                    si_t.shape[1], int(fuse_proj), ptr(out), out.stride(0), ptr(so_t), so_0,
                                    so_t.shape[1] if so_t is not None else 0, _abi.num_sms(), stream_ptr()), "adsr_swin_attn_bf16")
    n_keys = 64                                                # this kernel covers 8 x 8 windows only (16 x 16: window_attention)
    flops = 2.0 * m * pa.C * 3 * pa.C + 4.0 * m * n_keys * pa.C + (2.0 * m * pa.C * pa.C if fuse_proj else 0.0)
    _count("swin_attn", flops, _t)


def conv3x3(x: torch.Tensor, b: int, h: int, wd: int, cin: int, w: PackedWeight, out: torch.Tensor, *, stride: int = 1,
            act: int = ACT_NONE, slope: float = 0.0, alpha: float = 1.0, res: Optional[torch.Tensor] = None,
            out_mode: int = OUT_ROWS, n_store: Optional[int] = None, ocol0: int = 0, chan_part: Optional[torch.Tensor] = None) -> bool:
    """x: [b*h*wd, ld] NHWC bf16 -> out rows (b*ho*wo) [at column ocol0] or pixel-shuffled [b, 2h, 2w, N/4].
    chan_part: optional fp32 [b * halo_parts(h, wd), round16(N)] scratch; returns True when the halo-tile kernel ran and filled it
    with per-image partial column sums (channel_mean_parts turns them into CALayer's pooled means)."""
    _cuda(x, "x")
    n_store = (w.N + 15) // 16 * 16 if n_store is None else n_store
    _t = _begin()
    wc = w.compact
    if (wc is not None and _HALO_CONV and stride == 1 and res is None and out_mode == OUT_ROWS and alpha == 1.0 and 8 <= wd <= 126
            and n_store <= wc.BN and n_store % 8 == 0 and ocol0 % 8 == 0 and act in (ACT_NONE, ACT_RELU, ACT_LRELU)):
        # narrow layer: halo tile + resident weights (csrc/conv_halo.cu); BAD_SHAPE = does not fit the SM, fall through
        st = lib().adsr_conv3x3_halo_bf16(ptr(x), x.stride(0), b, h, wd, cin, ptr(wc.data), ptr(wc.bias), wc.N, wc.BN, act, slope,
                                          ptr(out), out.stride(0), ocol0, n_store, ptr(chan_part), _abi.num_sms(), stream_ptr())
        if st != 1:                       # ADSR_ERR_BAD_SHAPE
            check(st, "adsr_conv3x3_halo_bf16")
            _count("conv3x3_halo", 2.0 * b * h * wd * 9 * cin * w.N, _t)
            return chan_part is not None
    check(lib().adsr_conv3x3_igemm_bf16(ptr(x), x.stride(0), b, h, wd, cin, stride, ptr(w.data), ptr(w.bias), w.N, w.BN,
                                        w.n_tiles, act, slope, alpha, ptr(res), res.stride(0) if res is not None else 0,
                                        ptr(out), out.stride(0), ocol0, out_mode, n_store, _abi.num_sms(), stream_ptr()),
          "adsr_conv3x3_igemm_bf16")
    _count("conv3x3", 2.0 * b * (-(-h // stride)) * (-(-wd // stride)) * 9 * cin * w.N, _t)
    return False


def halo_parts(h: int, wd: int) -> int:
    """Partial-sum rows per image written by the halo conv: 4 row quadrants per 128-position tile of the padded raster."""
    return 4 * ((h * (wd + 2) + 127) // 128)


def channel_mean_parts(part: torch.Tensor, b: int, parts: int, c: int, hw: int, mean: torch.Tensor, w1=None, b1=None, w2=None, b2=None,
                       cr: int = 0) -> None:
    """mean [b, c] <- pooled means from the halo conv's partial sums; with the CALayer weights given: the sigmoid scales instead
    (pass them to rcab_ca_scale with cr=0)."""
    _t = _begin()
    check(lib().adsr_channel_mean_parts(ptr(part), b, parts, part.stride(0), c, hw, ptr(mean), ptr(w1), ptr(b1), ptr(w2), ptr(b2), cr,
                                        stream_ptr()), "adsr_channel_mean_parts")
    _count("channel_mean_parts", 0.0, _t)


def layernorm_rows(x: torch.Tensor, out: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, c: int, eps: float = 1e-5,
                   m: Optional[int] = None) -> None:
    _cuda(x, "x")
    m = x.shape[0] if m is None else m
    _t = _begin()
    check(lib().adsr_layernorm_rows(ptr(x), x.stride(0), ptr(out), out.stride(0), ptr(gamma), ptr(beta), m, c, eps,
                                    stream_ptr()), "adsr_layernorm_rows")
    _count("layernorm", 0.0, _t)


def window_attention(qkv: torch.Tensor, out: torch.Tensor, table: torch.Tensor, b: int, h: int, w: int, ws: int,
                     shift: int, heads: int, hd: int, hdp: int) -> None:
    _cuda(qkv, "qkv")
    _t = _begin()
    check(lib().adsr_window_attention(ptr(qkv), qkv.stride(0), ptr(out), out.stride(0), ptr(table), b, h, w, ws, shift,
                                      heads, hd, hdp, stream_ptr()), "adsr_window_attention")
    _count("window_attention", 4.0 * b * h * w * ws * ws * heads * hd, _t)


def window_index_map(h: int, w: int, ws: int, shift: int, device) -> tuple[torch.Tensor, torch.Tensor]:
    n = (h // ws) * (w // ws) * ws * ws
    src = torch.empty(n, dtype=torch.int32, device=device)
    reg = torch.empty(n, dtype=torch.int32, device=device)
    _t = _begin()
    check(lib().adsr_window_index_map(h, w, ws, shift, ptr(src), ptr(reg), stream_ptr()), "adsr_window_index_map")
    _count("index_map", 0.0, _t)
    return src, reg


def ln_shift_partition(x: torch.Tensor, windows: torch.Tensor, gamma, beta, b, h, w, c, ws, shift, eps=1e-5) -> None:
    _cuda(x, "x")
    _t = _begin()
    check(lib().adsr_ln_shift_partition(ptr(x), x.stride(0), ptr(windows), windows.stride(0), ptr(gamma), ptr(beta), eps, b,
                                        h, w, c, ws, shift, stream_ptr()), "adsr_ln_shift_partition")
    _count("ln_shift_partition", 0.0, _t)


def window_reverse_unshift(windows: torch.Tensor, x: torch.Tensor, b, h, w, c, ws, shift) -> None:
    _cuda(x, "x")
    _t = _begin()
    check(lib().adsr_window_reverse_unshift(ptr(windows), windows.stride(0), ptr(x), x.stride(0), b, h, w, c, ws, shift,
                                            stream_ptr()), "adsr_window_reverse_unshift")
    _count("window_reverse", 0.0, _t)


def drct_head(x: torch.Tensor, weight, bias, mean, img_range: float, gamma, beta, c: int, x0: torch.Tensor,
              slab: torch.Tensor, eps: float = 1e-5, stats_out: Optional[torch.Tensor] = None) -> None:
    _cuda(x, "x")
    b, nc, h, w = x.shape
    _t = _begin()
    check(lib().adsr_drct_head(ptr(x), b, nc, h, w, ptr(weight), ptr(bias), ptr(mean), img_range, ptr(gamma), ptr(beta), eps,
                               c, ptr(x0), x0.stride(0), ptr(slab), slab.stride(0), ptr(stats_out),
                               stats_out.shape[1] if stats_out is not None else 0, stream_ptr()), "adsr_drct_head")
    _count("drct_head", 2.0 * b * h * w * 9 * nc * c, _t)


def conv_last_quant(x: torch.Tensor, b: int, h: int, w: int, cin: int, weight, bias, nc: int, mean, img_range: float,
                    rgb_range: float, out: Optional[torch.Tensor], out_u8: Optional[torch.Tensor]) -> None:
    _cuda(x, "x")
    _t = _begin()
    check(lib().adsr_conv_last_quant(ptr(x), x.stride(0), b, h, w, cin, ptr(weight), ptr(bias), nc, ptr(mean), img_range,
                                     rgb_range, ptr(out), ptr(out_u8), stream_ptr()), "adsr_conv_last_quant")
    _count("conv_last", 2.0 * b * h * w * 9 * cin * nc, _t)


def u8_to_float(x_u8: torch.Tensor, rgb_range: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 NHWC (decoded PNGs) -> fp32 NCHW in [0, rgb_range]: the loader's `np2Tensor` (src/data.py:11-17) on the device."""
    _cuda(x_u8, "x_u8")
    assert x_u8.dtype == torch.uint8 and x_u8.dim() == 4
    x_u8 = x_u8.contiguous()
    b, h, w, nc = x_u8.shape
    if out is None:
        out = torch.empty(b, nc, h, w, dtype=torch.float32, device=x_u8.device)
    _t = _begin()
    check(lib().adsr_u8_to_float_nchw(ptr(x_u8), b, nc, h, w, rgb_range, ptr(out), stream_ptr()), "adsr_u8_to_float_nchw")
    _count("u8_to_float", 0.0, _t)
    return out


def quantize_u8(x: torch.Tensor, rgb_range: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 NCHW in [0, rgb_range] -> uint8 NHWC, truncating (src/evaluate.py:214-215)."""
    _cuda(x, "x")
    x = x.contiguous().float()
    b, nc, h, w = x.shape
    if out is None:
        out = torch.empty(b, h, w, nc, dtype=torch.uint8, device=x.device)
    _t = _begin()
    check(lib().adsr_quantize_u8(ptr(x), b, nc, h, w, rgb_range, ptr(out), stream_ptr()), "adsr_quantize_u8")
    _count("quantize_u8", 0.0, _t)
    return out


def score_images(sr_u8: torch.Tensor, hr_u8: torch.Tensor, window_sizes: Sequence[int],
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 NHWC pairs -> fp64 [B, n_ws + 2] = SSIM per window size, MSE, PSNR."""
    _cuda(sr_u8, "sr_u8")
    assert sr_u8.shape == hr_u8.shape and sr_u8.dtype == torch.uint8 and hr_u8.dtype == torch.uint8
    sr_u8, hr_u8 = sr_u8.contiguous(), hr_u8.contiguous()
    b, h, w, c = sr_u8.shape
    n_ws = len(window_sizes)
    if out is None:
        out = torch.empty(b, n_ws + 2, dtype=torch.float64, device=sr_u8.device)
    arr = (ctypes.c_int32 * max(n_ws, 1))(*window_sizes)
    _t = _begin()
    check(lib().adsr_score_images(ptr(sr_u8), ptr(hr_u8), b, h, w, c, arr, n_ws, ptr(out), stream_ptr()),
          "adsr_score_images")
    _count("score_images", 0.0, _t)
    return out


def anomaly_maps(sr_u8: torch.Tensor, hr_u8: torch.Tensor, win_size: int, sigma: float = 0.0,
                 out: Optional[tuple] = None) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """uint8 NHWC pairs -> (ssim_map fp32 [B, H, W] = 1 - SSIM per pixel for one window size, se_map fp32 [B, H, W] = squared error
    averaged over the channels, map_max fp64 [B, 2] = per-image max of both maps), Gaussian-smoothed when sigma > 0.
    out: caller-owned (ssim_map, se_map, map_max, scratch) to write into; scratch is the fp32 [B, H, W] buffer of the smoothing and
    may be None when sigma == 0.  Without `out` everything is allocated here.  Two kernels, six with the smoothing."""
    _cuda(sr_u8, "sr_u8")
    _cuda(hr_u8, "hr_u8")
    if sr_u8.dtype != torch.uint8 or hr_u8.dtype != torch.uint8:
        raise TypeError(f"anomaly_maps takes uint8 images, got {sr_u8.dtype} / {hr_u8.dtype}")
    if sr_u8.dim() != 4 or sr_u8.shape != hr_u8.shape or sr_u8.device != hr_u8.device:
        raise ValueError(f"anomaly_maps needs two [B, H, W, C] images of one shape on one device, got {tuple(sr_u8.shape)} on "
                         f"{sr_u8.device} and {tuple(hr_u8.shape)} on {hr_u8.device}")
    sr_u8, hr_u8 = sr_u8.contiguous(), hr_u8.contiguous()
    b, h, w, c = sr_u8.shape
    if out is None:
        f32 = dict(dtype=torch.float32, device=sr_u8.device)
        out = (torch.empty(b, h, w, **f32), torch.empty(b, h, w, **f32),
               torch.empty(b, 2, dtype=torch.float64, device=sr_u8.device), torch.empty(b, h, w, **f32) if sigma > 0 else None)
    ssim_map, se_map, map_max, scratch = out
    for t, name, dt, shape in ((ssim_map, "ssim_map", torch.float32, (b, h, w)), (se_map, "se_map", torch.float32, (b, h, w)),
                               (map_max, "map_max", torch.float64, (b, 2)), (scratch, "scratch", torch.float32, (b, h, w))):
        if t is None and name == "scratch":
            continue
        if t.dtype != dt or tuple(t.shape) != shape or not t.is_contiguous() or t.device != sr_u8.device:
            raise ValueError(f"anomaly_maps: {name} must be a contiguous {dt} tensor of shape {shape} on {sr_u8.device}")
    _t = _begin()
    check(lib().adsr_anomaly_maps(ptr(sr_u8), ptr(hr_u8), b, h, w, c, int(win_size), float(sigma), ptr(ssim_map), ptr(se_map),
                                  ptr(scratch), ptr(map_max), stream_ptr()), "adsr_anomaly_maps")
    global LAUNCHES
    LAUNCHES += 5 if sigma > 0 else 1                  # raw maps [+ row / column Gaussian passes of both maps]; _count adds the max
    _count("anomaly_maps", 0.0, _t)
    return ssim_map, se_map, map_max


def gms_workspace_bytes(b: int, h: int, w: int) -> int:
    """Bytes of scratch adsr_gms_map needs for B images of H x W (both gray pyramids, the per-level similarity planes, the Gaussian
    scratch)."""
    n = int(lib().adsr_gms_workspace_bytes(int(b), int(h), int(w)))
    if n < 0:
        raise ValueError(f"gms_map: unsupported batch shape {b} x {h} x {w}")
    return n


def gms_map(sr_u8: torch.Tensor, hr_u8: torch.Tensor, sigma: float = 0.0,
            out: Optional[tuple] = None) -> tuple[torch.Tensor, torch.Tensor]:
    """uint8 NHWC pairs -> (gms_map fp32 [B, H, W] = the multi-scale gradient-magnitude-similarity map (1/4) sum over 4 pyramid levels
    of the upsampled 1 - GMS of the gray planes, map_max fp64 [B] = per-image max of the map), Gaussian-smoothed like anomaly_maps when
    sigma > 0.  out: caller-owned (gms_map, map_max, workspace) to write into; workspace is uint8 [>= gms_workspace_bytes(B, H, W)].
    Without `out` everything is allocated here.  Four kernels, six with the smoothing."""
    _cuda(sr_u8, "sr_u8")
    _cuda(hr_u8, "hr_u8")
    if sr_u8.dtype != torch.uint8 or hr_u8.dtype != torch.uint8:
        raise TypeError(f"gms_map takes uint8 images, got {sr_u8.dtype} / {hr_u8.dtype}")
    if sr_u8.dim() != 4 or sr_u8.shape != hr_u8.shape or sr_u8.device != hr_u8.device:
        raise ValueError(f"gms_map needs two [B, H, W, C] images of one shape on one device, got {tuple(sr_u8.shape)} on "
                         f"{sr_u8.device} and {tuple(hr_u8.shape)} on {hr_u8.device}")
    sr_u8, hr_u8 = sr_u8.contiguous(), hr_u8.contiguous()
    b, h, w, c = sr_u8.shape
    ws_bytes = gms_workspace_bytes(b, h, w)
    if out is None:
        out = (torch.empty(b, h, w, dtype=torch.float32, device=sr_u8.device), torch.empty(b, dtype=torch.float64, device=sr_u8.device),
               torch.empty(ws_bytes, dtype=torch.uint8, device=sr_u8.device))
    gms, map_max, workspace = out
    for t, name, dt, shape in ((gms, "gms_map", torch.float32, (b, h, w)), (map_max, "map_max", torch.float64, (b,))):
        if t.dtype != dt or tuple(t.shape) != shape or not t.is_contiguous() or t.device != sr_u8.device:
            raise ValueError(f"gms_map: {name} must be a contiguous {dt} tensor of shape {shape} on {sr_u8.device}")
    if workspace.dtype != torch.uint8 or not workspace.is_contiguous() or workspace.device != sr_u8.device or workspace.numel() < ws_bytes:
        raise ValueError(f"gms_map: workspace must be a contiguous uint8 tensor of at least {ws_bytes} bytes on {sr_u8.device}")
    _t = _begin()
    check(lib().adsr_gms_map(ptr(sr_u8), ptr(hr_u8), b, h, w, c, float(sigma), ptr(gms), ptr(map_max), ptr(workspace), stream_ptr()),
          "adsr_gms_map")
    global LAUNCHES
    LAUNCHES += 5 if sigma > 0 else 3                  # pyramid, levels, combine [+ row / column Gaussian passes]; _count adds the max
    _count("gms_map", 0.0, _t)
    return gms, map_max


def localisation_workspace_bytes(n: int) -> int:
    """Bytes of scratch adsr_localisation_metrics needs for n pixels (two key / region buffer pairs, sort histograms, tile sums)."""
    b = int(lib().adsr_localisation_workspace_bytes(int(n)))
    if b < 0:
        raise ValueError(f"localisation metrics: unsupported pixel count {n}")
    return b


def localisation_metrics(scores: torch.Tensor, regions: torch.Tensor, region_sizes: torch.Tensor, n_ok: int, fpr_limit: float,
                         workspace: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """Pixel AUROC, AU-PRO@fpr_limit, pixel AP and F1-max of one map: scores fp32 [n], regions int32 [n] (-1 = defect-free, else an
    index into region_sizes int64 [R]), n_ok defect-free pixels -> out fp64 [8] = (pixel AUROC, AU-PRO, NaN scores, defect-free pixels
    seen, out-of-range region indices, pixel AP, F1-max, F1 threshold).  workspace: uint8 [>= localisation_workspace_bytes(n)].
    Sixteen kernels, no synchronisation."""
    for t, name, dt in ((scores, "scores", torch.float32), (regions, "regions", torch.int32), (region_sizes, "region_sizes", torch.int64),
                        (workspace, "workspace", torch.uint8), (out, "out", torch.float64)):
        _cuda(t, name)
        if t.dtype != dt or not t.is_contiguous():
            raise ValueError(f"localisation_metrics: {name} must be a contiguous {dt} tensor")
    n = scores.numel()
    if regions.numel() != n or out.numel() < 8:
        raise ValueError(f"localisation_metrics: {n} scores, {regions.numel()} region indices, out of {out.numel()} values")
    _t = _begin()
    check(lib().adsr_localisation_metrics(ptr(scores), ptr(regions), n, ptr(region_sizes), region_sizes.numel(), int(n_ok),
                                          float(fpr_limit), ptr(workspace), workspace.numel(), ptr(out), stream_ptr()),
          "adsr_localisation_metrics")
    global LAUNCHES
    LAUNCHES += 15                                     # 4 radix passes x 3 kernels + tile sums + tile scan + curve; _count adds the last
    _count("localisation_metrics", 0.0, _t)
    return out


def _check_tensors(what: str, *specs) -> None:
    for t, name, dt in specs:
        _cuda(t, name)
        if t.dtype != dt or not t.is_contiguous():
            raise ValueError(f"{what}: {name} must be a contiguous {dt} tensor")


def score_quantile(scores: torch.Tensor, k: int, workspace: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """The exact k-th smallest of the fp32 scores [n], 1 <= k <= n (-0.0 reported as +0.0) -> out fp64 [2] = (score, NaN scores; the
    score is NaN when fewer than k scores are not NaN).  workspace: uint8 [>= localisation_workspace_bytes(n)].  A radix select: eight
    kernels, no synchronisation."""
    _check_tensors("score_quantile", (scores, "scores", torch.float32), (workspace, "workspace", torch.uint8),
                   (out, "out", torch.float64))
    n = scores.numel()
    if not 1 <= int(k) <= n or out.numel() < 2:
        raise ValueError(f"score_quantile: rank {k} of {n} scores, out of {out.numel()} values")
    _t = _begin()
    check(lib().adsr_score_quantile(ptr(scores), n, int(k), ptr(workspace), workspace.numel(), ptr(out), stream_ptr()),
          "adsr_score_quantile")
    global LAUNCHES
    LAUNCHES += 7                                      # 4 passes x (histogram + pick); _count adds the last
    _count("score_quantile", 0.0, _t)
    return out


def threshold_metrics(scores: torch.Tensor, regions: torch.Tensor, region_sizes: Optional[torch.Tensor], threshold: float,
                      workspace: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """Pixel counts of the prediction `scores >= threshold` (an fp32 value, not NaN) against the regions of localisation_metrics:
    out fp64 [7] = (TP, FP, FN, TN, PRO@threshold (NaN without regions), NaN scores, out-of-range region indices).  region_sizes may be
    None when no pixel belongs to a region.  Two kernels, no synchronisation."""
    specs = [(scores, "scores", torch.float32), (regions, "regions", torch.int32), (workspace, "workspace", torch.uint8),
             (out, "out", torch.float64)]
    if region_sizes is not None:
        specs.append((region_sizes, "region_sizes", torch.int64))
    _check_tensors("threshold_metrics", *specs)
    n = scores.numel()
    if regions.numel() != n or out.numel() < 7:
        raise ValueError(f"threshold_metrics: {n} scores, {regions.numel()} region indices, out of {out.numel()} values")
    _t = _begin()
    check(lib().adsr_threshold_metrics(ptr(scores), ptr(regions), n, ptr(region_sizes),
                                       0 if region_sizes is None else region_sizes.numel(), float(threshold), ptr(workspace),
                                       workspace.numel(), ptr(out), stream_ptr()), "adsr_threshold_metrics")
    global LAUNCHES
    LAUNCHES += 1                                      # counting pass; _count adds the reduction
    _count("threshold_metrics", 0.0, _t)
    return out


def score_images_strided(sr: torch.Tensor, hr: torch.Tensor, layout: str, window_sizes: Sequence[int], *, div: float = 1.0,
                         clamp01: bool = False, zero_pad: bool = False, c1: float = 1e-4, c2: float = 9e-4,
                         psnr_peak: float = 1.0) -> torch.Tensor:
    """Generic scorer behind psnr/ssim_numpy (float or uint8 HWC) and psnr/ssim_torch (fp32 NCHW views).
    layout: "hwc" -> tensors [B, H, W, C]; "chw" -> [B, C, H, W] (any strides, e.g. a shaved crop)."""
    _cuda(sr, "sr")
    assert sr.shape == hr.shape and sr.dtype == hr.dtype and sr.dtype in (torch.uint8, torch.float32)
    if layout == "hwc":
        b, h, w, c = sr.shape
        st = lambda t: (t.stride(0), t.stride(1), t.stride(2), t.stride(3))
    else:
        b, c, h, w = sr.shape
        st = lambda t: (t.stride(0), t.stride(2), t.stride(3), t.stride(1))
    n_ws = len(window_sizes)
    out = torch.empty(b, n_ws + 2, dtype=torch.float64, device=sr.device)
    arr = (ctypes.c_int32 * max(n_ws, 1))(*window_sizes)
    s_sr, s_hr = (ctypes.c_int64 * 4)(*st(sr)), (ctypes.c_int64 * 4)(*st(hr))
    _t = _begin()
    check(lib().adsr_score_images_strided(ptr(sr), ptr(hr), int(sr.dtype == torch.float32), b, h, w, c, s_sr, s_hr, div,
                                          int(clamp01), int(zero_pad), c1, c2, psnr_peak, arr, n_ws, ptr(out), stream_ptr()),
          "adsr_score_images_strided")
    _count("score_images", 0.0, _t)
    return out


def validate_images(sr: torch.Tensor, hr: torch.Tensor, rgb_range: float, win_size: int = 11) -> torch.Tensor:
    """fp32 [B, C, H, W] views (any strides, e.g. the shaved crop) -> fp64 [B, 3] = ssim_torch, mse, psnr_torch per image of the
    ROUND-quantised SR against HR: the body of the reference's validation loop (src/trainer.py:266-281) in one launch."""
    _cuda(sr, "sr")
    assert sr.shape == hr.shape and sr.dtype == torch.float32 and hr.dtype == torch.float32
    b, c, h, w = sr.shape
    st = lambda t: (ctypes.c_int64 * 4)(t.stride(0), t.stride(2), t.stride(3), t.stride(1))
    out = torch.empty(b, 3, dtype=torch.float64, device=sr.device)
    _t = _begin()
    check(lib().adsr_validate_images(ptr(sr), ptr(hr), b, h, w, c, st(sr), st(hr), float(rgb_range), int(win_size), ptr(out),
                                     stream_ptr()), "adsr_validate_images")
    _count("score_images", 0.0, _t)
    return out


def bicubic_affine(x: torch.Tensor, scale: int, mat: torch.Tensor, bias: torch.Tensor, out: torch.Tensor) -> None:
    _cuda(x, "x")
    b, nc, h, w = x.shape
    _t = _begin()
    check(lib().adsr_bicubic_affine(ptr(x), b, nc, h, w, scale, ptr(mat), ptr(bias), ptr(out), stream_ptr()),
          "adsr_bicubic_affine")
    _count("bicubic", 0.0, _t)


def conv3x3_small(x: torch.Tensor, weight, bias, c: int, out1: torch.Tensor, out2: Optional[torch.Tensor] = None,
                  col2: int = 0) -> None:
    _cuda(x, "x")
    b, nc, h, w = x.shape
    _t = _begin()
    check(lib().adsr_conv3x3_small(ptr(x), b, nc, h, w, ptr(weight), ptr(bias), c, ptr(out1), out1.stride(0), ptr(out2),
                                   out2.stride(0) if out2 is not None else 0, col2, stream_ptr()), "adsr_conv3x3_small")
    _count("conv3x3_small", 2.0 * b * h * w * 9 * nc * c, _t)


def channel_mean(x: torch.Tensor, b: int, hw: int, c: int, mean: torch.Tensor) -> None:
    _cuda(x, "x")
    _t = _begin()
    check(lib().adsr_channel_mean(ptr(x), x.stride(0), b, hw, c, ptr(mean), stream_ptr()), "adsr_channel_mean")
    _count("channel_mean", 0.0, _t)


def rcab_ca_scale(res: torch.Tensor, x: torch.Tensor, out: torch.Tensor, mean, w1, b1, w2, b2, b: int, hw: int, c: int,
                  cr: int) -> None:
    _cuda(res, "res")
    _t = _begin()
    check(lib().adsr_rcab_ca_scale(ptr(res), res.stride(0), ptr(x), x.stride(0), ptr(out), out.stride(0), ptr(mean), ptr(w1),
                                   ptr(b1), ptr(w2), ptr(b2), b, hw, c, cr, stream_ptr()), "adsr_rcab_ca_scale")
    _count("rcab_ca_scale", 0.0, _t)
