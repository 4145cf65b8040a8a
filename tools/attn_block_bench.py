"""Timing of the fused attention half (csrc/swin_attn.cu) per DRCT block shape (CUDA events, L2 flushed), next to the
separate qkv GEMM + window attention + proj GEMM it replaces."""
import importlib, sys, os
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PKG = "anomaly-detection-super-resolution_b200"
ops = importlib.import_module(PKG + ".ops"); pack = importlib.import_module(PKG + ".pack")
dev = "cuda"
B = int(os.environ.get("B", 256)); H = W = 32
M = B * H * W
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

def timeit(fn, reps=5):
    fn(); torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return min(ts), sum(ts) / len(ts)

shapes = [(180, 6, 0), (212, 4, 4), (244, 2, 0), (276, 6, 4), (308, 4, 0)]
if os.environ.get("ATTN_ONLY"):
    shapes = [s for s in shapes if s[0] == int(os.environ["ATTN_ONLY"])]
for (C, heads, shift) in shapes:
    hd = C // heads; hdp = pack.head_pad(hd)
    x = torch.randn(M, 320, device=dev).to(torch.bfloat16)
    y = torch.empty_like(x)
    qkv_w, qkv_b = torch.randn(3 * C, C, device=dev) * 0.05, torch.randn(3 * C, device=dev) * 0.1
    proj_w, proj_b = torch.randn(C, C, device=dev) * 0.05, torch.randn(C, device=dev) * 0.1
    g, bt = torch.ones(C, device=dev), torch.zeros(C, device=dev)
    table = torch.randn(225, heads, device=dev) * 0.2
    pa = pack.pack_swin_attn(qkv_w, qkv_b, g, bt, 1e-5, proj_w, proj_b, heads)
    pq = pack.pack_qkv_weight(qkv_w, qkv_b, heads, g, bt, 1e-5)
    pp = pack.pack_proj_weight(proj_w, proj_b, heads)
    stats = torch.zeros(M, 2, 2, device=dev)
    xf = x[:, :C].float(); stats[:, 0, 0] = xf.sum(1); stats[:, 0, 1] = (xf * xf).sum(1)
    st_y = torch.zeros(M, 8, 2, device=dev)
    qkv = torch.empty(M, 3 * heads * hdp, device=dev, dtype=torch.bfloat16)
    att = torch.empty(M, heads * hdp, device=dev, dtype=torch.bfloat16)
    mode = ops.swin_attn_mode(C, heads, hdp, True)
    fl = 2.0 * M * C * 3 * C + 4.0 * M * 64 * C + 2.0 * M * C * C

    def fused():
        if mode == 2:
            ops.swin_attn(x, pa, table, y, B, H, W, shift, (stats, 2), True, stats_out=(st_y, 0))
        else:
            ops.swin_attn(x, pa, table, att, B, H, W, shift, (stats, 2), False)
            ops.tc_gemm(att, heads * hdp, pp, y, res=x, stats_out=(st_y, 0))

    def separate():
        ops.tc_gemm(x, C, pq, qkv, stats_in=(stats, 2))
        ops.window_attention(qkv, att, table, B, H, W, 8, shift, heads, hd, hdp)
        ops.tc_gemm(att, heads * hdp, pp, y, res=x, stats_out=(st_y, 0))

    def attn_only():
        ops.swin_attn(x, pa, table, att, B, H, W, shift, (stats, 2), False)

    def proj_only():
        ops.tc_gemm(att, heads * hdp, pp, y, res=x, stats_out=(st_y, 0))

    bf, af = timeit(fused)
    bs, as_ = timeit(separate)
    line = (f"attn half C={C} heads={heads} hd={hd:3d} shift={shift} mode={mode}: fused {bf*1e3:7.1f} us (avg {af*1e3:7.1f}) "
            f"{fl/bf/1e9:6.1f} TFLOP/s   separate {bs*1e3:7.1f} us")
    fa = 2.0 * M * C * 3 * C + 4.0 * M * 64 * C
    ba, _ = timeit(attn_only)
    line += f"   | attn-only {ba*1e3:7.1f} us {fa/ba/1e9:6.1f} TF"
    bp, _ = timeit(proj_only)
    line += f"   proj GEMM {bp*1e3:6.1f} us"
    print(line)
