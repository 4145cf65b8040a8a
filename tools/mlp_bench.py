"""Timing of the fused Swin MLP kernel per DRCT block shape (CUDA events, L2 flushed), next to the unfused GEMM pair."""
import importlib, sys, os
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PKG = "anomaly-detection-super-resolution_b200"
ops = importlib.import_module(PKG + ".ops"); pack = importlib.import_module(PKG + ".pack")
dev = "cuda"
M = int(os.environ.get("M", 262144))
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

shapes = [(180, 360), (212, 424), (244, 488), (276, 276), (308, 308)]
if os.environ.get('MLP_ONLY'):
    shapes = [s for s in shapes if s[0] == int(os.environ['MLP_ONLY'])]
for (C, H) in shapes:
    y = torch.randn(M, 320, device=dev).to(torch.bfloat16); z = torch.empty_like(y)
    pm = pack.pack_swin_mlp(torch.randn(H, C, device=dev) * 0.05, torch.randn(H, device=dev), torch.ones(C, device=dev),
                            torch.zeros(C, device=dev), 1e-5, torch.randn(C, H, device=dev) * 0.05, torch.randn(C, device=dev))
    stats = torch.zeros(M, 2, 2, device=dev)
    yf = y[:, :C].float(); stats[:, 0, 0] = yf.sum(1); stats[:, 0, 1] = (yf * yf).sum(1)
    best, avg = timeit(lambda: ops.swin_mlp(y, C, pm, z, stats_in=(stats, 2)))
    fl = 4.0 * M * C * H
    print(f"swin_mlp C={C} H={H}: {best*1e3:8.1f} us (avg {avg*1e3:8.1f})  {fl/best/1e9:7.1f} TFLOP/s  {4.0*M*C/best/1e6:7.1f} GB/s(y+z)")
    # the same with the RDG's adjust 1x1 conv fused in (z never written) next to MLP + separate adjust GEMM
    if C == 308:                    # adjust5 (308 -> 180) + the RDG residual folded in, next to plain MLP + the row-tile GEMM it replaces
        wa5, ba5 = torch.randn(180, C, device=dev) * 0.05, torch.randn(180, device=dev)
        pm5 = pack.pack_swin_mlp_conv_res(torch.randn(H, C, device=dev) * 0.05, torch.randn(H, device=dev), torch.ones(C, device=dev),
                                          torch.zeros(C, device=dev), 1e-5, torch.randn(C, H, device=dev) * 0.05, torch.randn(C, device=dev), wa5, ba5, 0.2)
        slab5 = torch.randn(M, 320, device=dev).to(torch.bfloat16); st5 = torch.zeros(M, 12, 2, device=dev)
        b5, a5 = timeit(lambda: ops.swin_mlp_conv_res(y, C, pm5, slab5, slab5, stats_in=(stats, 2), stats_out=(st5, 0)))
        padj5 = pack.pack_gemm_weight(wa5, ba5, rows_kernel=True)
        def sep5():
            ops.swin_mlp(y, C, pm, z, stats_in=(stats, 2))
            ops.tc_gemm(z, C, padj5, slab5, alpha=0.2, res=slab5, stats_out=(st5, 0))
        bs5, _ = timeit(sep5)
        print(f"   + adjust5 and residual folded in: {b5*1e3:8.1f} us (avg {a5*1e3:8.1f})   separate MLP + adjust5 GEMM {bs5*1e3:8.1f} us   plan {pm5.plan.tolist()[:14]}")
    if C + 32 > 320: continue      # adjust5 is not a 32-channel conv
    wa, ba = torch.randn(32, C, device=dev) * 0.05, torch.randn(32, device=dev)
    margs = (torch.randn(H, C, device=dev) * 0.05, torch.randn(H, device=dev), torch.ones(C, device=dev),
             torch.zeros(C, device=dev), 1e-5, torch.randn(C, H, device=dev) * 0.05, torch.randn(C, device=dev), wa, ba)
    slab = torch.zeros(M, 320, device=dev, dtype=torch.bfloat16); st_s = torch.zeros(M, 12, 2, device=dev)
    pma = pack.pack_swin_mlp(*margs)
    padj = pack.pack_gemm_weight(wa, ba)
    bf, af = timeit(lambda: ops.swin_mlp_adjust(y, C, pma, slab, C, stats_in=(stats, 2), stats_out=(st_s, 2)))
    def sep():
        ops.swin_mlp(y, C, pm, z, stats_in=(stats, 2))
        ops.tc_gemm(z, C, padj, slab, act=ops.ACT_LRELU, slope=0.2, ocol0=C, n_store=32, stats_out=(st_s, 2))
    bs, _ = timeit(sep)
    print(f"   + adjust folded into fc2: {bf*1e3:8.1f} us (avg {af*1e3:8.1f})   separate MLP + adjust GEMM {bs*1e3:8.1f} us   plan {pma.plan.tolist()[:14]}")
