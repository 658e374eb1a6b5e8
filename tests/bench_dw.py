"""Depthwise micro-benchmark (not a test): CUDA-graph timed launches of the depthwise shapes of the
Xception-SPNet step, rotating over enough buffers that every launch reads cold data (> 126 MB L2).
Usage: python tests/bench_dw.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from spnet_b200 import ops
dev = torch.device("cuda:0")
SHAPES = [("b2s1", 64, 93, 125, 64), ("b2s2", 64, 93, 125, 128), ("b3s2", 64, 47, 63, 256), ("b4s2", 64, 24, 32, 728),
          ("mid", 64, 12, 16, 728), ("b14s2", 64, 6, 8, 1536)]
for name, B, H, W, C in SHAPES:
    nbytes = B * H * W * C * 2
    nbuf = max(2, int(400e6 // (3 * nbytes)) + 1)
    xs = [torch.randn(B, H, W, C, device=dev).to(torch.bfloat16) for _ in range(nbuf)]
    gs = [torch.randn(B, H, W, C, device=dev).to(torch.bfloat16) for _ in range(nbuf)]
    os_ = [torch.empty(B, H, W, C, device=dev, dtype=torch.bfloat16) for _ in range(nbuf)]
    k = torch.randn(3, 3, C, device=dev) * 0.3
    dk = torch.zeros(3, 3, C, device=dev)
    a = torch.rand(C, device=dev) + 0.5
    b = torch.randn(C, device=dev) * 0.2
    mean = torch.randn(C, device=dev) * 0.1
    rstd = torch.rand(C, device=dev) + 0.5
    stats = torch.zeros(2 * C, device=dev, dtype=torch.float64)
    res = []
    for kind in ("fwd", "bwd", "bwd+add"):
        def run(i):
            if kind == "fwd":
                ops.dwconv3x3_fwd(xs[i], k, a, b, True, out=os_[i])
            elif kind == "bwd":
                ops.dwconv3x3_bwd_fused(gs[i], xs[i], k, dk, in_a=a, in_b=b, relu=True, bn_mean=mean, bn_rstd=rstd,
                                        stats=stats, out=os_[i])
            else:
                ops.dwconv3x3_bwd_fused(gs[i], xs[i], k, dk, relu=True, add_src=xs[(i + 1) % nbuf], out=os_[i])
        try:
            run(0); torch.cuda.synchronize()
            reps = max(nbuf, 12)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for r in range(reps):
                    run(r % nbuf)
            g.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); g.replay(); e1.record(); torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / (2 * reps)
            passes = {"fwd": 2, "bwd": 3, "bwd+add": 4}[kind]
            res.append("%s %6.1f us %5.0f GB/s" % (kind, us, passes * nbytes / us / 1e3))
        except Exception as e:
            res.append("%s failed: %s" % (kind, str(e)[:60]))
    print("%-6s  %s" % (name, "  |  ".join(res)), flush=True)
