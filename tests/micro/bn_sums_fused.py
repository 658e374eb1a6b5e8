"""Times the BatchNorm-backward sums of the Xception step (384x512, batch 64, bf16) at every site where the kernel
that writes the gradient also accumulates them: the old route (producer, then bn_bwd_reduce over (gin, z)) against
the fused producer (depthwise backward with `zo`, max-pool backward with `z`).

Each route is captured as a CUDA graph over input sets rotated through more than twice the 126 MB L2, and timed
with CUDA events over several replays. Prints one line per site, and writes the figures as JSON to argv[1] if
given."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch  # noqa: E402
from spnet_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
BT = torch.bfloat16
B = 64
# (site, H, W, C, epilogue, relu on load, masked): the depthwise backward of each block's first sepconv
DW_SITES = [
    ("block2_sepconv1 -> block1_conv2_bn (masked)", 93, 125, 64, "strided", 0, True),
    ("block3_sepconv1 -> block2 residual bn", 47, 63, 128, "strided", 1, False),
    ("block4_sepconv1 -> block3 residual bn", 24, 32, 256, "strided", 1, False),
    ("block5..12_sepconv1 -> sepconv3 bn / block4 residual bn", 12, 16, 728, "src", 1, False),
    ("block13_sepconv1 -> block12_sepconv3_bn", 12, 16, 728, "strided", 1, False),
    ("block14_sepconv1 -> block13 residual bn", 6, 8, 1024, "none", 0, False),
]
POOL_SITES = [("block%d max-pool -> block%d_sepconv2_bn" % (b, b), H, W, C)
              for b, (H, W, C) in zip((2, 3, 4, 13), ((93, 125, 128), (47, 63, 256), (24, 32, 728), (12, 16, 1024)))]


def nrot_for(nbytes):
    return max(2, int(300e6 // nbytes) + 1)


def time_graph(fn, nrot, reps=10):
    for i in range(nrot):  # warm-up: first launches configure the kernels
        fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(nrot):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * nrot)


def bench_dw(site, H, W, C, epi, relu, masked):
    shape = (B, H, W, C)
    n = B * H * W * C
    nrot = nrot_for(5 * n * 2)
    rnd = lambda *s: torch.randn(*s, device=dev).to(BT)  # noqa: E731
    gs, xs, zs, outs = ([rnd(*shape) for _ in range(nrot)] for _ in range(4))
    adds = [rnd(*shape) for _ in range(nrot)] if epi == "src" else [None] * nrot
    sadds = [rnd(B, (H + 1) // 2, (W + 1) // 2, C) for _ in range(nrot)] if epi == "strided" else [None] * nrot
    k = torch.randn(3, 3, C, device=dev) * 0.3
    dk = torch.zeros(3, 3, C, device=dev)
    mean, rstd = torch.randn(C, device=dev) * 0.1, torch.rand(C, device=dev) + 0.5
    ma, mb = (torch.randn(C, device=dev), torch.randn(C, device=dev)) if masked else (None, None)
    st = ops.stats_alloc(2 * C, dev)

    def old(i):
        ops.dwconv3x3_bwd_fused(gs[i], xs[i], k, dk, relu=relu, add_src=adds[i], add_strided=sadds[i], out=outs[i])
        ops.bn_bwd_reduce(outs[i], zs[i], mean, rstd, st, relu_a=ma, relu_b=mb, act=1)

    def new(i):
        ops.dwconv3x3_bwd_fused(gs[i], xs[i], k, dk, relu=relu, add_src=adds[i], add_strided=sadds[i], out=outs[i],
                                zo=zs[i], zo_mean=mean, zo_rstd=rstd, zo_stats=st, mask_a=ma, mask_b=mb)

    def producer(i):
        ops.dwconv3x3_bwd_fused(gs[i], xs[i], k, dk, relu=relu, add_src=adds[i], add_strided=sadds[i], out=outs[i])

    return {"producer_us": time_graph(producer, nrot), "old_us": time_graph(old, nrot), "new_us": time_graph(new, nrot)}


def bench_pool(site, H, W, C):
    OH, OW = (H + 1) // 2, (W + 1) // 2
    nrot = nrot_for(B * H * W * C * 2 * 2 + B * OH * OW * C * 3)
    zs = [torch.randn(B, H, W, C, device=dev).to(BT) for _ in range(nrot)]
    gs = [torch.randn(B, OH, OW, C, device=dev).to(BT) for _ in range(nrot)]
    ams = [torch.empty(B, OH, OW, C, device=dev, dtype=torch.uint8) for _ in range(nrot)]
    outs = [torch.empty(B, H, W, C, device=dev, dtype=BT) for _ in range(nrot)]
    a, b = torch.randn(C, device=dev), torch.randn(C, device=dev) * 0.2
    for i in range(nrot):
        ops.maxpool3s2_add_fwd(zs[i], a, b, argmax=ams[i])
    mean, rstd = torch.randn(C, device=dev) * 0.1, torch.rand(C, device=dev) + 0.5
    st = ops.stats_alloc(2 * C, dev)

    def producer(i):
        ops.maxpool3s2_bwd(gs[i], ams[i], H, W, out=outs[i])

    def old(i):
        producer(i)
        ops.bn_bwd_reduce(outs[i], zs[i], mean, rstd, st)

    def new(i):
        ops.maxpool3s2_bwd(gs[i], ams[i], H, W, out=outs[i], z=zs[i], mean=mean, rstd=rstd, stats=st)

    return {"producer_us": time_graph(producer, nrot), "old_us": time_graph(old, nrot), "new_us": time_graph(new, nrot)}


def main():
    rows = []
    for s in DW_SITES:
        r = dict(site=s[0], kernel="dw3x3_bwd", shape=[B] + list(s[1:4]), **bench_dw(*s))
        rows.append(r)
    for s in POOL_SITES:
        r = dict(site=s[0], kernel="maxpool3s2_bwd", shape=[B] + list(s[1:4]), **bench_pool(*s))
        rows.append(r)
    print("%-48s %-22s %10s %10s %10s %9s" % ("site", "shape", "producer", "old", "new", "saved"))
    for r in rows:
        print("%-48s %-22s %8.1fus %8.1fus %8.1fus %7.1fus" % (r["site"], "x".join(map(str, r["shape"])), r["producer_us"],
                                                             r["old_us"], r["new_us"], r["old_us"] - r["new_us"]))
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump({"device": torch.cuda.get_device_name(0), "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
