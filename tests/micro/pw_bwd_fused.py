"""Times the backward of Xception's block-2 pointwise convolutions and their BatchNorm (384x512, batch 64, bf16): the
unfused route (bn_bwd_dz, then the weight-gradient and data-gradient GEMMs) against ops.pw_bwd_bn, which keeps dz on
chip. Also times the block-3 sites (128 -> 256), which keep the unfused route.

Each route is captured as a CUDA graph over input sets rotated through more than twice the 126 MB L2, and timed with
CUDA events over several replays. The bandwidth column is the route's algorithmic traffic (unfused: 5 passes over the
[M, cout] tensors and 2 over [M, cin]; fused: 2 and 2) over its time. Prints one line per site, and writes the figures
as JSON to argv[1] if given."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch  # noqa: E402
from spnet_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
BT = torch.bfloat16
# (site, M, cin, cout) at batch 64, 384x512
SITES = [("block2_sepconv1", 64 * 93 * 125, 64, 128), ("block2_sepconv2", 64 * 93 * 125, 128, 128),
         ("conv2d_4 (block 2 residual)", 64 * 47 * 63, 64, 128), ("block3_sepconv1", 64 * 47 * 63, 128, 256),
         ("conv2d_5 (block 3 residual)", 64 * 24 * 32, 128, 256)]


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


def bench(M, cin, cout):
    p_out, p_in = M * cout * 2, M * cin * 2
    nrot = max(2, int(300e6 // (3 * p_out + 2 * p_in)) + 1)
    gs = [torch.randn(M, cout, device=dev).to(BT) for _ in range(nrot)]
    zs = [torch.randn(M, cout, device=dev).to(BT) for _ in range(nrot)]
    ts = [torch.randn(M, cin, device=dev).to(BT) for _ in range(nrot)]
    gas = [torch.empty(M, cin, device=dev, dtype=BT) for _ in range(nrot)]
    dz = torch.empty(M, cout, device=dev, dtype=BT)
    W = (torch.randn(cin, cout, device=dev) * 0.1).to(BT)
    gW = torch.zeros(cin, cout, device=dev)
    a, mean = torch.randn(cout, device=dev), torch.randn(cout, device=dev) * 0.1
    rstd, c1, c2 = torch.rand(cout, device=dev) + 0.5, torch.randn(cout, device=dev) * 0.1, torch.randn(cout, device=dev) * 0.1

    def old(i):
        ops.bn_bwd_dz(gs[i], zs[i], a, mean, rstd, c1, c2, out=dz)
        ops.gemm(ts[i], True, dz, True, gW, cin, cout, M, out_mode=ops.OUT_ATOMIC, splits=0, lda=cin, ldb=cout)
        ops.gemm(dz, False, W, False, gas[i], M, cin, cout, out_mode=ops.OUT_T, ldb=cout)

    def new(i):
        ops.pw_bwd_bn(gs[i], zs[i], ts[i], W, a, mean, rstd, c1, c2, gas[i], gW, M, cin, cout)

    r = {"old_us": time_graph(old, nrot), "old_bytes": 5 * p_out + 2 * p_in, "fused_bytes": 2 * p_out + 2 * p_in}
    if cout == 128:
        r["new_us"] = time_graph(new, nrot)
    return r


def main():
    rows = []
    for site, M, cin, cout in SITES:
        rows.append(dict(site=site, M=M, cin=cin, cout=cout, **bench(M, cin, cout)))
    print("%-30s %8s %8s %10s %10s %10s %10s %8s" % ("site", "M", "cin>cout", "old", "old GB/s", "new", "new GB/s", "saved"))
    for r in rows:
        old_bw = r["old_bytes"] / r["old_us"] / 1e3
        if "new_us" in r:
            print("%-30s %8d %8s %8.1fus %10.0f %8.1fus %10.0f %6.1fus" % (
                r["site"], r["M"], "%d>%d" % (r["cin"], r["cout"]), r["old_us"], old_bw, r["new_us"],
                r["fused_bytes"] / r["new_us"] / 1e3, r["old_us"] - r["new_us"]))
        else:
            print("%-30s %8d %8s %8.1fus %10.0f %10s %10s %8s" % (r["site"], r["M"], "%d>%d" % (r["cin"], r["cout"]),
                                                                r["old_us"], old_bw, "-", "-", "-"))
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump({"device": torch.cuda.get_device_name(0), "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
