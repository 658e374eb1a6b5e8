"""Times the stem / block-1 small-channel convolutions at the bench shape (B=64, 192x256x3 after the folded
average pool)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from spnet_b200 import ops
dev = "cuda"
B, H, W = 64, 192, 256
bf = torch.bfloat16
x0 = torch.rand(B, 2 * H, 2 * W, 1, device=dev) * 2 - 1
x = torch.randn(B, H, W, 3, device=dev).to(bf)
y = torch.empty_like(x)
g = torch.randn(B, H, W, 3, device=dev).to(bf)
gin = torch.empty_like(x)
w33 = torch.randn(3, 3, 3, 3, device=dev) * 0.2
k4 = torch.randn(4, 4, 1, 3, device=dev) * 0.2
a = torch.rand(3, device=dev) + 0.5
b = torch.randn(3, device=dev) * 0.1
st = ops.stats_alloc(6, dev)
dw = torch.zeros(3, 3, 3, 3, device=dev)
dk4 = torch.zeros(4, 4, 1, 3, device=dev)
skip = torch.empty(B, H, W, 1, device=dev, dtype=bf)
OH1, OW1 = (H - 3) // 2 + 1, (W - 3) // 2 + 1
w32 = torch.randn(3, 3, 3, 32, device=dev) * 0.2
z11 = torch.empty(B, OH1, OW1, 32, device=dev, dtype=bf)
g11 = torch.randn(B, OH1, OW1, 32, device=dev).to(bf)
st32 = ops.stats_alloc(64, dev)
dw32 = torch.zeros(3, 3, 3, 32, device=dev)
flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)

cases = [
    ("stem conv1 4x4s2 1->3 fwd", lambda: ops.conv_small_fwd(0, x0, k4, y, skip=skip, stats=st)),
    ("stem conv 3->3 fwd", lambda: ops.conv_small_fwd(1, x, w33, y, in_a=a, in_b=b, act=2, stats=st)),
    ("stem conv 3->3 dgrad", lambda: ops.conv_small_dgrad(1, g, w33, gin, mask_z=x, mask_a=a, mask_b=b, act=2)),
    ("stem conv 3->3 wgrad", lambda: ops.conv_small_wgrad(1, x, g, dw, in_a=a, in_b=b, act=2)),
    ("stem conv1 wgrad", lambda: ops.conv_small_wgrad(0, x0, g, dk4)),
    ("block1_conv1 fwd", lambda: ops.conv_small_fwd(2, x, w32, z11, stats=st32)),
    ("block1_conv1 dgrad", lambda: ops.conv_small_dgrad(2, g11, w32, gin)),
    ("block1_conv1 wgrad", lambda: ops.conv_small_wgrad(2, x, g11, dw32)),
]
for name, fn in cases:
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(10):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    print("%-28s %7.1f us (median of 10, cold L2)" % (name, ts[len(ts) // 2]), flush=True)
