"""Profiling driver (not a test): the round-2 kernels at the bench shapes, two launches each.
   ncu --set full --clock-control none --import-source on -k regex:'gemm_tc_kernel|ellipse_iou_exact|bn3_bwd_dz|stem_out_fwd|normalize_u8|assign_grid|yolo_ellipse_loss_ann|slab_reduce|acc_to_f32' \
       -o gpurun_out/r2_kernels python tests/micro/r2_kernels.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, torch
from spnet_b200 import ops, utils
dev = torch.device("cuda:0")
torch.manual_seed(0)
B, rows, C, n = 64, 64 * 12 * 16, 728, 24
# (1) the batched middle-flow weight gradient: 24 GEMMs [728 x 12288] x [12288 x 728] stacked along K, one launch
T = (torch.randn(n, rows, C, device=dev) * 0.5).to(torch.bfloat16)
G = (torch.randn(n, rows, C, device=dev) * 0.5).to(torch.bfloat16)
stride = C * (C + 11)
buf = torch.zeros(n * stride, device=dev)
for _ in range(2):
    ops.gemm(T.view(n * rows, C), True, G.view(n * rows, C), True, buf, C, C, n * rows, out_mode=ops.OUT_SLAB, splits=n,
             lda=C, ldb=C, ldd=C, slab_stride=stride)
# (2) Dense head forward: fixed-order split-K (slabs) + slab_reduce
F = 6 * 8 * 2048
feat = torch.randn(B, F, device=dev).to(torch.bfloat16)
Wh = (torch.randn(F, 576, device=dev) * 0.01).to(torch.bfloat16)
slabs = torch.zeros(59, B, 576, device=dev)
y = torch.empty(B, 576, device=dev)
bias = torch.zeros(576, device=dev)
for _ in range(2):
    ops.gemm(feat, False, Wh, True, slabs, B, 576, F, out_mode=ops.OUT_SLAB, splits=59)
    ops.slab_reduce(slabs, 59, B, 576, y, bias=bias)
# (3) exact IoU raster: 256 images x 72 slots, ~4 ellipses per image
rng = np.random.default_rng(0)
N = 256
P = np.zeros((N, 576), np.float32); P[:, 6::8] = 1.0
Tt = P.copy()
for i in range(N):
    for s in rng.choice(72, 4, replace=False):
        th = rng.uniform(0, 2 * np.pi)
        Tt[i, s * 8:(s + 1) * 8] = [rng.uniform(60, 450), rng.uniform(60, 320), rng.uniform(20, 140), rng.uniform(15, 100), np.cos(th), np.sin(th), 0, 3]
        P[i, s * 8:(s + 1) * 8] = Tt[i, s * 8:(s + 1) * 8] + rng.normal(0, 3, 8).astype(np.float32) * [1, 1, 1, 1, 0.02, 0.02, 0, 0.1]
Pd, Td = torch.from_numpy(P).to(dev), torch.from_numpy(Tt).to(dev)
for _ in range(2):
    ops.ellipse_iou(Pd, Td)
# (4) 3-channel stem passes (vectorised), uint8 normalisation, device grid assignment, fused annotation loss
px = 64 * 192 * 256
g3 = torch.randn(px * 3, device=dev).to(torch.bfloat16); z3 = torch.randn(px * 3, device=dev).to(torch.bfloat16)
one = torch.ones(3, device=dev); zero = torch.zeros(3, device=dev)
lib = __import__("spnet_b200._lib", fromlist=["lib"]).lib()
s_ = torch.cuda.current_stream().cuda_stream
xu = torch.randint(0, 256, (64, 384, 512, 1), device=dev, dtype=torch.uint8)
lists = [[[100.0 + 60 * k, 80.0 + 50 * k, 40, 20, 1, 0, 0, 3] for k in range(5)] for _ in range(4096)]
ann, cnt = utils.pack_annotations(lists)
d_, m_, r_ = utils.grid_tables([6, 6, 2, 8], dev)
ann_d, cnt_d = torch.from_numpy(ann).to(dev), torch.from_numpy(cnt).to(dev)
yp = torch.randn(64, 576, device=dev)
for _ in range(2):
    lib.bn3_bwd_dz(g3.data_ptr(), z3.data_ptr(), one.data_ptr(), zero.data_ptr(), one.data_ptr(), zero.data_ptr(), zero.data_ptr(),
                   g3.data_ptr(), 1, px, s_)
    ops.normalize_u8(xu)
    ops.assign_grid(ann_d, cnt_d, d_, m_, r_)
    ops.yolo_ellipse_loss_ann(ann_d[:64].contiguous(), cnt_d[:64].contiguous(), d_, m_, r_, yp, grad=torch.empty_like(yp))
torch.cuda.synchronize()
print("done")
