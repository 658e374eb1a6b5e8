"""Kernel-level parity: every C-ABI kernel against a plain fp32 PyTorch / numpy statement of
the same op on the same seeded inputs (torch is the checker here, never the thing tested)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import numpy_side as ns  # noqa: E402


def _ops():
    from spnet_b200 import ops
    return ops


def dev():
    return torch.device("cuda:0")


def tol(dtype):
    return dict(rtol=2e-2, atol=2e-2) if dtype == torch.bfloat16 else dict(rtol=1e-4, atol=1e-5)


def nchw(x):
    return x.float().permute(0, 3, 1, 2).contiguous()


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def dw_ref(x, k, a=None, b=None, relu=False):
    """x NHWC (any dtype), k [3,3,C] -> NHWC fp32."""
    v = x.float()
    if a is not None:
        v = v * a + b
    if relu == 2:
        v = torch.clamp(v, 0.0, 6.0)
    elif relu:
        v = torch.relu(v)
    C = x.shape[-1]
    w = k.permute(2, 0, 1).reshape(C, 1, 3, 3)
    return nhwc(F.conv2d(nchw(v), w, padding=1, groups=C))


# ------------------------------------------------------------------ loss
@pytest.mark.parametrize("loss_type", ["same", "hybrid"])
@pytest.mark.parametrize("B", [1, 7, 64])
def test_loss_matches_my_loss(loss_type, B):
    ops = _ops()
    rng = np.random.default_rng(B)
    yt = rng.standard_normal((B, 576)).astype(np.float32) * 0.3
    yt[:, 6::8] = (rng.random((B, 72)) > 0.7).astype(np.float32)
    yp = yt + rng.standard_normal((B, 576)).astype(np.float32) * 0.2
    total, parts = ns.my_loss(yt.astype(np.float64), yp.astype(np.float64), loss_type)
    gref = ns.my_loss_grad(yt.astype(np.float64), yp.astype(np.float64), loss_type)
    grad = torch.empty(B, 576, device=dev())
    out = ops.yolo_ellipse_loss(torch.tensor(yt, device=dev()), torch.tensor(yp, device=dev()),
                                hybrid=(loss_type != "same"), grad=grad).cpu().numpy()
    np.testing.assert_allclose(out[0], total, rtol=2e-6)
    np.testing.assert_allclose(out[1:], parts, rtol=2e-6, atol=1e-9)
    np.testing.assert_allclose(grad.cpu().numpy(), gref, rtol=2e-5, atol=1e-9)


def test_selective_sigmoid_and_loss_chain():
    ops = _ops()
    rng = np.random.default_rng(0)
    x = (rng.random((2, 16)) - 0.5).astype(np.float32)
    y = ops.selective_sigmoid_fwd(torch.tensor(x, device=dev()), 6, None, 8).cpu().numpy()
    changed = np.argwhere(np.abs(y - x) > 1e-6)
    assert sorted(set(changed[:, 1].tolist())) == [6, 14]  # reference tests/test_selectivesigmoid.py
    np.testing.assert_allclose(y, ns.selective_sigmoid(x), rtol=1e-6)
    dy = rng.standard_normal((2, 16)).astype(np.float32)
    dx = ops.selective_sigmoid_bwd(torch.tensor(y, device=dev()), torch.tensor(dy, device=dev()), 6, None, 8).cpu().numpy()
    ref = dy.copy()
    ref[:, 6::8] *= y[:, 6::8] * (1 - y[:, 6::8])
    np.testing.assert_allclose(dx, ref, rtol=1e-6)
    # fused: loss(sel_sigmoid=True) == loss on sigmoid'ed predictions, gradient chained
    yt = rng.standard_normal((5, 576)).astype(np.float32)
    yt[:, 6::8] = (rng.random((5, 72)) > 0.5)
    raw = rng.standard_normal((5, 576)).astype(np.float32)
    total, _ = ns.my_loss(yt.astype(np.float64), ns.selective_sigmoid(raw.astype(np.float64)))
    g = ns.my_loss_grad(yt.astype(np.float64), ns.selective_sigmoid(raw.astype(np.float64)))
    s = ns.selective_sigmoid(raw.astype(np.float64))[:, 6::8]
    g[:, 6::8] *= s * (1 - s)
    grad = torch.empty(5, 576, device=dev())
    out = ops.yolo_ellipse_loss(torch.tensor(yt, device=dev()), torch.tensor(raw, device=dev()), sel_sigmoid=True,
                                grad=grad).cpu().numpy()
    np.testing.assert_allclose(out[0], total, rtol=3e-6)
    np.testing.assert_allclose(grad.cpu().numpy(), g, rtol=3e-5, atol=1e-9)


def test_decode_matches_numpy():
    ops = _ops()
    rng = np.random.default_rng(3)
    means, ranges = ns.setup_means_and_ranges([6, 6, 2, 8])[7:9]
    y = (rng.standard_normal((9, 576)) * 0.4).astype(np.float32)
    y[:, 6::8] = rng.random((9, 72)).astype(np.float32)
    y[0, 2::8] = 0.5 / 71  # rounding ties
    denorm, ints, exists = ops.decode_detections(torch.tensor(y, device=dev()), torch.tensor(means, device=dev()),
                                                 torch.tensor(ranges, device=dev()))
    ref = ns.denorm_Y(y, means, ranges)
    assert ref.dtype == np.float32
    np.testing.assert_array_equal(denorm.cpu().numpy(), ref)  # bit-exact
    ints = ints.cpu().numpy()
    exists = exists.cpu().numpy()
    for j in range(9):
        for an in range(72):
            cx, cy, a, b, angle, noobj, rings = ns.cleanup_antinode_vars(ref[j, an * 8:(an + 1) * 8])
            assert tuple(ints[j, an]) == (cx, cy, a, b, noobj)
            assert bool(exists[j, an]) == (noobj == 0 and rings > 0 and a >= 0 and b >= 0)


# ------------------------------------------------------------------ depthwise
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(2, 12, 16, 728), (3, 47, 63, 128), (1, 6, 8, 2048), (2, 5, 5, 40), (1, 93, 125, 64)])
@pytest.mark.parametrize("mode", ["plain", "relu", "affine_relu", "affine", "affine_relu6"])
def test_dwconv_fwd(dtype, shape, mode):
    ops = _ops()
    torch.manual_seed(1)
    B, H, W, C = shape
    x = (torch.randn(shape, device=dev()) * (5.0 if mode == "affine_relu6" else 1.0)).to(dtype)
    k = torch.randn(3, 3, C, device=dev()) * 0.3
    a = b = None
    if mode in ("affine_relu", "affine", "affine_relu6"):
        a = torch.rand(C, device=dev()) + 0.5
        b = torch.randn(C, device=dev()) * 0.2 + 0.3  # a non-zero shift makes the padding order visible
    relu = 2 if mode == "affine_relu6" else mode in ("relu", "affine_relu")
    out = ops.dwconv3x3_fwd(x, k, a, b, relu)
    ref = dw_ref(x, k, a, b, relu)
    torch.testing.assert_close(out.float(), ref, **tol(dtype))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(2, 12, 16, 728), (2, 47, 63, 128), (2, 7, 9, 24), (1, 93, 125, 64), (3, 6, 8, 1024), (2, 24, 32, 256)])
@pytest.mark.parametrize("mode", ["bn_relu", "relu_add", "plain_strided", "bn_relu6"])
def test_dwconv_bwd_fused(dtype, shape, mode):
    """Fused dgrad + wgrad + ReLU mask + BatchNorm-backward sums against autograd."""
    ops = _ops()
    torch.manual_seed(4)
    B, H, W, C = shape
    x = (torch.randn(shape, device=dev()) * (5.0 if mode == "bn_relu6" else 1.0)).to(dtype)
    k = torch.randn(3, 3, C, device=dev()) * 0.3
    g = torch.randn(shape, device=dev()).to(dtype)
    a = b = mean = rstd = stats = add = sadd = None
    relu = 2 if mode == "bn_relu6" else mode != "plain_strided"
    if mode in ("bn_relu", "bn_relu6"):
        a = torch.rand(C, device=dev()) + 0.5
        b = torch.randn(C, device=dev()) * 0.2
        mean = torch.randn(C, device=dev()) * 0.1
        rstd = torch.rand(C, device=dev()) + 0.5
        stats = ops.stats_alloc(2 * C, dev())
    elif mode == "relu_add":
        add = torch.randn(shape, device=dev()).to(dtype)
    else:
        sadd = torch.randn(B, (H + 1) // 2, (W + 1) // 2, C, device=dev()).to(dtype)
    pre = x.float() * a + b if a is not None else x.float()
    v = (torch.clamp(pre, 0.0, 6.0) if relu == 2 else (torch.relu(pre) if relu else pre)).detach().requires_grad_(True)
    kr = k.clone().requires_grad_(True)
    y = nhwc(F.conv2d(nchw(v), kr.permute(2, 0, 1).reshape(C, 1, 3, 3), padding=1, groups=C))
    y.backward(g.float())
    ref = v.grad * ((pre > 0) & (pre < 6)) if relu == 2 else (v.grad * (pre > 0) if relu else v.grad.clone())
    dk = torch.zeros(3, 3, C, device=dev())
    gin = ops.dwconv3x3_bwd_fused(g, x, k, dk, in_a=a, in_b=b, relu=relu, bn_mean=mean, bn_rstd=rstd, stats=stats,
                                  add_src=add, add_strided=sadd)
    if stats is not None:
        gq = gin.double()
        xh = (x.double() - mean.double()) * rstd.double()
        sv = ops.stats_values(stats).to(gq.device)
        torch.testing.assert_close(sv[:C], gq.sum((0, 1, 2)), rtol=1e-4, atol=1e-3)
        torch.testing.assert_close(sv[C:], (gq * xh).sum((0, 1, 2)), rtol=1e-4, atol=1e-3)
    if add is not None:
        ref = ref + add.float()
    if sadd is not None:
        ref[:, ::2, ::2, :] += sadd.float()
    torch.testing.assert_close(gin.float(), ref, **tol(dtype))
    scale = float(kr.grad.abs().max())
    t = dict(rtol=2e-2, atol=2e-2 * scale) if dtype == torch.bfloat16 else dict(rtol=2e-4, atol=2e-4 * scale)
    torch.testing.assert_close(dk, kr.grad, **t)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("off", [(0, 0), (1, 1), (0, 1), (1, 0)])
def test_subsample_scatter_colstats(dtype, off):
    ops = _ops()
    torch.manual_seed(6)
    B, H, W, C = 2, 12 + (1 - off[0]), 16 + (1 - off[1]), 72  # odd sizes go with offset 0
    x = torch.randn(B, H, W, C, device=dev()).to(dtype)
    y = ops.gather_s2(x, off=off)
    torch.testing.assert_close(y, x[:, off[0]::2, off[1]::2, :].contiguous())
    back = torch.empty_like(x)
    ops.scatter_s2(y, back, off=off)
    ref = torch.zeros_like(x)
    ref[:, off[0]::2, off[1]::2, :] = y
    torch.testing.assert_close(back, ref)
    st = ops.stats_alloc(2 * C, dev())
    ops.colstats(x, st)
    sv = ops.stats_values(st).to(x.device)
    torch.testing.assert_close(sv[:C], x.double().sum((0, 1, 2)), rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(sv[C:], (x.double() ** 2).sum((0, 1, 2)), rtol=1e-5, atol=1e-4)


# ------------------------------------------------------------------ GEMM
def _gemm_case(M, N, K, a_mn, b_mn, out_mode, splits, stats, dtype):
    ops = _ops()
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device=dev())
    Bm = torch.randn(K, N, device=dev())
    A_l, B_l = A.to(dtype), Bm.to(dtype)
    ref = A_l.float() @ B_l.float()
    A_st = A_l.t().contiguous() if a_mn else A_l.contiguous()          # [K,M] or [M,K]
    B_st = B_l.contiguous() if b_mn else B_l.t().contiguous()          # [K,N] or [N,K]
    out_dtype = dtype if out_mode == ops.OUT_T else torch.float32
    D = torch.zeros(M, N, device=dev(), dtype=out_dtype)
    cs = ops.stats_alloc(2 * N, dev()) if stats else None
    ops.gemm(A_st, a_mn, B_st, b_mn, D, M, N, K, out_mode=out_mode, splits=splits, colstats=cs)
    t = dict(rtol=2e-2, atol=2e-2 * K ** 0.5) if out_dtype == torch.bfloat16 else dict(rtol=1e-3, atol=1e-3 * K ** 0.5)
    torch.testing.assert_close(D.float(), ref, **t)
    if stats:
        Dd = D.double()
        cv = ops.stats_values(cs).to(Dd.device)
        torch.testing.assert_close(cv[:N], Dd.sum(0), rtol=1e-4, atol=1e-2)
        torch.testing.assert_close(cv[N:], (Dd * Dd).sum(0), rtol=1e-4, atol=1e-2)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (False, True), (True, True), (True, False)])
@pytest.mark.parametrize("M,N,K", [(256, 128, 64), (300, 728, 728), (1000, 256, 128), (64, 576, 1024), (128, 128, 2048),
                                   (5000, 64, 128), (264, 32, 200)])
def test_gemm_store(dtype, a_mn, b_mn, M, N, K):
    if a_mn and M % 8:
        pytest.skip("MN-major A needs M % 8 == 0 (TMA 16-byte stride)")
    ops = _ops()
    _gemm_case(M, N, K, a_mn, b_mn, ops.OUT_T, 1, True, dtype)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_gemm_splitk_atomic_and_f32_store(dtype):
    ops = _ops()
    _gemm_case(64, 576, 4096, False, True, ops.OUT_ATOMIC, 7, False, dtype)
    _gemm_case(728, 728, 3000 if dtype == torch.float32 else 3072, True, True, ops.OUT_ATOMIC, 4, False, dtype)
    _gemm_case(512, 576, 64, True, True, ops.OUT_F32, 1, False, dtype)
    _gemm_case(200, 264, 72, False, False, ops.OUT_F32, 1, True, dtype)
    _gemm_case(128, 64, 4000, True, True, ops.OUT_ATOMIC, 5, False, dtype)     # 64-wide tiles, split-K
    _gemm_case(288, 64, 520, True, True, ops.OUT_F32, 1, True, dtype)


# ------------------------------------------------------------------ batch norm pieces
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_bn_train_fwd_bwd(dtype):
    ops = _ops()
    torch.manual_seed(5)
    rows, C = 1000, 728
    z = (torch.randn(rows, C, device=dev()) * 2 + 0.5).to(dtype)
    gamma = torch.rand(C, device=dev()) + 0.5
    beta = torch.randn(C, device=dev()) * 0.1
    zf = z.double()
    stats = ops.stats_from_values(torch.cat([zf.sum(0), (zf * zf).sum(0)]), dev())
    a, b, mean, rstd = (torch.empty(C, device=dev()) for _ in range(4))
    mm = torch.zeros(C, device=dev())
    mv = torch.ones(C, device=dev())
    ops.bn_finalize(stats, rows, gamma, beta, a, b, mean, rstd, mm, mv)
    assert int(stats.abs().max()) == 0
    zr = z.float().requires_grad_(True)
    gr = gamma.clone().requires_grad_(True)
    br = beta.clone().requires_grad_(True)
    y = F.batch_norm(zr, None, None, gr, br, training=True, eps=1e-3)
    out = ops.bn_apply(z, a, b, act=1)
    torch.testing.assert_close(out.float(), torch.relu(y).detach(), **tol(dtype))
    torch.testing.assert_close(mm, 0.01 * z.float().mean(0), rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(mv, 0.99 + 0.01 * z.float().var(0, unbiased=True), rtol=1e-4, atol=1e-6)
    x = torch.randn(rows, C, device=dev()).to(dtype)
    out2 = ops.bn_apply(z, a, b, act=0, x=x)
    torch.testing.assert_close(out2.float(), (y + x.float()).detach(), **tol(dtype))
    # backward through relu(bn(z))
    g = torch.randn(rows, C, device=dev()).to(dtype)
    torch.relu(y).backward(g.float())
    gy = g.clone()
    bstats = ops.stats_alloc(2 * C, dev())
    ops.bn_bwd_reduce(gy, z, mean, rstd, bstats, relu_a=a, relu_b=b, act=1)
    dgamma, dbeta, c1, c2 = (torch.empty(C, device=dev()) for _ in range(4))
    ops.bn_bwd_finalize(bstats, rows, dgamma, dbeta, c1, c2)
    gz = ops.bn_bwd_dz(gy, z, a, mean, rstd, c1, c2)
    t = dict(rtol=3e-2, atol=3e-2) if dtype == torch.bfloat16 else dict(rtol=1e-3, atol=1e-4)
    torch.testing.assert_close(gz.float(), zr.grad, **t)
    tg = dict(rtol=3e-2, atol=0.5) if dtype == torch.bfloat16 else dict(rtol=1e-3, atol=1e-3)
    torch.testing.assert_close(dgamma, gr.grad, **tg)
    torch.testing.assert_close(dbeta, br.grad, **tg)


# ------------------------------------------------------------------ pooling
def tf_same_maxpool_ref(y):
    """y NHWC fp32 -> maxpool 3x3 s2 TF-SAME via explicit -inf padding."""
    B, H, W, C = y.shape
    def pads(n):
        out = (n + 1) // 2
        tot = max((out - 1) * 2 + 3 - n, 0)
        return tot // 2, tot - tot // 2
    pt, pb = pads(H)
    pl, pr = pads(W)
    yp = F.pad(nchw(y), (pl, pr, pt, pb), value=float("-inf"))
    return nhwc(F.max_pool2d(yp, 3, 2))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(2, 24, 32, 256), (2, 93, 125, 128), (1, 47, 63, 256), (2, 12, 16, 728), (1, 5, 5, 1024)])
def test_maxpool_add_fwd_bwd(dtype, shape):
    ops = _ops()
    torch.manual_seed(7)
    B, H, W, C = shape
    z = torch.randn(shape, device=dev()).to(dtype)
    a = torch.randn(C, device=dev())  # negative scales too: affine must precede the max
    b = torch.randn(C, device=dev()) * 0.2
    OH, OW = (H + 1) // 2, (W + 1) // 2
    res = torch.randn(B, OH, OW, C, device=dev()).to(dtype)
    ra = torch.rand(C, device=dev()) + 0.5
    rb = torch.randn(C, device=dev()) * 0.2
    argmax = torch.empty(B, OH, OW, C, device=dev(), dtype=torch.uint8)
    out = ops.maxpool3s2_add_fwd(z, a, b, res, ra, rb, argmax=argmax)
    yr = (z.float() * a + b).requires_grad_(True)
    ref = tf_same_maxpool_ref(yr) + (res.float() * ra + rb)
    torch.testing.assert_close(out.float(), ref.detach(), **tol(dtype))
    g = torch.randn(B, OH, OW, C, device=dev()).to(dtype)
    ref.backward(g.float())
    gin = ops.maxpool3s2_bwd(g, argmax, H, W)
    torch.testing.assert_close(gin.float(), yr.grad, **tol(dtype))
    sub = ops.gather_s2(z)
    torch.testing.assert_close(sub, z[:, ::2, ::2, :].contiguous())


@pytest.mark.parametrize("shape", [(2, 24, 32, 64), (2, 23, 31, 64), (1, 7, 9, 128)])
def test_maxpool_bf16_exact_and_ties(shape):
    """bf16 pooling takes the maximum on the raw inputs (monotone affine): the output must equal the fp32 formula bit
    for bit, also with zero / negative scales and with many equal inputs, and the gradient must go to the FIRST
    maximum of every window (torch's rule as well)."""
    ops = _ops()
    torch.manual_seed(9)
    B, H, W, C = shape
    z = torch.randint(-3, 4, shape, device=dev()).float().bfloat16()       # seven distinct values: ties everywhere
    a = torch.randn(C, device=dev())
    a[::5] = 0.0
    b = torch.randn(C, device=dev()) * 0.2
    OH, OW = (H + 1) // 2, (W + 1) // 2
    argmax = torch.empty(B, OH, OW, C, device=dev(), dtype=torch.uint8)
    out = ops.maxpool3s2_add_fwd(z, a, b, argmax=argmax)
    yr = torch.addcmul(b, z.float(), a).requires_grad_(True)                # fma(v, a, b) like the kernel
    ref = tf_same_maxpool_ref(yr)
    assert torch.equal(out, ref.detach().bfloat16())
    g = torch.randn(B, OH, OW, C, device=dev()).bfloat16()
    ref.backward(g.float())
    gin = ops.maxpool3s2_bwd(g, argmax, H, W)
    live = (a != 0).view(1, 1, 1, C)     # a = 0: every tap is a maximum; both pick the first, but y is constant
    torch.testing.assert_close((gin.float() * live), (yr.grad * live).bfloat16().float(), rtol=1e-2, atol=1e-2)
    # gradient mass is conserved per channel whatever the tie rule
    torch.testing.assert_close(gin.float().sum((0, 1, 2)), g.float().sum((0, 1, 2)), rtol=2e-2, atol=0.3)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(2, 35, 35, 64), (1, 17, 20, 128), (2, 8, 9, 32)])
def test_maxpool_valid_fwd_bwd(dtype, shape):
    ops = _ops()
    torch.manual_seed(10)
    B, H, W, C = shape
    x = torch.randn(shape, device=dev()).to(dtype)
    OH, OW = (H - 3) // 2 + 1, (W - 3) // 2 + 1
    out = torch.empty(B, OH, OW, C, device=dev(), dtype=dtype)
    argmax = torch.empty(B, OH, OW, C, device=dev(), dtype=torch.uint8)
    ops.maxpool3s2_valid_fwd(x, out, argmax)
    xr = x.float().requires_grad_(True)
    ref = nhwc(F.max_pool2d(nchw(xr), 3, 2))
    assert torch.equal(out.float(), ref.detach())
    g = torch.randn(B, OH, OW, C, device=dev()).to(dtype)
    ref.backward(g.float())
    gin = torch.full(shape, float("nan"), device=dev(), dtype=dtype)
    ops.maxpool3s2_valid_bwd(g, argmax, gin)
    torch.testing.assert_close(gin.float(), xr.grad, **tol(dtype))


# ------------------------------------------------------------------ stem / block1
def leaky(v):
    return F.leaky_relu(v, 0.1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("hw", [(48, 64), (37, 37)])
def test_stem_and_block1_convs(dtype, hw):
    ops = _ops()
    torch.manual_seed(11)
    B, (H, W) = 2, hw
    x0 = torch.rand(B, H, W, 1, device=dev()) * 2 - 1
    k3 = torch.randn(3, 3, 1, 3, device=dev()) * 0.5
    k4 = torch.empty(4, 4, 1, 3, device=dev())
    ops.stem_k3_to_k4(k3, k4)
    H2, W2 = H // 2, W // 2
    p1 = torch.empty(B, H2, W2, 3, device=dev(), dtype=dtype)
    s0 = torch.empty(B, H2, W2, 1, device=dev(), dtype=dtype)
    st = ops.stats_alloc(6, dev())
    ops.conv_small_fwd(0, x0, k4, p1, skip=s0, stats=st)
    k3r = k3.clone().requires_grad_(True)
    conv = F.conv2d(nchw(x0), k3r.permute(3, 2, 0, 1), padding=1)
    ref_p1 = nhwc(F.avg_pool2d(conv, 2))
    ref_s0 = nhwc(F.avg_pool2d(nchw(x0), 2))
    torch.testing.assert_close(p1.float(), ref_p1.detach(), **tol(dtype))
    torch.testing.assert_close(s0.float(), ref_s0, **tol(dtype))
    torch.testing.assert_close(ops.stats_values(st).to(p1.device)[:3], p1.double().sum((0, 1, 2)), rtol=1e-5, atol=1e-3)
    torch.testing.assert_close(ops.stats_values(st).to(p1.device)[3:], (p1.double() ** 2).sum((0, 1, 2)), rtol=1e-5, atol=1e-3)
    # conv1 weight gradient through the avgpool fold
    g1 = torch.randn(B, H2, W2, 3, device=dev()).to(dtype)
    ref_p1.backward(g1.float())
    g4 = torch.zeros(4, 4, 1, 3, device=dev())
    ops.conv_small_wgrad(0, x0, g1, g4)
    g3 = torch.zeros(3, 3, 1, 3, device=dev())
    ops.stem_k4grad_to_k3grad(g4, g3)
    sc = float(k3r.grad.abs().max())
    torch.testing.assert_close(g3, k3r.grad, rtol=1e-3, atol=1e-3 * sc)

    # 3->3 conv with affine + leaky on load
    a = torch.rand(3, device=dev()) + 0.5
    b = torch.randn(3, device=dev()) * 0.3
    w33 = (torch.randn(3, 3, 3, 3, device=dev()) * 0.4)
    c2 = torch.empty(B, H2, W2, 3, device=dev(), dtype=dtype)
    st2 = ops.stats_alloc(6, dev())
    ops.conv_small_fwd(1, p1, w33, c2, in_a=a, in_b=b, act=2, stats=st2)
    pr = p1.float().requires_grad_(True)
    wr = w33.clone().requires_grad_(True)
    act_in = leaky(pr * a + b)
    act_leaf = act_in.detach().requires_grad_(True)
    ref_c2 = nhwc(F.conv2d(nchw(act_leaf), wr.permute(3, 2, 0, 1), padding=1))
    torch.testing.assert_close(c2.float(), ref_c2.detach(), **tol(dtype))
    torch.testing.assert_close(ops.stats_values(st2).to(c2.device)[:3], c2.double().sum((0, 1, 2)), rtol=1e-5, atol=1e-3)
    g2 = torch.randn(B, H2, W2, 3, device=dev()).to(dtype)
    ref_c2.backward(g2.float())
    dw = torch.zeros(3, 3, 3, 3, device=dev())
    ops.conv_small_wgrad(1, p1, g2, dw, in_a=a, in_b=b, act=2)
    sc = float(wr.grad.abs().max())
    tw = dict(rtol=2e-2, atol=2e-2 * sc) if dtype == torch.bfloat16 else dict(rtol=1e-3, atol=1e-3 * sc)
    torch.testing.assert_close(dw, wr.grad, **tw)
    gin = torch.empty(B, H2, W2, 3, device=dev(), dtype=dtype)
    ops.conv_small_dgrad(1, g2, w33, gin, mask_z=p1, mask_a=a, mask_b=b, act=2)
    pre = p1.float() * a + b
    ref_gin = act_leaf.grad * torch.where(pre > 0, torch.ones_like(pre), torch.full_like(pre, 0.1))
    torch.testing.assert_close(gin.float(), ref_gin, **tol(dtype))

    # stem output: bn3 + skip, dropout off and on
    d = torch.empty(B, H2, W2, 3, device=dev(), dtype=dtype)
    ops.stem_out_fwd(c2, a, b, s0, d)
    torch.testing.assert_close(d.float(), c2.float() * a + b + s0.float(), **tol(dtype))
    seed = torch.tensor([1234], device=dev(), dtype=torch.int64)
    dd = torch.empty_like(d)
    ops.stem_out_fwd(c2, a, b, s0, dd, rate=0.1, seed=seed)
    keep = (dd.float() != 0)
    frac = 1 - keep.float().mean().item()
    assert 0.05 < frac < 0.15
    torch.testing.assert_close(dd.float()[keep], (d.float() / 0.9)[keep], **tol(dtype))
    gd = torch.randn_like(d.float()).to(dtype)
    gdo = torch.empty_like(gd)
    ops.stem_out_bwd(gd, gdo, rate=0.1, seed=seed)
    torch.testing.assert_close(gdo.float(), torch.where(keep, gd.float() / 0.9, torch.zeros_like(gd.float())), **tol(dtype))

    # block1_conv1: 3x3 s2 valid 3->32
    w1 = torch.randn(3, 3, 3, 32, device=dev()) * 0.3
    OH, OW = (H2 - 3) // 2 + 1, (W2 - 3) // 2 + 1
    z11 = torch.empty(B, OH, OW, 32, device=dev(), dtype=dtype)
    st3 = ops.stats_alloc(64, dev())
    ops.conv_small_fwd(2, d, w1, z11, stats=st3)
    dr = d.float().requires_grad_(True)
    w1r = w1.clone().requires_grad_(True)
    ref_z = nhwc(F.conv2d(nchw(dr), w1r.permute(3, 2, 0, 1), stride=2))
    torch.testing.assert_close(z11.float(), ref_z.detach(), **tol(dtype))
    torch.testing.assert_close(ops.stats_values(st3).to(z11.device)[:32], z11.double().sum((0, 1, 2)), rtol=1e-5, atol=1e-3)
    gz = torch.randn(B, OH, OW, 32, device=dev()).to(dtype)
    ref_z.backward(gz.float())
    dw1 = torch.zeros(3, 3, 3, 32, device=dev())
    ops.conv_small_wgrad(2, d, gz, dw1)
    sc = float(w1r.grad.abs().max())
    torch.testing.assert_close(dw1, w1r.grad, rtol=2e-2 if dtype == torch.bfloat16 else 1e-3, atol=(2e-2 if dtype == torch.bfloat16 else 1e-3) * sc)
    gd1 = torch.empty(B, H2, W2, 3, device=dev(), dtype=dtype)
    ops.conv_small_dgrad(2, gz, w1, gd1)
    torch.testing.assert_close(gd1.float(), dr.grad, **tol(dtype))

    # bn3 backward helpers
    mean = c2.float().mean((0, 1, 2))
    var = c2.float().var((0, 1, 2), unbiased=False)
    rstd = 1 / torch.sqrt(var + 1e-3)
    gam = torch.rand(3, device=dev()) + 0.5
    bst = ops.stats_alloc(6, dev())
    ops.bn3_bwd_reduce(gd, c2, mean, rstd, bst)
    c1, cc2, dg, db = (torch.empty(3, device=dev()) for _ in range(4))
    n = B * H2 * W2
    ops.bn_bwd_finalize(bst, n, dg, db, c1, cc2)
    out = torch.empty_like(gd)
    ops.bn3_bwd_dz(gd, c2, gam * rstd, mean, rstd, c1, cc2, out)
    c2r = c2.float().requires_grad_(True)
    F.batch_norm(c2r.reshape(-1, 3), None, None, gam, None, training=True, eps=1e-3).backward(gd.float().reshape(-1, 3))
    torch.testing.assert_close(out.float(), c2r.grad, rtol=3e-2 if dtype == torch.bfloat16 else 1e-3, atol=3e-2 if dtype == torch.bfloat16 else 1e-4)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("stride,pad,accumulate", [(1, 0, False), (2, 1, False), (1, 0, True)],
                         ids=["valid", "stride2_pad1", "accumulate"])
def test_im2col_col2im(stride, pad, accumulate, dtype):
    """block1_conv2's column route (fp32 and deterministic modes, 'valid'): im2col of relu(a*x+b) from bn_apply; col2im
    of the column gradient, masked by the ReLU inside bn_bwd_reduce. Also the same pair with stride 2 and a leading pad
    of 1, and a col2im that adds into the gradient already there."""
    ops = _ops()
    torch.manual_seed(13)
    B, H, W, C = 2, 11, 13, 32
    x = torch.randn(B, H, W, C, device=dev()).to(dtype)
    a = torch.rand(C, device=dev()) + 0.5
    b = torch.randn(C, device=dev()) * 0.2
    pre = x.float() * a + b
    act = ops.bn_apply(x, a, b, act=1)
    OH, OW = (H + 2 * pad - 3) // stride + 1, (W + 2 * pad - 3) // stride + 1
    col = torch.empty(B * OH * OW, 9 * C, device=dev(), dtype=dtype)
    ops.im2col(act, col, 3, 3, stride, pad, pad, OH, OW)
    ref = F.unfold(nchw(torch.relu(pre)), 3, padding=pad, stride=stride)  # [B, C*9, L] with channel-major rows
    ref = ref.reshape(B, C, 9, -1).permute(0, 3, 2, 1).reshape(B * OH * OW, 9 * C)
    torch.testing.assert_close(col.float(), ref, **tol(dtype))
    gcol = torch.randn_like(col.float()).to(dtype)
    gin0 = torch.randn_like(x.float()).to(dtype)
    gin = gin0.clone() if accumulate else torch.full_like(x, float("nan"))  # without accumulate col2im overwrites
    ops.col2im(gcol, gin, 3, 3, stride, pad, pad, OH, OW, accumulate=accumulate)
    mean, rstd = torch.zeros(C, device=dev()), torch.ones(C, device=dev())
    ops.bn_bwd_reduce(gin, x, mean, rstd, ops.stats_alloc(2 * C, dev()), relu_a=a, relu_b=b, act=1)
    gref = gcol.float().reshape(B, -1, 9, C).permute(0, 3, 2, 1).reshape(B, C * 9, -1)
    gref = nhwc(F.fold(gref, (H, W), 3, padding=pad, stride=stride)) + (gin0.float() if accumulate else 0)
    torch.testing.assert_close(gin.float(), gref * (pre > 0), **tol(dtype))


# ------------------------------------------------------------------ optimiser
def test_adam_keras_sumsq_and_colsum():
    ops = _ops()
    torch.manual_seed(17)
    n, n_l2 = 10000, 3000
    p = torch.randn(n, device=dev())
    g = torch.randn(n, device=dev()) * 0.1
    m = torch.randn(n, device=dev()) * 0.01
    v = torch.rand(n, device=dev()) * 0.01
    p0, m0, v0 = p.clone().double(), m.clone().double(), v.clone().double()
    lr, t = 3e-4, 5
    lr_t = lr * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)
    lr_dev = torch.tensor([lr_t], device=dev(), dtype=torch.float32)
    pb = torch.empty(n, device=dev(), dtype=torch.bfloat16)
    ops.adam_keras_step(p, g, m, v, lr_dev, n_l2=n_l2, l2=1e-4, p_bf16=pb)
    gg = g.double().clone()
    gg[:n_l2] += 2e-4 * p0[:n_l2]
    mr = 0.9 * m0 + 0.1 * gg
    vr = 0.999 * v0 + 0.001 * gg * gg
    pr = p0 - lr_t * mr / (vr.sqrt() + 1e-7)
    torch.testing.assert_close(p.double(), pr, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(m.double(), mr, rtol=1e-5, atol=1e-8)
    torch.testing.assert_close(v.double(), vr, rtol=1e-5, atol=1e-9)
    torch.testing.assert_close(pb, p.to(torch.bfloat16))
    acc = ops.stats_alloc(1, dev())
    out = torch.zeros(1, device=dev())
    ops.sumsq(p, n_l2, 1e-4, acc)
    ops.acc_to_f32(acc, out)
    torch.testing.assert_close(out[0].double(), 1e-4 * (p[:n_l2].double() ** 2).sum(), rtol=1e-4, atol=0)
    assert int(acc.abs().max()) == 0  # acc_to_f32 clears the accumulator for the next step
    # frozen mask (one byte per 8 parameters) and bf16 gradients
    p2, m2, v2 = p.clone(), m.clone(), v.clone()
    mask = torch.zeros(n // 8, device=dev(), dtype=torch.uint8)
    mask[100:300] = 1
    gb = g.to(torch.bfloat16)
    ops.adam_keras_step(p2, g, m2, v2, lr_dev, n_l2=n_l2, l2=1e-4, frozen8=mask, g_bf16=gb)
    fr = mask.repeat_interleave(8).bool()
    assert torch.equal(p2[fr], p[fr]) and torch.equal(m2[fr], m[fr]) and torch.equal(v2[fr], v[fr])
    gg2 = gb.double()
    gg2[:n_l2] += 2e-4 * p.double()[:n_l2]
    mr2 = 0.9 * m.double() + 0.1 * gg2
    vr2 = 0.999 * v.double() + 0.001 * gg2 * gg2
    pr2 = p.double() - lr_t * mr2 / (vr2.sqrt() + 1e-7)
    torch.testing.assert_close(p2.double()[~fr], pr2[~fr], rtol=1e-5, atol=1e-7)
    cs = torch.empty(576, device=dev())
    gy = torch.randn(5, 576, device=dev())
    ops.colsum(gy, cs)
    torch.testing.assert_close(cs, gy.sum(0), rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------ full-size, size-independent properties
# (BASELINE.json configs[1] shapes: batch 64, 384x512 -> layer shapes below; no CPU oracle at these sizes)
@pytest.mark.parametrize("M,N,K,a_mn,b_mn", [(12288, 728, 728, False, True), (744000, 128, 64, False, True),
                                              (728, 728, 12288, True, True), (49152, 728, 256, False, False)])
def test_fullsize_gemm_tcgen05_matches_fp32_ffma(M, N, K, a_mn, b_mn):
    """tcgen05 GEMM (bf16 operands) vs the independent fp32 FFMA GEMM (the same operands as fp32), both through
    ops.gemm, which picks the kernel from the operand dtype."""
    ops = _ops()
    torch.manual_seed(M % 1000 + N + K)
    A = (torch.randn((K, M) if a_mn else (M, K), device=dev()) * 0.5).to(torch.bfloat16)
    B = (torch.randn((K, N) if b_mn else (N, K), device=dev()) * 0.5).to(torch.bfloat16)
    mode = ops.OUT_ATOMIC if a_mn else ops.OUT_F32
    D1 = torch.zeros(M, N, device=dev())
    ops.gemm(A, a_mn, B, b_mn, D1, M, N, K, out_mode=mode, splits=0 if a_mn else 1)
    D2 = torch.zeros(M, N, device=dev())
    ops.gemm(A.float(), a_mn, B.float(), b_mn, D2, M, N, K, out_mode=ops.OUT_F32)
    scale = float(D2.abs().max())
    torch.testing.assert_close(D1, D2, rtol=1e-3, atol=2e-4 * scale)


@pytest.mark.parametrize("shape", [(64, 93, 125, 128), (64, 12, 16, 728)])
def test_fullsize_depthwise_adjoint_identities(shape):
    """<dw_k(x), g> = <x, dw_k^T(g)> = <k, dk>: forward, data gradient and weight gradient of the packed
    kernels are mutually consistent at the benchmark's layer shapes (fp32, no activation)."""
    ops = _ops()
    torch.manual_seed(21)
    B, H, W, C = shape
    x = torch.randn(shape, device=dev())
    g = torch.randn(shape, device=dev())
    k = torch.randn(3, 3, C, device=dev()) * 0.3
    y = ops.dwconv3x3_fwd(x, k)
    dk = torch.zeros(3, 3, C, device=dev())
    gin = ops.dwconv3x3_bwd_fused(g, x, k, dk)
    lhs = float((y.double() * g.double()).sum())
    mid = float((x.double() * gin.double()).sum())
    rhs = float((k.double() * dk.double()).sum())
    assert abs(lhs - mid) / abs(lhs) < 1e-4, (lhs, mid)
    assert abs(lhs - rhs) / abs(lhs) < 1e-4, (lhs, rhs)
    # linearity in the input
    y2 = ops.dwconv3x3_fwd(2.0 * x + 1.0, k)
    ones = ops.dwconv3x3_fwd(torch.ones_like(x), k)
    torch.testing.assert_close(y2, 2.0 * y + ones, rtol=1e-4, atol=1e-4)


# ----------------------------------------------------------------------------- implicit-GEMM convolutions
# (B, H, W, Cin, Cout, KH, KW, pad): Xception block1_conv2 ('valid' 3x3, 32 -> 64), InceptionResNetV2 branch
# shapes (3x3 / 5x5 'same', 1x7, 7x1, 1x3, 3x1; ragged channel counts; tiny feature maps spanning images)
CONV_TC_CASES = [
    (2, 31, 43, 32, 64, 3, 3, "valid"),
    (3, 21, 29, 48, 64, 5, 5, "same"),
    (2, 21, 29, 64, 96, 3, 3, "same"),
    (5, 10, 14, 128, 160, 1, 7, "same"),
    (5, 10, 14, 160, 192, 7, 1, "same"),
    (9, 4, 6, 192, 224, 1, 3, "same"),
    (9, 4, 6, 224, 256, 3, 1, "same"),
    (2, 46, 62, 80, 192, 3, 3, "valid"),
    (1, 9, 140, 32, 32, 3, 3, "same"),
]


def _conv_tc_inputs(case, seed=0):
    B, H, W, Cin, Cout, KH, KW, pad = case
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn(B, H, W, Cin, generator=g).to(dev()).bfloat16()
    wt = (torch.randn(KH, KW, Cin, Cout, generator=g) / (KH * KW * Cin) ** 0.5).to(dev()).bfloat16()
    if pad == "same":
        OH, OW, pt, pl = H, W, (KH - 1) // 2, (KW - 1) // 2
    else:
        OH, OW, pt, pl = H - KH + 1, W - KW + 1, 0, 0
    return x, wt, OH, OW, pt, pl


def _conv_ref(x, wt, pad, KH, KW):
    p = ((KH - 1) // 2, (KW - 1) // 2) if pad == "same" else 0
    return F.conv2d(nchw(x), wt.float().permute(3, 2, 0, 1).contiguous(), padding=p)


@pytest.mark.parametrize("case", CONV_TC_CASES)
def test_conv_tc_fwd_and_stats(case):
    ops = _ops()
    B, H, W, Cin, Cout, KH, KW, pad = case
    x, wt, OH, OW, pt, pl = _conv_tc_inputs(case)
    ref = nhwc(_conv_ref(x, wt, pad, KH, KW))
    y = torch.full((B, OH, OW, Cout), float("nan"), device=dev(), dtype=torch.bfloat16)
    stats = ops.stats_alloc(2 * Cout, dev())
    ops.conv_tc_fwd(x, wt, y, pt, pl, colstats=stats)
    torch.testing.assert_close(y.float(), ref, rtol=2e-2, atol=2e-2)
    yf = y.double().view(-1, Cout)
    sv = ops.stats_values(stats).to(yf.device)
    torch.testing.assert_close(sv[:Cout], yf.sum(0), rtol=1e-5, atol=1e-3)
    torch.testing.assert_close(sv[Cout:], (yf * yf).sum(0), rtol=1e-5, atol=1e-3)


KWFOLD_CASES = [(2, 46, 62, 32, 64, 3, 3), (3, 21, 141, 32, 64, 3, 3), (5, 9, 70, 16, 24, 3, 3), (2, 12, 40, 32, 128, 2, 5),
                (1, 30, 131, 64, 64, 3, 3)]


@pytest.mark.parametrize("case", KWFOLD_CASES)
def test_conv_tc_kwfold_fwd_wgrad(case):
    """'valid' convolution with the KW taps folded into the channel axis (overlapping-row tensor map): block1_conv2's
    route. Forward + fused statistics against torch, weight gradient against fp64."""
    ops = _ops()
    B, H, W, Cin, Cout, KH, KW = case
    x, wt, OH, OW, _, _ = _conv_tc_inputs((B, H, W, Cin, Cout, KH, KW, "valid"), seed=5)
    ref = nhwc(_conv_ref(x, wt, "valid", KH, KW))
    y = torch.full((B, OH, OW, Cout), float("nan"), device=dev(), dtype=torch.bfloat16)
    stats = ops.stats_alloc(2 * Cout, dev())
    ops.conv_tc_fwd_kwfold(x, wt, y, colstats=stats)
    torch.testing.assert_close(y.float(), ref, rtol=2e-2, atol=2e-2)
    yf = y.double().view(-1, Cout)
    sv = ops.stats_values(stats).to(yf.device)
    torch.testing.assert_close(sv[:Cout], yf.sum(0), rtol=1e-5, atol=1e-3)
    torch.testing.assert_close(sv[Cout:], (yf * yf).sum(0), rtol=1e-5, atol=1e-3)
    g = torch.Generator(device="cpu").manual_seed(6)
    gy = torch.randn(B, OH, OW, Cout, generator=g).to(dev()).bfloat16()
    xr = nchw(x).double().cpu()
    wr = wt.double().permute(3, 2, 0, 1).contiguous().cpu().requires_grad_(True)
    F.conv2d(xr, wr).backward(nchw(gy).double().cpu())
    ref_w = wr.grad.permute(2, 3, 1, 0).contiguous().float().to(dev())
    gw = torch.zeros(KH, KW, Cin, Cout, device=dev())
    ops.conv_tc_wgrad_kwfold(x, gy, gw)
    scale = float(ref_w.abs().max())
    torch.testing.assert_close(gw, ref_w, rtol=2e-3, atol=2e-3 * scale)


def test_conv_tc_fwd_channel_slices():
    """Input and output as channel slices of wider NHWC buffers (concat targets), untouched neighbours."""
    ops = _ops()
    case = (3, 21, 29, 64, 96, 3, 3, "same")
    B, H, W, Cin, Cout, KH, KW, pad = case
    x, wt, OH, OW, pt, pl = _conv_tc_inputs(case, seed=3)
    xw = torch.randn(B, H, W, Cin + 40, device=dev()).bfloat16()
    xw[..., 8:8 + Cin] = x
    yw = torch.full((B, OH, OW, Cout + 64), 7.0, device=dev(), dtype=torch.bfloat16)
    ops.conv_tc_fwd(xw[..., 8:8 + Cin], wt, yw[..., 32:32 + Cout], pt, pl, ldx=Cin + 40, ldy=Cout + 64)
    ref = nhwc(_conv_ref(x, wt, pad, KH, KW))
    torch.testing.assert_close(yw[..., 32:32 + Cout].float(), ref, rtol=2e-2, atol=2e-2)
    assert bool((yw[..., :32] == 7.0).all()) and bool((yw[..., 32 + Cout:] == 7.0).all())


@pytest.mark.parametrize("case", CONV_TC_CASES)
def test_conv_tc_dgrad_wgrad(case):
    ops = _ops()
    B, H, W, Cin, Cout, KH, KW, pad = case
    x, wt, OH, OW, pt, pl = _conv_tc_inputs(case, seed=1)
    g = torch.Generator(device="cpu").manual_seed(2)
    gy = torch.randn(B, OH, OW, Cout, generator=g).to(dev()).bfloat16()
    # exact reference: fp64 on the CPU (cuDNN's fp32 weight-gradient algorithms are themselves ~1e-3 of the scale)
    xr = nchw(x).double().cpu().requires_grad_(True)
    wr = wt.double().permute(3, 2, 0, 1).contiguous().cpu().requires_grad_(True)
    p = ((KH - 1) // 2, (KW - 1) // 2) if pad == "same" else 0
    F.conv2d(xr, wr, padding=p).backward(nchw(gy).double().cpu())
    gx = torch.full((B, H, W, Cin), float("nan"), device=dev(), dtype=torch.bfloat16)
    ops.conv_tc_dgrad(gy, wt, gx, pt, pl)
    torch.testing.assert_close(gx.float(), nhwc(xr.grad).float().to(dev()), rtol=2e-2, atol=2e-2)
    gw = torch.zeros(KH, KW, Cin, Cout, device=dev())
    ops.conv_tc_wgrad(x, gy, gw, pt, pl)
    ref_w = wr.grad.permute(2, 3, 1, 0).contiguous().float().to(dev())
    scale = float(ref_w.abs().max())
    torch.testing.assert_close(gw, ref_w, rtol=2e-3, atol=2e-3 * scale)
    ops.conv_tc_wgrad(x, gy, gw, pt, pl)  # reduce-add: a second call accumulates
    torch.testing.assert_close(gw, 2 * ref_w, rtol=2e-3, atol=4e-3 * scale)
