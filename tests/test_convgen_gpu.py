"""The glue kernels of the dense-convolution backbone (csrc/convgen.cu, and the cast / inference-affine kernels of the
shared engine base) against fp64, at the shapes InceptionResNetV2-SPNet runs them and at the edges: 1-, 2- and 3-wide
maps, one channel vector, ragged row counts, the concat offsets and pitches of the program. Every written region is
prefilled with NaN and surrounded by canary elements that must survive bit for bit.

Tolerances: an fp32 result within 1e-5 x sum|terms| of the fp64 value; a bf16 result at most one bf16 ulp beyond that;
copies bit-exact."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from test_parity_configs_gpu import record  # noqa: E402

DT = {"fp32": torch.float32, "bf16": torch.bfloat16}
VEC = {"fp32": 4, "bf16": 8}
PAD = 64   # canary elements on either side of a written region (keeps 16-byte alignment)


def dev():
    return torch.device("cuda:0")


def guarded(shape, dtype, init=None):
    """A tensor of `shape` inside a buffer with PAD canary elements before and after it; NaN unless init is given."""
    n = int(np.prod(shape))
    buf = torch.randn(n + 2 * PAD, device=dev()).mul_(1e3).to(dtype)
    t = buf[PAD:PAD + n].view(shape)
    t.copy_(init) if init is not None else t.fill_(float("nan"))
    return buf, t, buf.clone()


def canaries_intact(buf, saved):
    return torch.equal(buf[:PAD], saved[:PAD]) and torch.equal(buf[-PAD:], saved[-PAD:])


def close(got, ref64, scale64):
    got = got.reshape(ref64.shape)
    if got.dtype == torch.bfloat16:
        ref = ref64.to(torch.bfloat16).double()
        ulp = torch.pow(2.0, torch.floor(torch.log2(ref.abs().clamp_min(1e-30))) - 7)
        excess = float((((got.double() - ref).abs() - 1e-5 * scale64) / ulp).max())
        assert excess <= 1.0 + 1e-9, excess
    else:
        q = float(((got.double() - ref64).abs() / (1e-5 * scale64).clamp_min(1e-300)).max())
        assert q <= 1.0, q


def nchw(t):
    return t.double().permute(0, 3, 1, 2).contiguous()


def nhwc(t):
    return t.permute(0, 2, 3, 1)


# ------------------------------------------------------------------ AveragePooling2D(3, 1, 'same')
@pytest.mark.parametrize("dt", sorted(DT))
@pytest.mark.parametrize("hw", [(1, 1), (1, 2), (2, 1), (2, 2), (3, 3), (1, 3), (3, 2), (13, 18)])
@pytest.mark.parametrize("cw", ["vec", 192, 320])
def test_avgpool3s1_forward_adjoint_and_accumulate(dt, hw, cw):
    from spnet_b200 import ops
    dtype = DT[dt]
    C = VEC[dt] if cw == "vec" else cw
    B, (H, W) = 2, hw
    torch.manual_seed(H * 100 + W + C)
    x = torch.randn(B, H, W, C, device=dev()).to(dtype)
    def pool(t):   # TF divides by the number of in-image cells of the window
        return nhwc(F.avg_pool2d(nchw(t), 3, 1, 1, count_include_pad=False))
    buf, out, saved = guarded((B, H, W, C), dtype)
    ops.avgpool3s1(x, out)
    close(out, pool(x), pool(x.abs()))
    assert canaries_intact(buf, saved)
    # backward: the adjoint, each window divided by ITS count of in-image cells
    g = torch.randn(B, H, W, C, device=dev()).to(dtype)
    xr = torch.zeros(B, C, H, W, device=dev(), dtype=torch.float64, requires_grad=True)
    p = F.avg_pool2d(xr, 3, 1, 1, count_include_pad=False)
    adj, = torch.autograd.grad(p, xr, nchw(g), retain_graph=True)
    adj_abs, = torch.autograd.grad(p, xr, nchw(g).abs())
    adj, adj_abs = nhwc(adj), nhwc(adj_abs)
    buf, gin, saved = guarded((B, H, W, C), dtype)
    ops.avgpool3s1(g, gin, bwd=True)
    close(gin, adj, adj_abs)
    assert canaries_intact(buf, saved)
    # <bwd(g), x> = <g, fwd(x)> in fp64 on the kernels' own outputs
    lhs, rhs = float((gin.double() * x.double()).sum()), float((g.double() * out.double()).sum())
    scale = float((gin.double() * x.double()).abs().sum() + (g.double() * out.double()).abs().sum())
    assert abs(lhs - rhs) <= (2.0 ** -8 if dtype == torch.bfloat16 else 1e-5) * scale, (lhs, rhs, scale)
    # accumulate = 1 adds into what is there
    g0 = torch.randn(B, H, W, C, device=dev()).to(dtype)
    buf, gacc, saved = guarded((B, H, W, C), dtype, init=g0)
    ops.avgpool3s1(g, gacc, bwd=True, accumulate=True)
    close(gacc, g0.double() + adj, g0.double().abs() + adj_abs)
    assert canaries_intact(buf, saved)


# ------------------------------------------------------------------ Concatenate and its adjoint
# (pitch, [(offset, width), ...]) of every concat of the program: mixed_5b, block35, block17, block8, mixed_6a, mixed_7a
CONCATS = {"mixed_5b": (320, [(0, 96), (96, 64), (160, 96), (256, 64)]), "block35": (128, [(0, 32), (32, 32), (64, 64)]),
           "block17": (384, [(0, 192), (192, 192)]), "block8": (448, [(0, 192), (192, 256)]),
           "mixed_6a": (1088, [(0, 384), (384, 384), (768, 320)]),
           "mixed_7a": (2080, [(0, 384), (384, 288), (672, 320), (992, 1088)])}


@pytest.mark.parametrize("dt", sorted(DT))
@pytest.mark.parametrize("concat", sorted(CONCATS))
@pytest.mark.parametrize("accumulate", [False, True])
def test_copy2d_concat_slices(dt, concat, accumulate):
    from spnet_b200 import ops
    dtype = DT[dt]
    ld, parts = CONCATS[concat]
    rows = 2 * 13 * 18 + 1
    torch.manual_seed(ld + rows)
    for off, c in parts:
        # forward: the branch into its slice of the concatenated tensor; the other columns stay as they were
        src = torch.randn(rows, c, device=dev()).to(dtype)
        d0 = torch.randn(rows, ld, device=dev()).to(dtype)
        buf, dst, saved = guarded((rows, ld), dtype, init=d0)
        ops.copy2d(src, 0, c, dst, off, ld, rows, c, accumulate=accumulate)
        if accumulate:
            close(dst[:, off:off + c], d0[:, off:off + c].double() + src.double(),
                  d0[:, off:off + c].double().abs() + src.double().abs())
        else:
            assert torch.equal(dst[:, off:off + c], src)
        assert torch.equal(dst[:, :off], d0[:, :off]) and torch.equal(dst[:, off + c:], d0[:, off + c:])
        assert canaries_intact(buf, saved)
        # adjoint: the slice of the concat gradient into the branch gradient (dense, pitch c)
        g = torch.randn(rows, ld, device=dev()).to(dtype)
        b0 = torch.randn(rows, c, device=dev()).to(dtype)
        buf, gb, saved = guarded((rows, c), dtype, init=b0 if accumulate else None)
        ops.copy2d(g, off, ld, gb, 0, c, rows, c, accumulate=accumulate)
        if accumulate:
            close(gb, b0.double() + g[:, off:off + c].double(), b0.double().abs() + g[:, off:off + c].double().abs())
        else:
            assert torch.equal(gb, g[:, off:off + c])
        assert canaries_intact(buf, saved)


# ------------------------------------------------------------------ scaled residual
@pytest.mark.parametrize("dt", sorted(DT))
@pytest.mark.parametrize("with_bias", [True, False])
@pytest.mark.parametrize("relu", [1, 0])
@pytest.mark.parametrize("accumulate_gx", [0, 1])
def test_residual_fwd_bwd(dt, with_bias, relu, accumulate_gx):
    from spnet_b200 import ops
    dtype = DT[dt]
    rows, C = 2 * 6 * 8 + 3, 1088
    torch.manual_seed(rows + C + relu)
    for scale in (0.17, 0.1, 0.2, 1.0):
        x = torch.randn(rows, C, device=dev()).to(dtype)
        u = torch.randn(rows, C, device=dev()).to(dtype)
        bias = (torch.randn(C, device=dev()) * 0.5).to(torch.bfloat16).float() if with_bias else None
        # the first rows: x + scale * (u + bias) == 0 exactly
        x[:5] = 0
        u[:5] = (-bias).to(dtype) if with_bias else 0
        buf, y, saved = guarded((rows, C), dtype)
        ops.residual_fwd(x, u, bias, scale, relu, y)
        b64 = bias.double() if with_bias else torch.zeros(C, device=dev(), dtype=torch.float64)
        ref = x.double() + scale * (u.double() + b64)
        close(y, torch.relu(ref) if relu else ref, x.double().abs() + scale * (u.double().abs() + b64.abs()))
        assert canaries_intact(buf, saved)
        assert bool((y[:5] == 0).all())
        gy = torch.randn(rows, C, device=dev()).to(dtype)
        gx0 = torch.randn(rows, C, device=dev()).to(dtype)
        bufx, gx, savedx = guarded((rows, C), dtype, init=gx0 if accumulate_gx else None)
        bufu, gu, savedu = guarded((rows, C), dtype)
        ops.residual_bwd(gy, y, scale, relu, gx, accumulate_gx, gu)
        gm = torch.where(y > 0, gy, torch.zeros_like(gy)) if relu else gy
        if accumulate_gx:
            close(gx, gx0.double() + gm.double(), gx0.double().abs() + gm.double().abs())
        else:
            assert torch.equal(gx, gm)
        close(gu, scale * gm.double(), scale * gm.double().abs())
        if relu:   # y == 0 exactly: no gradient passes
            assert bool((gu[:5] == 0).all()) and (accumulate_gx or bool((gx[:5] == 0).all()))
        assert canaries_intact(bufx, savedx) and canaries_intact(bufu, savedu)


# ------------------------------------------------------------------ bias gradient: column sums
def _colsum_per(C, V):
    """Row lanes per CTA of spnet_colsum_rows (its launch arithmetic)."""
    CV = C // V
    chunks = -(-CV // 128)
    return 256 // -(-CV // chunks), chunks


@pytest.mark.parametrize("dt,C,n_chunks", [("bf16", 8, 1), ("bf16", 320, 1), ("bf16", 1088, 2), ("bf16", 2080, 3),
                                           ("fp32", 4, 1), ("fp32", 512, 1), ("fp32", 1088, 3)])
@pytest.mark.parametrize("with_acc", [False, True])
def test_colsum_rows(dt, C, n_chunks, with_acc):
    from spnet_b200 import ops
    dtype = DT[dt]
    per, chunks = _colsum_per(C, VEC[dt])
    assert chunks == n_chunks
    torch.manual_seed(C)
    for rows in sorted({1, per - 1, per, 24, 192, 100003}):
        g = torch.randn(rows, C, device=dev()).to(dtype)
        out0 = torch.randn(C, device=dev())
        buf, out, saved = guarded((C,), torch.float32, init=out0)
        acc = ops.stats_alloc(C + 5, dev()) if with_acc else None
        ops.colsum_rows(g, out, acc=acc)
        close(out, out0.double() + g.double().sum(0), out0.double().abs() + g.double().abs().sum(0))
        assert canaries_intact(buf, saved)
        if with_acc:
            assert not bool(acc.any())   # cleared for the next use


def test_colsum_rows_row_order():
    """The accumulator form gives the same bits whatever the order of the rows; the atomic form's fp32 partial sums
    depend on which rows meet in which thread (recorded, not asserted)."""
    from spnet_b200 import ops
    torch.manual_seed(17)
    res = {}
    for dt, C in (("bf16", 2080), ("bf16", 320), ("fp32", 1088)):
        g = torch.randn(100003, C, device=dev()).to(DT[dt])
        perm = torch.randperm(g.shape[0], device=dev())
        acc = ops.stats_alloc(C, dev())
        outs = {}
        for form in ("accumulators", "atomics"):
            for order, t in (("rows", g), ("permuted", g[perm].contiguous())):
                out = torch.zeros(C, device=dev())
                ops.colsum_rows(t, out, acc=acc if form == "accumulators" else None)
                outs[form, order] = out
        torch.cuda.synchronize()
        res["%s_C%d" % (dt, C)] = {
            "accumulators_bit_identical": torch.equal(outs["accumulators", "rows"], outs["accumulators", "permuted"]),
            "atomics_bit_identical": torch.equal(outs["atomics", "rows"], outs["atomics", "permuted"]),
            "atomics_channels_differing": int((outs["atomics", "rows"] != outs["atomics", "permuted"]).sum())}
        ref = g.double().sum(0)
        for k, o in outs.items():
            close(o, ref, g.double().abs().sum(0))
    record("colsum_rows_row_order", res)
    assert all(v["accumulators_bit_identical"] for v in res.values()), res


# ------------------------------------------------------------------ fp32 -> bf16 working copy
@pytest.mark.parametrize("n", [1, 7, 8 * 1000 + 3])
def test_cast_f32_to_bf16(n):
    from spnet_b200 import ops
    torch.manual_seed(n)
    special = torch.tensor([1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, -(1.0 + 2 ** -8), 2.0 + 2 ** -7, 0.0, -0.0, float("inf"),
                            float("-inf"), float("nan"), 3.4028235e38, -3.39e38, 1e-40, -1e-41, 1.4e-45, 1.1754942e-38,
                            9.2e-39, 65504.0, 1.0 - 2 ** -9], device=dev())
    src = torch.randn(n, device=dev()) * torch.exp(torch.randn(n, device=dev()) * 8)
    src[:min(n, special.numel())] = special[:min(n, special.numel())]
    if n < special.numel():   # every special value, n at a time
        chunks = [special[i:i + n] for i in range(0, special.numel(), n)]
    else:
        chunks = [src]
    for s in chunks:
        s = s.contiguous()
        m = s.numel()
        buf, dst, saved = guarded((m,), torch.bfloat16)
        ops.cast_f32_to_bf16(s, dst)
        ref = s.to(torch.bfloat16)
        nan = torch.isnan(s)
        assert bool(torch.isnan(dst[nan]).all())
        assert torch.equal(dst[~nan].view(torch.int16), ref[~nan].view(torch.int16))
        assert canaries_intact(buf, saved)


# ------------------------------------------------------------------ inference-mode BatchNorm affine
@pytest.mark.parametrize("C", [3, 128, 2080])
@pytest.mark.parametrize("with_gamma", [True, False])
@pytest.mark.parametrize("save", [False, True])
def test_bn_inference_affine(C, with_gamma, save):
    from spnet_b200 import arch, ops
    torch.manual_seed(C)
    gamma = torch.rand(C, device=dev()) + 0.5 if with_gamma else None
    beta, mm = torch.randn(C, device=dev()), torch.randn(C, device=dev())
    mv = torch.rand(C, device=dev()) * 2 + 1e-4
    mv[0] = 0.0
    bufs = [guarded((C,), torch.float32) for _ in range(4)]
    a, b, sm, sr = (t for _, t, _ in bufs)
    ops.bn_inference_affine(gamma, beta, mm, mv, a, b, eps=arch.BN_EPS, save_mean=sm if save else None,
                            save_rstd=sr if save else None)
    rstd = 1.0 / torch.sqrt(mv.double() + float(np.float32(arch.BN_EPS)))
    a64 = (gamma.double() if with_gamma else 1.0) * rstd
    assert float(((a.double() - a64).abs() / a64).max()) < 4e-7
    close(b, beta.double() - mm.double() * a.double(), beta.double().abs() + (mm.double() * a.double()).abs())
    if save:
        assert torch.equal(sm, mm)
        assert float(((sr.double() - rstd).abs() / rstd).max()) < 4e-7
    else:
        assert bool(torch.isnan(sm).all() and torch.isnan(sr).all())
    assert all(canaries_intact(bb, s) for bb, _, s in bufs)


# ------------------------------------------------------------------ im2col / col2im at the program's geometries
GEOMS = {"1x7_pad_0_3": (6, 8, 1, 7, 1, 0, 3), "7x1_pad_3_0": (6, 8, 7, 1, 1, 3, 0), "1x3_pad_0_1": (2, 3, 1, 3, 1, 0, 1),
         "3x1_pad_1_0": (2, 3, 3, 1, 1, 1, 0), "5x5_same": (13, 18, 5, 5, 1, 2, 2), "3x3_same": (13, 18, 3, 3, 1, 1, 1),
         "3x3_s2_valid_odd": (13, 17, 3, 3, 2, 0, 0), "3x3_s2_valid_even": (14, 18, 3, 3, 2, 0, 0),
         "3x3_s2_valid_mixed": (13, 18, 3, 3, 2, 0, 0)}


@pytest.mark.parametrize("dt", sorted(DT))
@pytest.mark.parametrize("geom", sorted(GEOMS))
@pytest.mark.parametrize("accumulate", [False, True])
def test_im2col_col2im_program_geometries(dt, geom, accumulate):
    from spnet_b200 import ops
    dtype = DT[dt]
    H, W, kh, kw, s, pt, pl = GEOMS[geom]
    B, C = 2, 48
    OH, OW = ((H - kh) // s + 1, (W - kw) // s + 1) if pt == pl == 0 and s == 2 else (H, W)
    pb, pr = (OH - 1) * s + kh - H - pt, (OW - 1) * s + kw - W - pl
    torch.manual_seed(H * W + kh * 10 + kw)
    x = torch.randn(B, H, W, C, device=dev()).to(dtype)
    M, K = B * OH * OW, kh * kw * C
    buf, col, saved = guarded((M, K), dtype)
    ops.im2col(x, col, kh, kw, s, pt, pl, OH, OW)
    ref = F.unfold(F.pad(nchw(x), (pl, pr, pt, pb)), (kh, kw), stride=s)       # [B, C*kh*kw, L]
    ref = ref.view(B, C, kh * kw, OH * OW).permute(0, 3, 2, 1).reshape(M, K)
    assert torch.equal(col, ref.to(dtype))
    assert canaries_intact(buf, saved)
    gcol = torch.randn(M, K, device=dev()).to(dtype)
    g0 = torch.randn(B, H, W, C, device=dev()).to(dtype)
    buf, gin, saved = guarded((B, H, W, C), dtype, init=g0 if accumulate else None)
    ops.col2im(gcol, gin, kh, kw, s, pt, pl, OH, OW, accumulate=accumulate)

    def fold(t):
        t = t.double().view(B, OH * OW, kh * kw, C).permute(0, 3, 2, 1).reshape(B, C * kh * kw, OH * OW)
        f = F.fold(t, (H + pt + pb, W + pl + pr), (kh, kw), stride=s)
        return nhwc(F.pad(f, (-pl, -pr, -pt, -pb)))
    base = g0.double() if accumulate else 0.0
    close(gin, base + fold(gcol), (g0.double().abs() if accumulate else 0.0) + fold(gcol.abs()))
    assert canaries_intact(buf, saved)
