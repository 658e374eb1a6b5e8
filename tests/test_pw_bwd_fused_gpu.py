"""Fused BatchNorm + pointwise-conv backward (ops.pw_bwd_bn): dz = bn_bwd_dz(g, z, ...) stays on chip, gA = dz W^T,
gW += t^T dz. gA must be bit-identical to bn_bwd_dz followed by the data-gradient GEMM (same bf16 dz, same K order);
gW must match the weight-gradient GEMM on the same dz up to fp32 reassociation, and an fp64 reference. With slabs the
weight gradient is bit-reproducible. g is left unchanged."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ops():
    from spnet_b200 import ops
    return ops


# (M, cin, cout): Xception's block-2 sites at batch 64 reduced to batch 2 (block2_sepconv1 / sepconv2 at 93x125,
# the residual conv2d_4 at 47x63), a ragged M below one tile and one just above, and a multi-wave M
SHAPES = [(2 * 93 * 125, 64, 128), (2 * 93 * 125, 128, 128), (2 * 47 * 63, 64, 128), (77, 128, 128), (129, 64, 128),
          (148 * 128 * 3 + 5, 128, 128)]


def _inputs(M, cin, cout, seed):
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, device=dev, generator=gen)  # noqa: E731
    g = rnd(M, cout).bfloat16()
    z = (rnd(M, cout) * 2 + 0.5).bfloat16()
    t = rnd(M, cin).bfloat16()
    W = (rnd(cin, cout) * 0.1).bfloat16()
    a = rnd(cout) * 0.5 + 1
    mean = rnd(cout) * 0.3
    rstd = rnd(cout).abs() + 0.5
    c1, c2 = rnd(cout) * 0.1, rnd(cout) * 0.1
    return g, z, t, W, a, mean, rstd, c1, c2


def _old_route(ops, g, z, t, W, a, mean, rstd, c1, c2, M, cin, cout):
    dz = ops.bn_bwd_dz(g, z, a, mean, rstd, c1, c2, out=torch.empty_like(g))
    gW = torch.zeros(cin, cout, device=g.device)
    ops.gemm(t, True, dz, True, gW, cin, cout, M, out_mode=ops.OUT_ATOMIC, splits=0, lda=cin, ldb=cout)
    gA = torch.empty(M, cin, device=g.device, dtype=torch.bfloat16)
    ops.gemm(dz, False, W, False, gA, M, cin, cout, out_mode=ops.OUT_T, ldb=cout)
    return dz, gA, gW


@pytest.mark.parametrize("M,cin,cout", SHAPES)
def test_pw_bwd_bn_matches_unfused_route(M, cin, cout):
    ops = _ops()
    g, z, t, W, a, mean, rstd, c1, c2 = _inputs(M, cin, cout, 1000 + M + cin)
    dz, gA_ref, gW_ref = _old_route(ops, g, z, t, W, a, mean, rstd, c1, c2, M, cin, cout)
    g0 = g.clone()
    gA = torch.full((M, cin), float("nan"), device=g.device, dtype=torch.bfloat16)
    gW = torch.ones(cin, cout, device=g.device)  # accumulates
    ops.pw_bwd_bn(g, z, t, W, a, mean, rstd, c1, c2, gA, gW, M, cin, cout)
    torch.cuda.synchronize()
    assert torch.equal(g, g0)
    assert torch.equal(gA.view(torch.int16), gA_ref.view(torch.int16))
    gW = gW - 1
    ref64 = t.double().t() @ dz.double()
    mag = t.double().abs().t() @ dz.double().abs()
    assert bool(((gW.double() - gW_ref.double()).abs() <= 1e-5 * mag + 1e-5).all())
    assert bool(((gW.double() - ref64).abs() <= 1e-5 * mag + 1e-5).all())


@pytest.mark.parametrize("M,cin,cout", [SHAPES[0], SHAPES[1], SHAPES[4]])
def test_pw_bwd_bn_slabs_are_reproducible(M, cin, cout):
    ops = _ops()
    g, z, t, W, a, mean, rstd, c1, c2 = _inputs(M, cin, cout, 7 + cin)
    dz, gA_ref, _ = _old_route(ops, g, z, t, W, a, mean, rstd, c1, c2, M, cin, cout)
    n = ops.pw_bwd_bn_slabs(M)
    outs = []
    for _ in range(2):
        slabs = torch.full((n * cin * cout,), float("nan"), device=g.device)  # every slab is written in full
        gA = torch.empty(M, cin, device=g.device, dtype=torch.bfloat16)
        gW = torch.zeros(cin, cout, device=g.device)
        ops.pw_bwd_bn(g, z, t, W, a, mean, rstd, c1, c2, gA, gW, M, cin, cout, slabs=slabs)
        outs.append((gA, gW))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][1], outs[1][1])
    assert torch.equal(outs[0][0].view(torch.int16), gA_ref.view(torch.int16))
    ref64 = t.double().t() @ dz.double()
    mag = t.double().abs().t() @ dz.double().abs()
    assert bool(((outs[0][1].double() - ref64).abs() <= 1e-5 * mag + 1e-5).all())
