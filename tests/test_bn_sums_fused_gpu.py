"""BatchNorm-backward sums folded into the kernels that write the gradient: the depthwise backward with an output
BatchNorm (`zo`, optional ReLU mask) and the max-pool backward with `z`. Each must write the same gradient bit for
bit as the same call without the sums (then masked by bn_bwd_reduce, where a mask is given), and its sums must match
bn_bwd_reduce on that gradient up to fp32 reassociation and an fp64 reference. The depthwise kernel gradient matches
the call without the sums up to fp32 reassociation (the stage with one more box may be tiled differently)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ops():
    from spnet_b200 import ops
    return ops


def dev():
    return torch.device("cuda:0")


def check_sums(ops, st, st_ref, g, z, mean, rstd):
    """st against bn_bwd_reduce's st_ref (fp32 reassociation) and against fp64 sums over the stored g."""
    C = z.shape[-1]
    gq = g.double().reshape(-1, C)
    xh = ((z.double() - mean.double()) * rstd.double()).reshape(-1, C)
    sv, sr = ops.stats_values(st).to(g.device), ops.stats_values(st_ref).to(g.device)
    for lo, terms in ((0, gq), (C, gq * xh)):
        mag = terms.abs().sum(0)
        # fp32 partial sums in a different order: a few ulp of fp32 relative to the sum of magnitudes
        assert bool(((sv[lo:lo + C] - sr[lo:lo + C]).abs() <= 2e-5 * mag + 1e-6).all())
        torch.testing.assert_close(sv[lo:lo + C], terms.sum(0), rtol=1e-4, atol=1e-3)


# the shapes the depthwise backward runs with an output BatchNorm in Xception at 384x512 (batch reduced), + ragged
DW_SHAPES = [(2, 93, 125, 64), (2, 47, 63, 128), (2, 24, 32, 256), (4, 12, 16, 728), (4, 6, 8, 1024), (3, 7, 9, 24)]
# (epilogue, relu on load): the combinations the Xception engine runs
DW_MODES = [("none", 0), ("add_src", 1), ("add_strided", 1), ("add_strided", 0)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", DW_SHAPES)
@pytest.mark.parametrize("mode", DW_MODES)
@pytest.mark.parametrize("masked", [False, True])
def test_dwconv_bwd_output_bn_sums(dtype, shape, mode, masked):
    ops = _ops()
    torch.manual_seed(11)
    B, H, W, C = shape
    epi, relu = mode
    x = torch.randn(shape, device=dev()).to(dtype)
    g = torch.randn(shape, device=dev()).to(dtype)
    zo = (torch.randn(shape, device=dev()) * 1.5 + 0.3).to(dtype)
    k = torch.randn(3, 3, C, device=dev()) * 0.3
    mean = torch.randn(C, device=dev()) * 0.2
    rstd = torch.rand(C, device=dev()) + 0.5
    ma = torch.randn(C, device=dev()) if masked else None  # negative scales too
    mb = torch.randn(C, device=dev()) * 0.2 if masked else None
    add = torch.randn(shape, device=dev()).to(dtype) if epi == "add_src" else None
    sadd = torch.randn(B, (H + 1) // 2, (W + 1) // 2, C, device=dev()).to(dtype) if epi == "add_strided" else None

    def run(with_zo):
        dk = torch.zeros(3, 3, C, device=dev())
        acc = ops.stats_alloc(9 * C, dev())  # order-independent across CTAs
        st = ops.stats_alloc(2 * C, dev())
        kw = dict(zo=zo, zo_mean=mean, zo_rstd=rstd, zo_stats=st, mask_a=ma, mask_b=mb) if with_zo else {}
        gin = ops.dwconv3x3_bwd_fused(g, x, k, dk, relu=relu, add_src=add, add_strided=sadd, acc=acc, **kw)
        return gin, dk, st

    gin, dk, st = run(True)
    ref, dk_ref, _ = run(False)
    st_ref = ops.stats_alloc(2 * C, dev())
    ops.bn_bwd_reduce(ref, zo, mean, rstd, st_ref, relu_a=ma, relu_b=mb, act=1)  # masks ref in place
    torch.cuda.synchronize()
    assert torch.equal(gin, ref)
    # the extra box can make the kernel pick lower tiles: the kernel-gradient partials are then summed in another order
    torch.testing.assert_close(dk, dk_ref, rtol=1e-5, atol=1e-5 * float(dk_ref.abs().max()))
    check_sums(ops, st, st_ref, gin, zo, mean, rstd)


def test_dwconv_bwd_output_bn_rejects_uninstantiated():
    ops = _ops()
    from spnet_b200._lib import SpnetError
    shape = (1, 6, 8, 64)
    t = torch.randn(shape, device=dev())
    C = shape[-1]
    v = torch.ones(C, device=dev())
    with pytest.raises(SpnetError):  # zo with a BN'd input: not a combination any engine runs
        ops.dwconv3x3_bwd_fused(t, t, torch.zeros(3, 3, C, device=dev()), torch.zeros(3, 3, C, device=dev()),
                                in_a=v, in_b=v, relu=1, zo=t, zo_mean=v, zo_rstd=v, zo_stats=ops.stats_alloc(2 * C, dev()))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(4, 93, 125, 128), (8, 47, 63, 256), (8, 24, 32, 728), (64, 12, 16, 1024), (2, 7, 9, 24)])
def test_maxpool_bwd_bn_sums(dtype, shape):
    ops = _ops()
    torch.manual_seed(12)
    B, H, W, C = shape
    OH, OW = (H + 1) // 2, (W + 1) // 2
    z = torch.randn(shape, device=dev()).to(dtype)
    a = torch.randn(C, device=dev())
    b = torch.randn(C, device=dev()) * 0.2
    argmax = torch.empty(B, OH, OW, C, device=dev(), dtype=torch.uint8)
    ops.maxpool3s2_add_fwd(z, a, b, argmax=argmax)
    g = torch.randn(B, OH, OW, C, device=dev()).to(dtype)
    mean = torch.randn(C, device=dev()) * 0.2
    rstd = torch.rand(C, device=dev()) + 0.5
    st = ops.stats_alloc(2 * C, dev())
    gin = ops.maxpool3s2_bwd(g, argmax, H, W, z=z, mean=mean, rstd=rstd, stats=st)
    ref = ops.maxpool3s2_bwd(g, argmax, H, W)
    st_ref = ops.stats_alloc(2 * C, dev())
    ops.bn_bwd_reduce(ref, z, mean, rstd, st_ref)
    torch.cuda.synchronize()
    assert torch.equal(gin, ref)
    check_sums(ops, st, st_ref, gin, z, mean, rstd)
