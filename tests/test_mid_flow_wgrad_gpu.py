"""The 24 middle-flow pointwise weight gradients of the Xception engine are one batched GEMM over the layers' stacked
depthwise outputs t_i (mid_t) and BatchNorm-backward outputs dz_i (mid_dz). Each layer's M = B*mh*mw rows are padded to
the GEMM's k-block (64 rows bf16, 16 fp32), so that the batched route runs at every size. At sizes that need the padding,
every gradient must equal t_i^T dz_i over the layer's M real rows and the pad rows must stay zero, also when fresh
activation buffers are filled with NaN (SPNET_B200_POISON)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype,H,W,B", [("bf16", 96, 128, 4), ("fp32", 131, 163, 3)])   # M = 48 and 60 rows -> 64
def test_padded_middle_flow_weight_gradients(monkeypatch, dtype, H, W, B):
    monkeypatch.setenv("SPNET_B200_POISON", "1")
    from spnet_b200 import arch
    from spnet_b200.engine import XceptionSPNetEngine
    from spnet_b200.selfcheck import make_case
    w, x, yt = make_case(H, W, B, seed=13)
    eng = XceptionSPNetEngine(H, W, B, dtype=dtype, weights=w, dropout_rate=0.0)
    eng.load_batch(x, yt)
    eng.grad_hook = lambda e: None   # stop before Adam: eng.g holds the step's gradients
    eng.train_step(lr=1e-4)
    torch.cuda.synchronize()
    mh, mw = eng.shapes["middle"]
    M = B * mh * mw
    assert M % (64 if dtype == "bf16" else 16) != 0
    t_all, dz_all = eng.mid_t.view(24, -1, 728), eng.mid_dz.view(24, -1, 728)
    assert not t_all[:, M:].any() and not dz_all[:, M:].any()
    names = ["block%d_sepconv%d/pointwise_kernel" % (b, j) for b in arch.MIDDLE_BLOCKS for j in (1, 2, 3)]
    for i, k in enumerate(names):
        t, dz = t_all[i, :M].double(), dz_all[i, :M].double()
        assert torch.isfinite(t).all() and torch.isfinite(dz).all() and dz.abs().max() > 0, k
        ref = t.t() @ dz
        mag = t.abs().t() @ dz.abs()
        got = eng.g[k].view(728, 728).double()
        # fp32 accumulation of M products (exact products in bf16): at most M rounding errors of mag each
        assert bool(((got - ref).abs() <= 1e-5 * mag + 1e-30).all()), (k, float((got - ref).abs().max()))
