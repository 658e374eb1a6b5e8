"""LANCZOS resize tables (ops.lanczos_tables) against Pillow, and the deferred-resize loaders of utils, on the CPU.

The device kernel (csrc/resize.cu) runs two integer passes over these tables; `_resize_np` restates those passes in
numpy, so equality with Image.resize here pins the arithmetic the kernel implements (tests/test_resize_gpu.py then
checks the kernel against the same Pillow bytes)."""
import numpy as np
import pytest
from PIL import Image

SIZE_PAIRS = [((384, 512), (331, 331)), ((384, 512), (32, 32)), ((480, 640), (331, 331)), ((37, 53), (331, 331)),
              ((331, 331), (331, 331)), ((384, 512), (300, 200))]


def _pass_np(src, bounds, coeffs):
    """One 8-bit pass of Pillow's resample along the last axis: int32 accumulation from 2^21, >> 22, clip to uint8."""
    acc = np.full(src.shape[:-1] + (bounds.shape[0],), 1 << 21, np.int64)
    for k in range(coeffs.shape[1]):
        idx = np.minimum(bounds[:, 0] + k, src.shape[-1] - 1)
        acc += src[..., idx].astype(np.int64) * np.where(k < bounds[:, 1], coeffs[:, k], 0)
    assert np.abs(acc).max() < 2 ** 31  # Pillow and the kernel accumulate in int32
    return np.clip(acc >> 22, 0, 255).astype(np.uint8)


def _resize_np(frame, OH, OW):
    from spnet_b200 import ops
    H, W = frame.shape
    xb, xc = ops.lanczos_tables(W, OW)
    yb, yc = ops.lanczos_tables(H, OH)
    mid = _pass_np(frame, xb, xc)                 # horizontal first, clipped to uint8
    return _pass_np(mid.T, yb, yc).T              # then vertical on the uint8 intermediate


def _pil(frame, OH, OW):
    rgb = Image.fromarray(frame).convert("RGB")
    return np.asarray(rgb.resize((OW, OH), Image.LANCZOS))[:, :, 0]


def _frames(H, W):
    rng = np.random.default_rng(H * 1000 + W)
    yy, xx = np.mgrid[:H, :W]
    sparse = np.where(rng.random((H, W)) < 0.02, 255, 0).astype(np.uint8)
    return {"random": rng.integers(0, 256, (H, W), dtype=np.uint8), "sparse": sparse,
            "checker": (((yy + xx) & 1) * 255).astype(np.uint8), "zeros": np.zeros((H, W), np.uint8),
            "full": np.full((H, W), 255, np.uint8)}


@pytest.mark.parametrize("src,dst", SIZE_PAIRS, ids=lambda p: "%dx%d" % p)
def test_tables_reproduce_pillow_lanczos(src, dst):
    for name, f in _frames(*src).items():
        np.testing.assert_array_equal(_resize_np(f, *dst), _pil(f, *dst), err_msg=name)


def test_table_shapes_and_weights():
    from spnet_b200 import ops
    xb, xc = ops.lanczos_tables(512, 331)
    yb, yc = ops.lanczos_tables(384, 331)
    assert xc.shape == (331, 11) and yc.shape == (331, 9)
    assert xb.dtype == xc.dtype == np.int32
    assert (xb[:, 0] >= 0).all() and (xb.sum(axis=1) <= 512).all() and (np.diff(xb[:, 0]) >= 0).all()
    for b, c in ((xb, xc), (yb, yc)):
        assert (np.abs(c.sum(axis=1) - (1 << 22)) <= c.shape[1]).all()     # each row sums to ~1.0 in 2^-22 units
        assert (c[np.arange(c.shape[1])[None, :] >= b[:, 1:2]] == 0).all()  # zero past each row's tap count
    ib, ic = ops.lanczos_tables(331, 331)  # same size: exact identity
    assert (ib[:, 0] + np.argmax(ic, axis=1) == np.arange(331)).all() and (ic.max(axis=1) == 1 << 22).all()
    assert (ic.sum(axis=1) == 1 << 22).all()
    with pytest.raises(ValueError):
        ops.lanczos_tables(0, 331)


def _write_pngs(tmp_path, n, odd_one=None):
    from spnet_b200 import fake_espi
    files = []
    for i in range(n):
        img, _ = fake_espi.make_frame(40 + i)
        img = img.reshape(img.shape[0], img.shape[1])
        if i == odd_one:
            img = np.asarray(Image.fromarray(img).resize((500, 380)))
        p = tmp_path / ("steelpan_%07d.png" % i)
        Image.fromarray(img).save(p)
        files.append(str(p))
    return files


def test_build_and_stream_defer_resize_give_native_frames(tmp_path):
    from spnet_b200 import utils
    files = _write_pngs(tmp_path, 5)
    X, dims = utils.build_X(5, files, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True)
    assert X.shape == (5, 384, 512, 1) and X.dtype == np.uint8 and tuple(dims) == (384, 512, 3)
    for i, f in enumerate(files):
        np.testing.assert_array_equal(X[i, :, :, 0], np.asarray(Image.open(f).convert("RGB"))[:, :, 0])
    resized, rdims = utils.build_X(5, files, force_dim=331, grayscale=True, raw_u8=True)
    assert tuple(rdims) == (331, 331, 3)
    for i in range(5):  # what the device resize has to reproduce
        np.testing.assert_array_equal(_resize_np(X[i, :, :, 0], 331, 331), resized[i, :, :, 0])
    chunks = list(utils.stream_X(files, 2, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True))
    assert [lo for lo, _ in chunks] == [0, 2, 4]
    np.testing.assert_array_equal(np.concatenate([c for _, c in chunks]), X)


def test_defer_resize_falls_back_when_sizes_differ(tmp_path):
    from spnet_b200 import utils
    files = _write_pngs(tmp_path, 5, odd_one=3)
    ref, ref_dims = utils.build_X(5, files, force_dim=331, grayscale=True, raw_u8=True)
    X, dims = utils.build_X(5, files, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True)
    assert X.shape == (5, 331, 331, 1) and tuple(dims) == tuple(ref_dims)
    np.testing.assert_array_equal(X, ref)
    chunks = list(utils.stream_X(files, 2, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True))
    assert [c.shape[1:3] for _, c in chunks] == [(384, 512), (331, 331), (384, 512)]  # only the ragged chunk falls back
    np.testing.assert_array_equal(chunks[1][1], ref[2:4])
    # without raw_u8 or grayscale the flag changes nothing
    Xf, _ = utils.build_X(2, files, force_dim=331, grayscale=True, defer_resize=True)
    np.testing.assert_array_equal(Xf, utils.build_X(2, files, force_dim=331, grayscale=True)[0])
