"""LANCZOS resize on the device (csrc/resize.cu, ops.resize_lanczos_u8) against Pillow, and the routes built on it:
SPNetModel.predict(resize=True) and predict_network's deferred resize at the monolithic 331x331 default."""
import numpy as np
import pytest
from PIL import Image

pytestmark = pytest.mark.gpu

SIZE_PAIRS = [((384, 512), (331, 331)), ((384, 512), (32, 32)), ((480, 640), (331, 331)), ((37, 53), (331, 331)),
              ((331, 331), (331, 331)), ((384, 512), (300, 200))]


def _pil(frame, OH, OW):
    return np.asarray(Image.fromarray(frame).convert("RGB").resize((OW, OH), Image.LANCZOS))[:, :, 0]


def _frames(n, H, W, seed):
    rng = np.random.default_rng(seed)
    out = rng.integers(0, 256, (n, H, W), dtype=np.uint8)
    yy, xx = np.mgrid[:H, :W]
    kinds = [np.where(rng.random((H, W)) < 0.02, 255, 0), ((yy + xx) & 1) * 255, np.zeros((H, W)), np.full((H, W), 255)]
    for i in range(min(n - 1, len(kinds))):
        out[i + 1] = kinds[i]
    return out


@pytest.mark.parametrize("n", [1, 3, 64])
@pytest.mark.parametrize("src,dst", SIZE_PAIRS, ids=lambda p: "%dx%d" % p)
def test_kernel_equals_lut_of_pillow(src, dst, n):
    import torch
    from spnet_b200 import ops
    x = _frames(n, *src, seed=n * 7 + src[0])
    got = ops.resize_lanczos_u8(torch.from_numpy(x).cuda(), *dst).cpu().numpy()
    lut = ops._u8_lut("cpu").numpy()
    want = lut[np.stack([_pil(f, *dst) for f in x])]
    assert got.shape == (n,) + dst
    np.testing.assert_array_equal(got, want)
    again = ops.resize_lanczos_u8(torch.from_numpy(x[:, :, :, None]).cuda(), *dst)  # [n, H, W, 1] takes the same path
    np.testing.assert_array_equal(again.cpu().numpy(), want)


def test_bad_arguments_raise_before_launch():
    import torch
    from spnet_b200 import ops
    from spnet_b200._lib import SpnetError, lib
    x = torch.zeros((2, 384, 512), dtype=torch.uint8, device="cuda")
    out = torch.empty((2, 331, 331), device="cuda")
    xb, xc = (torch.from_numpy(a).cuda() for a in ops.lanczos_tables(512, 331))
    yb, yc = (torch.from_numpy(a).cuda() for a in ops.lanczos_tables(384, 331))
    lut = ops._u8_lut(x.device)
    s = torch.cuda.current_stream().cuda_stream
    good = [x.data_ptr(), 2, 384, 512, xb.data_ptr(), xc.data_ptr(), 11, yb.data_ptr(), yc.data_ptr(), 9, lut.data_ptr(),
            out.data_ptr(), 331, 331, s]
    L = lib()
    L.resize_lanczos_u8(*good)
    torch.cuda.synchronize()
    for i, v in [(0, None), (4, None), (10, None), (11, None), (1, 0), (1, 70000), (2, 0), (3, -1), (6, 0), (9, 0),
                 (12, 0), (13, 0), (13, 1 << 20)]:  # the last: one band's rows do not fit shared memory
        bad = list(good)
        bad[i] = v
        before = L.launches
        with pytest.raises(SpnetError, match="resize_lanczos_u8"):
            L.resize_lanczos_u8(*bad)
        assert L.launches == before
    torch.cuda.synchronize()  # nothing was launched, so nothing can have faulted
    with pytest.raises(TypeError):
        ops.resize_lanczos_u8(torch.zeros((1, 8, 8), device="cuda"), 4, 4)
    with pytest.raises(ValueError):
        ops.resize_lanczos_u8(x, 331, 331, out=torch.empty((1, 331, 331), device="cuda"))


def _write_pngs(path, n, seed, odd_one=None):
    from spnet_b200 import fake_espi
    path.mkdir(exist_ok=True)
    for i in range(n):
        img, _ = fake_espi.make_frame(seed + i)
        img = img.reshape(img.shape[0], img.shape[1])
        if i == odd_one:
            img = np.asarray(Image.fromarray(img).resize((500, 380)))
        Image.fromarray(img).save(path / ("steelpan_%07d.png" % i))
    return sorted(str(p) for p in path.glob("*.png"))


@pytest.fixture
def model331():
    import spnet.config as cf
    from spnet import models
    cf.model_type, cf.compute_dtype = "monolithic", "bf16"
    model, _ = models.setup_model(np.zeros((1, 331, 331, 1), np.float32), 576, try_checkpoint=False, freeze_fac=0.0,
                                  quick_setup=True)
    return model


def test_predict_resize_equals_host_resized(tmp_path, model331):
    import torch
    from spnet import utils
    files = _write_pngs(tmp_path, 5, 700)
    native, _ = utils.build_X(5, files, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True)
    host, _ = utils.build_X(5, files, force_dim=331, grayscale=True, raw_u8=True)
    assert native.shape == (5, 384, 512, 1) and host.shape == (5, 331, 331, 1)
    for bs in (2, 5):  # 2: a ragged last batch
        want = model331.predict(host, batch_size=bs)
        np.testing.assert_array_equal(model331.predict(native, batch_size=bs, resize=True), want)
        np.testing.assert_array_equal(model331.predict(torch.from_numpy(native).cuda(), batch_size=bs, resize=True), want)
        np.testing.assert_array_equal(model331.predict(torch.from_numpy(native).pin_memory(), batch_size=bs, resize=True), want)
        # frames already at the model's size pass through resize=True unchanged
        np.testing.assert_array_equal(model331.predict(host, batch_size=bs, resize=True), want)
        np.testing.assert_array_equal(model331.predict(torch.from_numpy(host).cuda(), batch_size=bs), want)
    with pytest.raises(ValueError):
        model331.predict(native.astype(np.float32), resize=True)
    with pytest.raises(ValueError):
        model331.predict(torch.from_numpy(native).float().cuda(), resize=True)
    with pytest.raises(ValueError):
        model331.predict(native)  # 384x512 frames for a 331x331 model without resize=True


def test_predict_resize_without_graph(tmp_path, model331, monkeypatch):
    import torch
    from spnet import utils
    files = _write_pngs(tmp_path, 3, 720)
    native, _ = utils.build_X(3, files, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True)
    host, _ = utils.build_X(3, files, force_dim=331, grayscale=True, raw_u8=True)
    monkeypatch.setenv("SPNET_B200_NO_GRAPH", "1")
    want = model331.predict(host, batch_size=2)
    np.testing.assert_array_equal(model331.predict(native, batch_size=2, resize=True), want)
    np.testing.assert_array_equal(model331.predict(torch.from_numpy(native).cuda(), batch_size=2, resize=True), want)


@pytest.mark.parametrize("odd_one", [None, 2])
def test_predict_network_deferred_resize_writes_host_route_csv(tmp_path, model331, monkeypatch, odd_one):
    """predict_network at the monolithic default (bf16, batch 2, no PNGs): the deferred route (uint8 frames at their
    decoded size, resized on the GPU) writes the CSV of the host route (PIL resize, host normalisation) byte for byte,
    whole-set and --stream; with one frame of another size the loaders fall back to the host resize."""
    import predict_spnet
    from spnet_b200 import ops
    _write_pngs(tmp_path / "frames", 6, 800, odd_one=odd_one)
    wpath = str(tmp_path / "weights.hdf5")
    model331.save_weights(wpath)
    calls = []
    real = ops.resize_lanczos_u8
    monkeypatch.setattr(ops, "resize_lanczos_u8", lambda *a, **k: calls.append(a[0].shape) or real(*a, **k))
    data = str(tmp_path / "frames")

    def csv(name, **kw):
        log_dir = str(tmp_path / name) + "/"
        predict_spnet.predict_network(weights_file=wpath, datapath=data, log_dir=log_dir, batch_size=2, draw_images=False,
                                      **kw)
        return open(log_dir + "hawley_spnet.csv").read()

    host = csv("host", raw_u8=False)
    assert not calls
    assert csv("device") == host
    assert len(calls) == (0 if odd_one is not None else 3)
    calls.clear()
    assert csv("device_stream", stream_chunk=4) == host
    assert len(calls) == (1 if odd_one is not None else 3)  # chunk [0, 4) holds the odd frame and falls back
    log_dir = str(tmp_path / "passed_model") + "/"  # a model handed over by train_spnet.py takes the same route
    predict_spnet.predict_network(model=model331, datapath=data, log_dir=log_dir, batch_size=2, draw_images=False)
    assert open(log_dir + "hawley_spnet.csv").read() == host
