"""PNG decoding on the device (csrc/png.cu, ops.png_decode_u8, spnet_b200/png.py) against Pillow, and the routes built
on it: utils.build_X / stream_X(device=True) and predict_network's default path."""
import io
import os
import sys
import zlib

import numpy as np
import pytest
from PIL import Image

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import png_corpus as pc  # noqa: E402

pytestmark = pytest.mark.gpu


def _fake_espi(seed):
    from spnet_b200 import fake_espi
    img, _ = fake_espi.make_frame(seed)
    return img.reshape(img.shape[0], img.shape[1])


def _pillow(data):
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))[:, :, 0]


def _pil_png(img):
    f = io.BytesIO()
    Image.fromarray(img).save(f, format="PNG")
    return f.getvalue()


def _decode(streams, H, W, bpp, canary=False):
    """Launch png_decode_u8 over the streams; returns (out [n, H, W] numpy, status numpy), and with canary=True checks
    the guard bytes just past out and scratch."""
    import torch
    from spnet_b200 import ops
    n = len(streams)
    offsets = np.zeros(n + 1, np.int64)
    np.cumsum([len(s) for s in streams], out=offsets[1:])
    buf = torch.from_numpy(np.frombuffer(b"".join(streams) or b"\0", np.uint8).copy()).cuda()
    per = H * (1 + W * bpp)
    out_full = torch.full((n * H * W + 64,), 0xA5, dtype=torch.uint8, device="cuda")
    scratch_full = torch.full((n * per + 64,), 0x5A, dtype=torch.uint8, device="cuda")
    out = out_full[:n * H * W].view(n, H, W)
    status = ops.png_decode_u8(buf[:int(offsets[-1])] if offsets[-1] else buf[:0], torch.from_numpy(offsets).cuda(), H, W,
                               bpp, out, scratch=scratch_full[:n * per])
    if canary:
        assert bool((out_full[n * H * W:] == 0xA5).all()) and bool((scratch_full[n * per:] == 0x5A).all())
    return out.cpu().numpy(), status.cpu().numpy()


def _corpus(H, W, colour, seed):
    """Frames of one size and colour type written with every filter, IDAT split and block type."""
    from spnet_b200 import png
    rng = np.random.default_rng(seed)
    files = []
    for k, mode in enumerate(("dynamic", "fixed", "stored")):
        px = rng.integers(0, 256, (H, W, pc.BPP[colour]), dtype=np.uint8)
        if k == 0:
            px[:, :, 0] = (np.arange(W)[None, :] * 3 + np.arange(H)[:, None]) & 255  # something the filters compress
        filters = list(rng.integers(0, 5, H))
        files.append(pc.png(px, colour, filters=filters, idat_sizes=[1, 0, 5, 977], mode=mode))
    return [(png.parse(d), _pillow(d)) for d in files]


@pytest.mark.parametrize("colour", [0, 2, 4, 6])
@pytest.mark.parametrize("W", [1, 7, 512, 513])
def test_kernel_equals_pillow_written_frames(colour, W):
    for H in (1, 5, 384 if W < 513 else 37):
        frames = _corpus(H, W, colour, seed=W * 10 + colour + H)
        out, status = _decode([p[3] for p, _ in frames], H, W, pc.BPP[colour], canary=True)
        assert not status.any()
        for k, (_, want) in enumerate(frames):
            np.testing.assert_array_equal(out[k], want)


@pytest.mark.parametrize("n", [1, 3, 64, 600])
def test_kernel_equals_pillow_on_fake_espi(n):
    from spnet_b200 import png
    datas = []
    for i in range(min(n, 24)):
        img = _fake_espi(4000 + i)
        if i % 2:
            cv2 = pytest.importorskip("cv2")
            datas.append(cv2.imencode(".png", img)[1].tobytes())
        else:
            datas.append(_pil_png(img))
    streams, want = [], []
    for i in range(n):
        d = datas[i % len(datas)]
        streams.append(png.parse(d)[3])
        if i < len(datas):
            want.append(_pillow(d))
    out, status = _decode(streams, 384, 512, 1, canary=True)
    assert not status.any()
    for i in range(n):
        np.testing.assert_array_equal(out[i], want[i % len(datas)])


def test_malformed_frames_next_to_valid_ones():
    H, W = 17, 33
    rng = np.random.default_rng(3)
    px = rng.integers(0, 256, (H, W, 1), dtype=np.uint8)
    raw = pc.filter_rows(px, [y % 5 for y in range(H)])
    good = zlib.compress(raw)
    want = _pillow(pc.png(px, 0, filters=[y % 5 for y in range(H)]))
    bad_filter = bytearray(raw)
    bad_filter[(1 + W) * 4] = 5
    bad = dict(pc.malformed_streams())
    bad.update({"short": zlib.compress(raw[:-1]), "long": zlib.compress(raw + b"\0"), "filter_5": zlib.compress(bytes(bad_filter)),
                "trailing_bytes": good + b"\0", "no_adler": good[:-4], "wrong_adler": good[:-1] + bytes([good[-1] ^ 1])})
    streams, kinds = [], []
    for name, z in bad.items():
        streams += [good, z]
        kinds += [None, name]
    out, status = _decode(streams, H, W, 1, canary=True)
    codes = {"short": -4, "long": -4, "filter_5": -6, "wrong_adler": -5, "no_adler": -5, "trailing_bytes": -5, "bad_fcheck": -1,
             "cm_not_8": -1, "fdict": -1}
    for k, name in enumerate(kinds):
        if name is None:
            assert status[k] == 0
            np.testing.assert_array_equal(out[k], want)
        else:
            assert status[k] < 0, name
            if name in codes:
                assert status[k] == codes[name], name


def test_bad_arguments_raise_before_launch():
    import torch
    from spnet_b200._lib import SpnetError, lib
    z = zlib.compress(b"\0" * (8 * 9))
    streams = torch.from_numpy(np.frombuffer(z, np.uint8).copy()).cuda()
    offsets = torch.tensor([0, len(z)], dtype=torch.int64, device="cuda")
    scratch = torch.empty(8 * 9, dtype=torch.uint8, device="cuda")
    out = torch.empty((8, 8), dtype=torch.uint8, device="cuda")
    status = torch.empty(1, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    good = [streams.data_ptr(), len(z), offsets.data_ptr(), 1, 8, 8, 1, scratch.data_ptr(), 72, out.data_ptr(),
            status.data_ptr(), s]
    L = lib()
    L.png_decode_u8(*good)
    torch.cuda.synchronize()
    assert int(status[0]) == 0 and not out.any()
    for i, v in [(0, None), (2, None), (7, None), (9, None), (10, None), (1, -1), (3, 0), (4, 0), (5, 0), (5, 8193),
                 (6, 0), (6, 5), (8, 71), (8, -1)]:
        bad = list(good)
        bad[i] = v
        before = L.launches
        with pytest.raises(SpnetError, match="png_decode_u8"):
            L.png_decode_u8(*bad)
        assert L.launches == before
    torch.cuda.synchronize()


def _write_dir(path, n, seed, extra=()):
    path.mkdir(exist_ok=True)
    for i in range(n):
        Image.fromarray(_fake_espi(seed + i)).save(path / ("steelpan_%07d.png" % i))
    for name, data in extra:
        (path / name).write_bytes(data)
    return sorted(str(p) for p in path.glob("*.png"))


def test_loaders_on_device_equal_host_route(tmp_path):
    import torch
    from spnet import utils
    img = _fake_espi(77)
    extra = [("steelpan_0000002a.png", _pil_png(np.stack([img] * 3, -1)[..., :3].copy())),  # RGB frame
             ("steelpan_0000003p.png", (lambda f: (Image.fromarray(img).convert("P").save(f, format="PNG"), f.getvalue())[1])(io.BytesIO())),
             ("steelpan_0000004i.png", pc.png(img[:, :, None], 0, interlace=True))]
    files = _write_dir(tmp_path / "ok", 7, 500, extra)
    host, dims = utils.build_X(len(files), files, force_dim=None, grayscale=True, raw_u8=True)
    dev, ddims = utils.build_X(len(files), files, force_dim=None, grayscale=True, raw_u8=True, device=True)
    assert torch.is_tensor(dev) and dev.is_cuda and dev.dtype == torch.uint8 and tuple(dims) == tuple(ddims)
    np.testing.assert_array_equal(dev.cpu().numpy(), host)
    for defer in (False, True):
        parts = list(utils.stream_X(files, 4, force_dim=331 if defer else None, grayscale=True, raw_u8=True,
                                    defer_resize=defer, device=True))
        assert [lo for lo, _ in parts] == [0, 4, 8]
        np.testing.assert_array_equal(np.concatenate([x.cpu().numpy() for _, x in parts]), host)
    # one frame of another size: the call, or the chunk, returns what the host route returns
    odd = _write_dir(tmp_path / "odd", 5, 600, [("steelpan_0000001x.png", _pil_png(img[:300, :400].copy()))])
    want, _ = utils.build_X(len(odd), odd, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True)
    got, _ = utils.build_X(len(odd), odd, force_dim=331, grayscale=True, raw_u8=True, defer_resize=True, device=True)
    assert isinstance(got, np.ndarray)
    np.testing.assert_array_equal(got, want)
    # a corrupt PNG raises the host route's exception
    bad = _write_dir(tmp_path / "bad", 3, 700, [("steelpan_0000001c.png", _pil_png(img)[:20000])])
    with pytest.raises(Exception) as e:
        utils.build_X(len(bad), bad, force_dim=None, grayscale=True, raw_u8=True)
    with pytest.raises(type(e.value)):
        utils.build_X(len(bad), bad, force_dim=None, grayscale=True, raw_u8=True, device=True)
    with pytest.raises(type(e.value)):
        list(utils.stream_X(bad, 2, force_dim=None, grayscale=True, raw_u8=True, device=True))
    # a short ancillary chunk that Pillow raises on while opening the file
    short = _write_dir(tmp_path / "short", 3, 800, [("steelpan_0000001s.png", pc.png(img[:, :, None], 0,
                                                                                  extra=[pc.chunk(b"sRGB", b"")]))])
    with pytest.raises(Exception) as e:
        utils.build_X(len(short), short, force_dim=None, grayscale=True, raw_u8=True)
    with pytest.raises(type(e.value)):
        utils.build_X(len(short), short, force_dim=None, grayscale=True, raw_u8=True, device=True)
    with pytest.raises(type(e.value)):
        list(utils.stream_X(short, 2, force_dim=None, grayscale=True, raw_u8=True, device=True))


def _model(kind):
    import spnet.config as cf
    from spnet import models
    cf.model_type, cf.compute_dtype = kind, "bf16"
    shape = (1, 331, 331, 1) if kind == "monolithic" else (1, 384, 512, 1)
    model, _ = models.setup_model(np.zeros(shape, np.float32), 576, try_checkpoint=False, freeze_fac=0.0, quick_setup=True)
    return model


@pytest.mark.parametrize("kind", ["monolithic", "big"])
@pytest.mark.parametrize("odd_one", [None, 2])
def test_predict_network_device_decode_writes_host_route_csv(tmp_path, monkeypatch, kind, odd_one):
    import predict_spnet
    from spnet_b200 import png
    model = _model(kind)
    d = tmp_path / "frames"
    files = _write_dir(d, 6, 900)
    if odd_one is not None:
        Image.fromarray(_fake_espi(950)[:380, :500].copy()).save(files[odd_one])
    wpath = str(tmp_path / "weights.hdf5")
    model.save_weights(wpath)
    launches = []
    real = png.Decoder._launch
    monkeypatch.setattr(png.Decoder, "_launch", lambda self, s, *a: launches.append(len(s)) or real(self, s, *a))

    def csv(name, **kw):
        log_dir = str(tmp_path / name) + "/"
        predict_spnet.predict_network(weights_file=wpath, datapath=str(d), log_dir=log_dir, batch_size=2, draw_images=False,
                                      **kw)
        return open(log_dir + "hawley_spnet.csv").read()

    if kind == "big" and odd_one is not None:  # neither route can stack frames of two sizes at their decoded size
        with pytest.raises(ValueError):
            csv("host", raw_u8=False)
        with pytest.raises(ValueError):
            csv("device")
        with pytest.raises(ValueError):
            csv("device_stream", stream_chunk=4)
        assert not launches
        return
    host = csv("host", raw_u8=False)
    assert not launches
    assert csv("device") == host
    assert launches == ([] if odd_one is not None else [6])
    launches.clear()
    assert csv("device_stream", stream_chunk=4) == host
    assert launches == ([2] if odd_one is not None else [4, 2])
