"""The host half of the device PNG route: the container parser (spnet_b200/png.py) against Pillow- and cv2-written
frames and every feature it must leave to Pillow, and the DEFLATE core of the kernel (csrc/inflate.cuh) built for the
host under AddressSanitizer and UBSan, against zlib over valid, malformed and corrupted streams."""
import io
import os
import random
import shutil
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest
from PIL import Image

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import png_corpus as pc  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def _fake_espi(seed):
    from spnet_b200 import fake_espi
    img, _ = fake_espi.make_frame(seed)
    return img.reshape(img.shape[0], img.shape[1])


def _pil_bytes(img, **kw):
    f = io.BytesIO()
    img.save(f, format="PNG", **kw)
    return f.getvalue()


def _channel0(data):
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))[:, :, 0]


def _raw_channel0(parsed):
    """Inflate + un-filter in numpy (zlib as the reference) -> channel 0, to check what parse() hands the kernel."""
    H, W, bpp, z = parsed
    raw = np.frombuffer(zlib.decompress(z), np.uint8).reshape(H, 1 + W * bpp)
    out = np.zeros((H, W * bpp), np.int32)
    for y in range(H):
        ft, x = raw[y, 0], raw[y, 1:].astype(np.int32)
        up = out[y - 1] if y else np.zeros(W * bpp, np.int32)
        for i in range(W * bpp):
            left = out[y, i - bpp] if i >= bpp else 0
            ul = up[i - bpp] if i >= bpp else 0
            pred = [0, left, up[i], (left + up[i]) >> 1, int(pc._paeth(np.int32(left), np.int32(up[i]), np.int32(ul)))][ft]
            out[y, i] = (x[i] + pred) & 255
    return out[:, ::bpp].astype(np.uint8)


def test_parser_accepts_pillow_and_cv2_frames():
    from spnet_b200 import png
    img = _fake_espi(11)
    data = _pil_bytes(Image.fromarray(img))
    p = png.parse(data)
    assert p is not None and p[:3] == (384, 512, 1)
    assert zlib.decompress(p[3])[0] == 0  # Pillow writes filter type 0
    cv2 = pytest.importorskip("cv2")
    ok, enc = cv2.imencode(".png", img)
    assert ok
    p = png.parse(enc.tobytes())
    assert p is not None and p[:3] == (384, 512, 1)
    assert enc.tobytes().count(b"IDAT") > 2  # cv2 splits the stream over many chunks


@pytest.mark.parametrize("colour", [0, 2, 4, 6])
def test_parser_output_is_what_pillow_decodes(colour):
    from spnet_b200 import png
    rng = np.random.default_rng(colour)
    px = rng.integers(0, 256, (9, 13, pc.BPP[colour]), dtype=np.uint8)
    data = pc.png(px, colour, filters=[y % 5 for y in range(9)], idat_sizes=[1, 0, 7],
                  extra=[pc.chunk(b"gAMA", struct.pack(">I", 45455)), pc.chunk(b"pHYs", b"\0" * 9)])
    p = png.parse(data)
    assert p is not None and p[:3] == (9, 13, pc.BPP[colour])
    np.testing.assert_array_equal(_raw_channel0(p), _channel0(data))


def _excluded():
    img = _fake_espi(12)[:40, :48]
    good = pc.png(img[:, :, None], 0, idat_sizes=[300])
    idat_at = good.index(b"IDAT") - 4
    cases = {
        "palette": _pil_bytes(Image.fromarray(img).convert("P")),
        "trns": _pil_bytes(Image.fromarray(img), transparency=0),
        "16bit": _pil_bytes(Image.fromarray(img.astype(np.uint16) * 257)),
        "interlaced": pc.png(img[:, :, None], 0, interlace=True),
        "unknown_chunk": pc.png(img[:, :, None], 0, extra=[pc.chunk(b"tEXt", b"k\0v")]),
        "private_chunk": pc.png(img[:, :, None], 0, extra=[pc.chunk(b"zzZz", b"x")]),
        "idat_not_consecutive": good[:idat_at] + good[idat_at:idat_at + 312] + pc.chunk(b"gAMA", struct.pack(">I", 45455))
        + good[idat_at + 312:],
        "bmp": (lambda f: (Image.fromarray(img).save(f, format="BMP"), f.getvalue())[1])(io.BytesIO()),
        "no_iend": good[:-12],
        "truncated": good[:len(good) // 2],
        "not_png": b"hello",
    }
    # whitelisted chunks at any length but their own (Pillow raises on some short ones), or after the image data
    for ctype, size in (("gAMA", 4), ("cHRM", 32), ("sRGB", 1), ("pHYs", 9), ("tIME", 7)):
        for k in (0, size - 1, size + 1):
            cases["%s_%d_bytes" % (ctype, k)] = pc.png(img[:, :, None], 0, extra=[pc.chunk(ctype.encode(), b"\1" * k)])
        cases[ctype + "_after_idat"] = good[:-12] + pc.chunk(ctype.encode(), b"\1" * size) + good[-12:]
    cases["iend_not_empty"] = good[:-12] + pc.chunk(b"IEND", b"x")
    for name, pos in (("ihdr", 8), ("idat", idat_at), ("iend", len(good) - 12)):
        length = struct.unpack_from(">I", good, pos)[0]
        crc_at = pos + 8 + length
        cases["bad_crc_" + name] = good[:crc_at] + bytes([good[crc_at] ^ 1]) + good[crc_at + 1:]
    return good, cases


def test_parser_sends_excluded_files_to_the_host_route():
    from spnet_b200 import png
    good, cases = _excluded()
    assert png.parse(good) is not None
    img = _fake_espi(12)[:40, :48, None]
    whitelisted = [pc.chunk(t, b"\1" * k) for t, k in ((b"gAMA", 4), (b"cHRM", 32), (b"sRGB", 1), (b"pHYs", 9), (b"tIME", 7))]
    assert png.parse(pc.png(img, 0, extra=whitelisted)) is not None
    for name, data in cases.items():
        assert png.parse(data) is None, name


def test_device_route_raises_where_pillow_raises_on_short_chunks(tmp_path):
    """Files whose short ancillary chunks make Pillow raise must not decode on the device route: parse() refuses them,
    read() reports the file (or its size), and the host route's exception is what the loaders raise."""
    from spnet_b200 import png, utils
    img = _fake_espi(12)[:40, :48, None]
    for ctype, k in ((b"sRGB", 0), (b"pHYs", 3), (b"gAMA", 2), (b"cHRM", 5)):
        data = pc.png(img, 0, extra=[pc.chunk(ctype, b"\1" * k)])
        f = tmp_path / (ctype.decode() + ".png")
        f.write_bytes(data)
        assert png.parse(data) is None
        with pytest.raises(Exception):
            utils._load_one((str(f), None, True, True))
        assert png.read(str(f)) in (None, (40, 48))


def test_read_reports_host_route_files_by_their_size(tmp_path):
    """read() returns the size of a file left to PIL (the loaders check sizes before decoding anything on the host),
    and None for a file PIL cannot open or one that does not exist."""
    from spnet_b200 import png
    _, cases = _excluded()
    for name in ("palette", "interlaced", "bmp", "bad_crc_idat", "truncated"):
        f = tmp_path / (name + ".png")
        f.write_bytes(cases[name])
        assert png.read(str(f)) == (40, 48), name
    f = tmp_path / "not.png"
    f.write_bytes(cases["not_png"])
    assert png.read(str(f)) is None
    assert png.read(str(tmp_path / "missing.png")) is None


# ---------------------------------------------------------------------------------------------- inflate core on the host
@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    exe = str(tmp_path_factory.mktemp("inflate") / "inflate_harness")
    subprocess.run([cxx, "-std=c++17", "-O1", "-g", "-fno-omit-frame-pointer", "-fsanitize=address,undefined",
                    "-fno-sanitize-recover=all", os.path.join(HERE, "inflate_harness.cpp"), "-o", exe], check=True)
    return exe


def _run(exe, cases, tmp_path, window=8192):
    """cases: [(stream, capacity)] -> [(status, output bytes)] from the sanitizer build."""
    src, dst = tmp_path / "cases.bin", tmp_path / "results.bin"
    with open(src, "wb") as f:
        for z, cap in cases:
            f.write(struct.pack("<QQ", len(z), cap) + z)
    r = subprocess.run([exe, str(src), str(dst), str(window)], capture_output=True, text=True,
                       env=dict(os.environ, ASAN_OPTIONS="detect_leaks=1:halt_on_error=1"))
    assert r.returncode == 0 and not r.stderr, r.stderr[-4000:]
    out, data, pos = [], open(dst, "rb").read(), 0
    for _ in cases:
        st, n = struct.unpack_from("<iQ", data, pos)
        pos += 12
        out.append((st, data[pos:pos + n]))
        pos += n
    assert pos == len(data)
    return out


def _payloads():
    rng = np.random.default_rng(5)
    img = _fake_espi(13)
    text = b"".join(b"frame %d of the steelpan set; " % i for i in range(40000))
    return {"empty": b"", "one": b"\x07", "random_70k": rng.integers(0, 256, 70000, dtype=np.uint8).tobytes(),
            "mixed_1m": (img.tobytes() * 6)[:600000] + text[:448576],
            "png_rows": pc.filter_rows(img[:, :, None], [y % 5 for y in range(img.shape[0])])}


STRATEGIES = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]


@pytest.mark.parametrize("window", [8192, 256])
def test_inflate_core_equals_zlib_on_valid_streams(harness, tmp_path, window):
    cases, want = [], []
    for data in _payloads().values():
        for level in range(10):
            for strategy in STRATEGIES:
                c = zlib.compressobj(level, zlib.DEFLATED, 15, 9, strategy)
                z = c.compress(data) + c.flush()
                cases.append((z, len(data)))
                want.append(data)
    for z in pc.single_code_streams().values():
        cases.append((z, 16))
        want.append(zlib.decompress(z))
    got = _run(harness, cases, tmp_path, window)
    for (st, out), w in zip(got, want):
        assert st == 0 and out == w


def test_inflate_core_rejects_every_malformed_class(harness, tmp_path):
    streams = pc.malformed_streams()
    for name, z in streams.items():
        with pytest.raises(zlib.error):
            zlib.decompress(z)
    data = bytes(range(256)) * 8
    exact = zlib.compress(data)
    cases = [(z, 1 << 16) for z in streams.values()] + [(exact, len(data) - 1), (exact + b"\0", len(data))]
    got = _run(harness, cases, tmp_path)
    names = list(streams) + ["longer_than_capacity", "bytes_after_trailer"]
    for name, (st, _) in zip(names, got):
        assert st < 0, name
    assert _run(harness, [(exact, len(data))], tmp_path) == [(0, data)]


def test_inflate_core_on_corrupted_streams(harness, tmp_path):
    """Seeded truncations and bit flips: wherever zlib raises the core reports an error, and wherever the core succeeds
    its bytes are zlib's. Any out-of-bounds access is a sanitizer report, which fails the run."""
    rnd = random.Random(1234)
    p = _payloads()
    sources = [zlib.compress(p["png_rows"][:6000], lvl) for lvl in (1, 6, 9)]
    sources += [pc.compress(p["mixed_1m"][:5000], "fixed"), pc.compress(p["mixed_1m"][:5000], "stored")]
    cases = []
    for z in sources:
        for _ in range(60):
            cut = rnd.randrange(len(z))
            cases.append(z[:cut])
        for _ in range(240):
            b = bytearray(z)
            for _ in range(rnd.choice((1, 1, 2, 4))):
                i = rnd.randrange(len(b))
                b[i] ^= 1 << rnd.randrange(8)
            cases.append(bytes(b))
    cap = 1 << 16
    got = _run(harness, [(z, cap) for z in cases], tmp_path)
    for z, (st, out) in zip(cases, got):
        try:
            ref = zlib.decompress(z)
        except zlib.error:
            assert st < 0
            continue
        if st == 0:
            assert out == ref
