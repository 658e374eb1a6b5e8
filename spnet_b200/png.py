"""PNG frames decoded on the device (csrc/png.cu, ops.png_decode_u8), byte for byte what the host route decodes:
channel 0 of np.asarray(Image.open(f).convert("RGB")), i.e. utils._load_one((f, None, True, True)).

The host reads each file and walks its chunks (parse); the IDAT payloads of the accepted frames travel to the GPU in
one copy per launch and are inflated and un-filtered there. Every file outside the subset parse accepts, and every
frame the kernel rejects, is decoded by utils._load_one. Where any of that host work fails, Decoder.frames gives up
and the caller runs the host route over the same files, so the bytes - or the exception raised - are the host route's.

Accepted: signature, IHDR first, bit depth 8, colour type 0 / 2 / 4 / 6, compression / filter / interlace 0, at most
MAX_WIDTH x MAX_PIXELS, every chunk CRC correct, then only ANCILLARY chunks at their specified length, consecutive IDAT
chunks and an empty IEND. The ANCILLARY chunks carry no pixel data; Pillow reads them while opening the file and raises
on some of them when they are short, hence the exact lengths. Palette, tRNS, iCCP, text, APNG, 16-bit and interlaced
PNGs, chunks after the image data, other formats and damaged files take the host route.
"""
import io
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

SIGNATURE = b"\x89PNG\r\n\x1a\n"
ANCILLARY = {b"gAMA": 4, b"cHRM": 32, b"sRGB": 1, b"pHYs": 9, b"tIME": 7}  # chunk type -> its length (PNG spec)
MAX_WIDTH = 8192  # the kernel keeps one row of channel 0 in shared memory (csrc/png.cu kWindow)
MAX_PIXELS = 1 << 26  # well under Pillow's decompression-bomb limit
_BPP = {0: 1, 4: 2, 2: 3, 6: 4}  # colour type -> bytes per pixel at bit depth 8
FRAMES_PER_LAUNCH = 2048


def parse(data):
    """PNG file bytes -> (H, W, bpp, zlib stream of the concatenated IDAT payloads), or None when the device route
    does not take the file."""
    if data[:8] != SIGNATURE:
        return None
    pos, n = 8, len(data)
    hdr, idat = None, []
    while True:
        if pos + 12 > n:
            return None  # no IEND
        length, = struct.unpack_from(">I", data, pos)
        ctype = data[pos + 4:pos + 8]
        end = pos + 12 + length
        if end > n:
            return None
        body = data[pos + 8:end - 4]
        if zlib.crc32(body, zlib.crc32(ctype)) != struct.unpack_from(">I", data, end - 4)[0]:
            return None
        if hdr is None:
            if ctype != b"IHDR" or length != 13:
                return None
            W, H, depth, colour, comp, filt, interlace = struct.unpack(">IIBBBBB", body)
            if (depth != 8 or colour not in _BPP or comp or filt or interlace or not 0 < W <= MAX_WIDTH
                    or not 0 < H or H * W > MAX_PIXELS):
                return None
            hdr = (H, W, _BPP[colour])
        elif ctype == b"IDAT":
            idat.append(body)
        elif ctype == b"IEND":
            return hdr + (b"".join(idat),) if idat and length == 0 else None
        elif idat or ANCILLARY.get(ctype) != length:
            return None  # after the image data only IDAT and IEND; before it only ANCILLARY at their lengths
        pos = end


def read(filename):
    """One file for the device route, on a worker thread: parse()'s tuple; (H, W) of a file the device route leaves
    to PIL; None when the file cannot be read or PIL cannot open it (the host route then raises what it raises)."""
    try:
        with open(filename, "rb") as f:
            data = f.read()
        p = parse(data)
        if p is not None:
            return p
        from PIL import Image
        w, h = Image.open(io.BytesIO(data)).size
        return (h, w)
    except Exception:
        return None


class Decoder:
    """Device decoding for the current CUDA stream, used from one thread and kept for one loader call (build_X, or one
    stream_X generator), so its pinned memory is released with it. The IDAT payloads of a launch are packed into one of
    two pinned staging buffers and sent with one asynchronous copy; a buffer is refilled only after the event recorded
    behind its copy has completed, and grows only to the largest launch it has carried."""

    def __init__(self):
        self._stage = [None, None]
        self._copied = [None, None]
        self._turn = 0

    def frames(self, files, items, device):
        """items[i] = read(files[i]). Returns the frames as CUDA uint8 [n, H, W, 1] on `device`, equal to the host
        route's, or None - before any host decoding where the headers tell - when they differ in size, a file cannot
        be opened, or PIL fails on a file it decodes here. The caller then runs the host route."""
        import torch
        from . import utils
        if any(it is None for it in items) or len({it[:2] for it in items}) != 1:
            return None
        H, W = items[0][:2]
        n = len(items)
        X = torch.empty((n, H, W, 1), dtype=torch.uint8, device=device)
        groups, checks = {}, []
        for i, it in enumerate(items):
            if len(it) == 4:
                groups.setdefault(it[2], []).append(i)
        for bpp, idx in groups.items():
            for a in range(0, len(idx), FRAMES_PER_LAUNCH):
                part = idx[a:a + FRAMES_PER_LAUNCH]
                if part[-1] - part[0] == len(part) - 1:  # consecutive frames: decode in place
                    checks.append((part, self._launch([items[i][3] for i in part], H, W, bpp, X[part[0]:part[-1] + 1])))
                else:
                    tmp = torch.empty((len(part), H, W, 1), dtype=torch.uint8, device=device)
                    checks.append((part, self._launch([items[i][3] for i in part], H, W, bpp, tmp)))
                    X.index_copy_(0, torch.tensor(part, device=device), tmp)
        on_host = [i for i, it in enumerate(items) if len(it) == 2]
        for part, status in checks:
            on_host += [part[j] for j in np.flatnonzero(status.cpu().numpy())]
        if on_host:
            try:
                with ThreadPoolExecutor(min(len(on_host), 64)) as ex:
                    arrs = list(ex.map(utils._load_one, [(files[i], None, True, True) for i in on_host]))
            except Exception:
                return None
            for i, arr in zip(on_host, arrs):
                X[i].copy_(torch.from_numpy(arr.copy()))  # PIL's array is read-only
        return X

    def _launch(self, streams, H, W, bpp, out):
        import torch
        from . import ops
        n = len(streams)
        head = 8 * (n + 1)
        offsets = np.zeros(n + 1, np.int64)
        np.cumsum([len(s) for s in streams], out=offsets[1:])
        total = head + int(offsets[-1])
        k, self._turn = self._turn, self._turn ^ 1
        if self._copied[k] is not None:
            self._copied[k].synchronize()
        if self._stage[k] is None or self._stage[k].numel() < total:
            self._stage[k] = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        host = self._stage[k].numpy()
        host[:head] = offsets.view(np.uint8)
        for s, o in zip(streams, offsets[:-1]):
            host[head + o:head + o + len(s)] = np.frombuffer(s, np.uint8)
        dev = torch.empty(total, dtype=torch.uint8, device=out.device)
        dev.copy_(self._stage[k][:total], non_blocking=True)
        self._copied[k] = torch.cuda.Event()
        self._copied[k].record()
        return ops.png_decode_u8(dev[head:], dev[:head].view(torch.int64), H, W, bpp, out)
