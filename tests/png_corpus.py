"""PNG files and zlib streams written byte by byte for the PNG decoder tests (test_png_host.py, test_png_gpu.py): a
small PNG writer with a chosen filter per row, IDAT split and compression, and a bit writer for hand-made DEFLATE
blocks, valid and malformed."""
import struct
import zlib

import numpy as np

BPP = {0: 1, 4: 2, 2: 3, 6: 4}


def chunk(ctype, body, crc=None):
    c = zlib.crc32(body, zlib.crc32(ctype)) if crc is None else crc
    return struct.pack(">I", len(body)) + ctype + body + struct.pack(">I", c)


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(px, filters):
    """px uint8 [H, W, bpp] -> the filtered scanlines (filter byte + bytes), filters[y] in 0..4."""
    H, W, bpp = px.shape
    rows = px.reshape(H, W * bpp).astype(np.int32)
    out = []
    for y in range(H):
        x = rows[y]
        up = rows[y - 1] if y else np.zeros_like(x)
        left = np.concatenate([np.zeros(bpp, np.int32), x[:-bpp]])
        ul = np.concatenate([np.zeros(bpp, np.int32), up[:-bpp]])
        pred = [0, left, up, (left + up) >> 1, _paeth(left, up, ul)][filters[y]]
        out.append(bytes([filters[y]]) + ((x - pred) & 255).astype(np.uint8).tobytes())
    return b"".join(out)


def compress(raw, mode="dynamic", level=6):
    """zlib stream of raw: 'dynamic' (zlib at `level`), 'fixed' (Z_FIXED) or 'stored' (level 0)."""
    if mode == "stored":
        level = 0
    c = zlib.compressobj(level, zlib.DEFLATED, 15, 8, zlib.Z_FIXED if mode == "fixed" else zlib.Z_DEFAULT_STRATEGY)
    return c.compress(raw) + c.flush()


def png(px, colour, filters=None, idat_sizes=None, mode="dynamic", extra=(), interlace=False):
    """PNG bytes of px uint8 [H, W, bpp] (bpp = BPP[colour]). filters: per row (default all 0); idat_sizes: the IDAT
    payload split (a list of chunk sizes, 0 allowed, cycled); extra: chunks written after IHDR."""
    H, W, bpp = px.shape
    assert bpp == BPP[colour]
    if interlace:  # Adam7, filter 0
        raw = b""
        for xs, ys, dx, dy in ((0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)):
            sub = px[ys::dy, xs::dx]
            if sub.shape[0] and sub.shape[1]:
                raw += filter_rows(sub, [0] * sub.shape[0])
    else:
        raw = filter_rows(px, filters if filters is not None else [0] * H)
    z = compress(raw, mode)
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, colour, 0, 0, 1 if interlace else 0))
    out += b"".join(extra)
    sizes = list(idat_sizes or [len(z)])
    pos, k = 0, 0
    while pos < len(z):
        s = sizes[k % len(sizes)]
        out += chunk(b"IDAT", z[pos:pos + s])
        pos += s
        k += 1
    return out + chunk(b"IEND", b"")


class Bits:
    """LSB-first bit writer (RFC 1951 3.1.1): values low bit first, Huffman codes high bit first."""

    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, value, nbits):
        self.v |= (value & ((1 << nbits) - 1)) << self.n
        self.n += nbits
        return self

    def code(self, code, length):
        for i in range(length - 1, -1, -1):
            self.put((code >> i) & 1, 1)
        return self

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")


def canonical(lengths):
    """{symbol: (code, length)} of a canonical Huffman code (RFC 1951 3.2.2)."""
    bl = [0] * 16
    for ln in lengths:
        if ln:
            bl[ln] += 1
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    out = {}
    for s, ln in enumerate(lengths):
        if ln:
            out[s] = (nxt[ln], ln)
            nxt[ln] += 1
    return out


CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


def dynamic_header(b, lit_lens, dist_lens, cl_lens=None, cl_symbols=None):
    """Write a dynamic block's header. cl_lens: the code-length code (19 lengths; default 4 bits for symbols 0-15,
    complete); cl_symbols: the (symbol, extra value) sequence to send (default: every length as itself)."""
    cl_lens = cl_lens or [4] * 16 + [0, 0, 0]
    b.put(len(lit_lens) - 257, 5).put(len(dist_lens) - 1, 5).put(19 - 4, 4)
    for s in CL_ORDER:
        b.put(cl_lens[s], 3)
    cl = canonical(cl_lens)
    for s, extra in (cl_symbols if cl_symbols is not None else [(ln, None) for ln in list(lit_lens) + list(dist_lens)]):
        b.code(*cl[s])
        if s == 16:
            b.put(extra, 2)
        elif s == 17:
            b.put(extra, 3)
        elif s == 18:
            b.put(extra, 7)
    return canonical(lit_lens), canonical(dist_lens)


def zwrap(deflate, data=b""):
    """zlib header + deflate bytes + the Adler-32 of data."""
    return b"\x78\x9c" + deflate + struct.pack(">I", zlib.adler32(data))


def fixed_code(sym):
    if sym < 144:
        return 0x30 + sym, 8
    if sym < 256:
        return 0x190 + sym - 144, 9
    if sym < 280:
        return sym - 256, 7
    return 0xC0 + sym - 280, 8


def malformed_streams():
    """{name: zlib stream} with one defect each, every one a stream zlib rejects."""
    s = {}
    s["bad_fcheck"] = b"\x78\x9d" + zlib.compress(b"abc")[2:]
    s["cm_not_8"] = b"\x79\x9c"[:1] + bytes([(31 - (0x79 * 256) % 31) % 31]) + zlib.compress(b"abc")[2:]
    flg = 0x20
    flg |= (31 - (0x78 * 256 + flg) % 31) % 31
    s["fdict"] = bytes([0x78, flg]) + b"\x00\x00\x00\x00" + zlib.compress(b"abc")[2:]
    s["block_type_3"] = zwrap(Bits().put(1, 1).put(3, 2).bytes())
    s["stored_len_nlen"] = zwrap(Bits().put(1, 1).put(0, 2).bytes() + struct.pack("<HH", 3, 0) + b"abc", b"abc")
    s["stored_truncated"] = b"\x78\x9c" + Bits().put(1, 1).put(0, 2).bytes() + struct.pack("<HH", 10, 0xFFF5) + b"abc"
    b = Bits().put(1, 1).put(2, 2)
    dynamic_header(b, [8] * 257, [1], cl_lens=[1] * 19)
    s["over_subscribed_code_lengths"] = zwrap(b.bytes())
    b = Bits().put(1, 1).put(2, 2)
    dynamic_header(b, [0] * 257, [0], cl_lens=[1] + [0] * 18, cl_symbols=[(0, None)] * 258)
    s["incomplete_code_lengths"] = zwrap(b.bytes())
    lit = [0] * 257
    lit[65], lit[256] = 2, 2  # two codes of length 2: incomplete, and not a single code of length 1
    b = Bits().put(1, 1).put(2, 2)
    lc, _ = dynamic_header(b, lit, [1])
    b.code(*lc[65]).code(*lc[256])
    s["incomplete_literal_lengths"] = zwrap(b.bytes(), b"A")
    lit = [0] * 257
    lit[65], lit[256] = 1, 1
    b = Bits().put(1, 1).put(2, 2)
    dynamic_header(b, lit, [1, 1, 1])  # three distance codes of length 1: over-subscribed
    s["over_subscribed_distances"] = zwrap(b.bytes())
    lit = [0] * 257
    lit[65], lit[66] = 1, 1
    b = Bits().put(1, 1).put(2, 2)
    dynamic_header(b, lit, [1])
    s["no_end_of_block"] = zwrap(b.bytes())
    b = Bits().put(1, 1).put(2, 2)
    dynamic_header(b, [8] * 257, [1], cl_lens=[4] * 15 + [0] + [4, 0, 0], cl_symbols=[(16, 0)])
    s["repeat_at_start"] = zwrap(b.bytes())
    b = Bits().put(1, 1).put(2, 2)
    dynamic_header(b, [8] * 257, [1], cl_lens=[4] * 15 + [0] + [0, 0, 4], cl_symbols=[(18, 127), (18, 127)])  # 276 > 258
    s["repeat_past_end"] = zwrap(b.bytes())
    for sym in (286, 287):
        s["literal_length_%d" % sym] = zwrap(Bits().put(1, 1).put(1, 2).code(*fixed_code(sym)).code(*fixed_code(256)).bytes())
    for d in (30, 31):
        b = Bits().put(1, 1).put(1, 2).code(*fixed_code(65)).code(*fixed_code(257)).code(d, 5).code(*fixed_code(256))
        s["distance_%d" % d] = zwrap(b.bytes(), b"AAAA")
    b = Bits().put(1, 1).put(1, 2).code(*fixed_code(65)).code(*fixed_code(257)).code(1, 5).code(*fixed_code(256))
    s["distance_too_far"] = zwrap(b.bytes(), b"AAAA")  # distance 2 after one byte
    z = zlib.compress(bytes(range(256)) * 40)
    s["truncated"] = z[:len(z) // 2]
    s["no_adler"] = z[:-4]
    s["wrong_adler"] = z[:-1] + bytes([z[-1] ^ 1])
    s["empty"] = b""
    s["header_only"] = b"\x78\x9c"
    return s


def single_code_streams():
    """Valid streams that use zlib's one exception: a literal/length or distance set of a single code of length 1."""
    lit = [0] * 257
    lit[256] = 1
    b = Bits().put(1, 1).put(2, 2)
    lc, _ = dynamic_header(b, lit, [0])  # end-of-block only, no distance codes
    b.code(*lc[256])
    only_eob = zwrap(b.bytes())
    lit = [0] * 258
    lit[65], lit[256], lit[257] = 1, 2, 2
    b = Bits().put(1, 1).put(2, 2)
    lc, dc = dynamic_header(b, lit, [1])  # one distance code (distance 1) of length 1
    b.code(*lc[65]).code(*lc[257]).code(*dc[0]).code(*lc[256])
    return {"only_end_of_block": only_eob, "single_distance_code": zwrap(b.bytes(), b"AAAA")}
