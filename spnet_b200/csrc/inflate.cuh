// zlib / DEFLATE decoder core (RFC 1950 / RFC 1951) for one stream on one thread: the inflate step of
// spnet_png_decode_u8 (png.cu). It is plain C++ behind SPNET_HD, so the same code compiles for the host, where
// tests/test_png_host.py runs it under AddressSanitizer and UBSan over valid, malformed and corrupted streams.
//
// Bounds: every input read is checked against the stream length; every output write against the capacity; every
// back-reference against the bytes produced so far. The caller provides the Huffman tables (Tables) and a
// power-of-two window that mirrors the last `win_size` output bytes; back-references within it read the window (shared
// memory on the device), older ones read the output itself.
//
// It rejects what zlib rejects: a bad CMF/FLG header or FDICT, block type 3, stored LEN != ~NLEN, over-subscribed or
// incomplete code sets (incomplete literal/length or distance sets only as a single code of length 1), no end-of-block
// code, a repeat with nothing to repeat or past HLIT + HDIST, literal/length symbols 286-287, distance symbols 30-31,
// distances before the start of the output and input that ends early. It does not check the Adler-32 trailer: it
// reports where the trailer starts and the caller checks it (png.cu over a warp, adler32 below on the host).
#pragma once
#include <stdint.h>

#include "../../include/spnet_b200.h"

#ifdef __CUDACC__
#define SPNET_HD __host__ __device__ __forceinline__
#else
#define SPNET_HD inline
#endif

namespace inflate {

constexpr int kFastBits = 9;  // first-level lookup: codes of up to 9 bits decode in one step, longer ones bit by bit

struct Tables {
    uint16_t lfast[1 << kFastBits];  // (symbol << 4) | code length, 0 = longer than kFastBits or no code
    uint16_t dfast[1 << kFastBits];
    uint16_t lcount[16], dcount[16];  // codes per length
    uint16_t lsym[288], dsym[32];     // symbols in canonical order
    uint16_t offs[16];                // build()'s scratch
    uint8_t lens[320];                // code lengths of one dynamic block
};

struct Bits {
    const uint8_t* in;
    long long len, pos;
    uint64_t buf;
    int cnt;
};

SPNET_HD void refill(Bits& b) {
    while (b.cnt <= 56 && b.pos < b.len) {
        b.buf |= (uint64_t)b.in[b.pos++] << b.cnt;
        b.cnt += 8;
    }
}

// n <= 32 bits; false when the stream holds fewer
SPNET_HD bool getbits(Bits& b, int n, unsigned& v) {
    if (b.cnt < n) refill(b);
    if (b.cnt < n) return false;
    v = (unsigned)(b.buf & ((1ull << n) - 1));
    b.buf >>= n;
    b.cnt -= n;
    return true;
}

// Canonical code of lens[0 .. n) into count / symbol and the first-level table. Returns < 0 for an over-subscribed
// set, > 0 for an incomplete one (the number of missing codes at length 15, scaled), 0 for a complete one.
SPNET_HD int build(const uint8_t* lens, int n, uint16_t* count, uint16_t* symbol, uint16_t* fast, uint16_t* offs) {
    for (int l = 0; l < 16; ++l) count[l] = 0;
    for (int s = 0; s < n; ++s) count[lens[s]]++;
    for (int i = 0; i < (1 << kFastBits); ++i) fast[i] = 0;
    if (count[0] == n) return 1;  // no codes: incomplete
    int left = 1;
    for (int l = 1; l < 16; ++l) {
        left = (left << 1) - count[l];
        if (left < 0) return left;
    }
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = (uint16_t)(offs[l] + count[l]);
    for (int s = 0; s < n; ++s)
        if (lens[s]) symbol[offs[lens[s]]++] = (uint16_t)s;
    unsigned code = 0;
    int idx = 0;
    for (int l = 1; l <= kFastBits; ++l, code <<= 1) {
        for (int k = 0; k < count[l]; ++k, ++code) {
            unsigned rev = 0;
            for (int j = 0; j < l; ++j) rev |= ((code >> j) & 1u) << (l - 1 - j);
            const uint16_t e = (uint16_t)((symbol[idx++] << 4) | l);
            for (unsigned r = rev; r < (1u << kFastBits); r += 1u << l) fast[r] = e;
        }
    }
    return left;
}

// One symbol: >= 0, or SPNET_PNG_ERR_DATA (no such code) / SPNET_PNG_ERR_TRUNCATED
SPNET_HD int decode(Bits& b, const uint16_t* fast, const uint16_t* count, const uint16_t* symbol) {
    refill(b);
    const uint16_t e = fast[b.buf & ((1u << kFastBits) - 1)];
    const int fl = e & 15;
    if (fl && fl <= b.cnt) {
        b.buf >>= fl;
        b.cnt -= fl;
        return e >> 4;
    }
    int code = 0, first = 0, index = 0;
    for (int l = 1; l < 16; ++l) {
        if (l > b.cnt) return SPNET_PNG_ERR_TRUNCATED;
        code |= (int)((b.buf >> (l - 1)) & 1u);
        const int c = count[l];
        if (code - c < first) {
            b.buf >>= l;
            b.cnt -= l;
            return symbol[index + (code - first)];
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return SPNET_PNG_ERR_DATA;
}

struct Out {
    uint8_t* out;
    long long cap, pos;
    uint8_t* win;
    unsigned mask;  // window size - 1
};

SPNET_HD void put(Out& o, uint8_t v) {
    o.out[o.pos] = v;
    o.win[o.pos & o.mask] = v;
    ++o.pos;
}

// Literal/length and distance codes of one compressed block.
SPNET_HD int codes(Bits& b, Out& o, const Tables& t) {
    for (;;) {
        int sym = decode(b, t.lfast, t.lcount, t.lsym);
        if (sym < 0) return sym;
        if (sym < 256) {
            if (o.pos >= o.cap) return SPNET_PNG_ERR_SIZE;
            put(o, (uint8_t)sym);
            continue;
        }
        if (sym == 256) return SPNET_PNG_OK;
        sym -= 257;
        if (sym >= 29) return SPNET_PNG_ERR_DATA;  // literal/length symbols 286 and 287
        // RFC 1951 3.2.5: base and extra bits of length codes 257-284 and distance codes 4-29 follow a pattern
        const int le = sym < 8 || sym == 28 ? 0 : (sym >> 2) - 1;
        const int lb = sym < 8 ? 3 + sym : (sym == 28 ? 258 : ((4 + (sym & 3)) << le) + 3);
        unsigned x;
        if (!getbits(b, le, x)) return SPNET_PNG_ERR_TRUNCATED;
        const int len = lb + (int)x;
        const int ds = decode(b, t.dfast, t.dcount, t.dsym);
        if (ds < 0) return ds;
        if (ds >= 30) return SPNET_PNG_ERR_DATA;  // distance symbols 30 and 31
        const int de = ds < 4 ? 0 : (ds >> 1) - 1;
        const int db = ds < 4 ? 1 + ds : ((2 + (ds & 1)) << de) + 1;
        if (!getbits(b, de, x)) return SPNET_PNG_ERR_TRUNCATED;
        const long long dist = db + (long long)x;
        if (dist > o.pos) return SPNET_PNG_ERR_DATA;
        if (len > o.cap - o.pos) return SPNET_PNG_ERR_SIZE;
        if (dist <= (long long)o.mask + 1) {
            for (int k = 0; k < len; ++k) put(o, o.win[(o.pos - dist) & o.mask]);
        } else {
            for (int k = 0; k < len; ++k) put(o, o.out[o.pos - dist]);
        }
    }
}

SPNET_HD int fixed_tables(Tables& t) {
    for (int s = 0; s < 288; ++s) t.lens[s] = s < 144 ? 8 : (s < 256 ? 9 : (s < 280 ? 7 : 8));
    build(t.lens, 288, t.lcount, t.lsym, t.lfast, t.offs);
    for (int s = 0; s < 32; ++s) t.lens[s] = 5;
    build(t.lens, 32, t.dcount, t.dsym, t.dfast, t.offs);  // symbols 30 and 31 have codes here; codes() rejects them
    return SPNET_PNG_OK;
}

SPNET_HD int dynamic_tables(Bits& b, Tables& t) {
    unsigned nlen, ndist, ncode;
    if (!getbits(b, 5, nlen) || !getbits(b, 5, ndist) || !getbits(b, 4, ncode)) return SPNET_PNG_ERR_TRUNCATED;
    nlen += 257;
    ndist += 1;
    ncode += 4;
    if (nlen > 286 || ndist > 30) return SPNET_PNG_ERR_DATA;
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
#pragma unroll
    for (int i = 0; i < 19; ++i) {  // unrolled, so order[] folds into the code rather than a stack array
        unsigned v = 0;
        if (i < (int)ncode && !getbits(b, 3, v)) return SPNET_PNG_ERR_TRUNCATED;
        t.lens[order[i]] = (uint8_t)v;
    }
    // the code-length code must be complete (zlib); it borrows the literal/length tables
    if (build(t.lens, 19, t.lcount, t.lsym, t.lfast, t.offs) != 0) return SPNET_PNG_ERR_DATA;
    unsigned idx = 0;
    while (idx < nlen + ndist) {
        const int sym = decode(b, t.lfast, t.lcount, t.lsym);
        if (sym < 0) return sym;
        if (sym < 16) {
            t.lens[idx++] = (uint8_t)sym;
            continue;
        }
        unsigned rep, x;
        uint8_t v = 0;
        if (sym == 16) {
            if (idx == 0) return SPNET_PNG_ERR_DATA;  // a repeat with nothing before it
            v = t.lens[idx - 1];
            if (!getbits(b, 2, x)) return SPNET_PNG_ERR_TRUNCATED;
            rep = 3 + x;
        } else if (sym == 17) {
            if (!getbits(b, 3, x)) return SPNET_PNG_ERR_TRUNCATED;
            rep = 3 + x;
        } else {
            if (!getbits(b, 7, x)) return SPNET_PNG_ERR_TRUNCATED;
            rep = 11 + x;
        }
        if (idx + rep > nlen + ndist) return SPNET_PNG_ERR_DATA;
        while (rep--) t.lens[idx++] = v;
    }
    if (t.lens[256] == 0) return SPNET_PNG_ERR_DATA;  // no end-of-block code
    // incomplete literal/length or distance sets: zlib accepts only a single code of length 1
    int err = build(t.lens, (int)nlen, t.lcount, t.lsym, t.lfast, t.offs);
    if (err < 0 || (err > 0 && (t.lcount[1] != 1 || nlen - t.lcount[0] != 1))) return SPNET_PNG_ERR_DATA;
    err = build(t.lens + nlen, (int)ndist, t.dcount, t.dsym, t.dfast, t.offs);
    if (err < 0 || (err > 0 && t.dcount[0] != ndist && (t.dcount[1] != 1 || ndist - t.dcount[0] != 1)))
        return SPNET_PNG_ERR_DATA;
    return SPNET_PNG_OK;
}

// Inflates the zlib stream in[0 .. len) into out[0 .. cap). win: win_size (a power of two) bytes of scratch.
// On SPNET_PNG_OK, *produced is the output length and *trailer the offset of the byte after the last block (where
// the Adler-32 trailer starts); otherwise a negative SPNET_PNG_ERR_* code.
SPNET_HD int inflate_zlib(const uint8_t* in, long long len, uint8_t* out, long long cap, Tables& t, uint8_t* win,
                          unsigned win_size, long long* produced, long long* trailer) {
    *produced = 0;
    *trailer = 0;
    if (len < 2) return SPNET_PNG_ERR_TRUNCATED;
    const unsigned cmf = in[0], flg = in[1];
    // CM 8 (deflate), CINFO <= 7 (window <= 32 KB), FCHECK, no preset dictionary
    if ((cmf & 15) != 8 || (cmf >> 4) > 7 || ((cmf << 8) | flg) % 31 != 0 || (flg & 0x20)) return SPNET_PNG_ERR_HEADER;
    Bits b{in, len, 2, 0, 0};
    Out o{out, cap, 0, win, win_size - 1};
    unsigned last;
    do {
        unsigned type;
        if (!getbits(b, 1, last) || !getbits(b, 2, type)) return SPNET_PNG_ERR_TRUNCATED;
        int err;
        if (type == 0) {
            b.buf >>= b.cnt & 7;  // to the byte boundary
            b.cnt -= b.cnt & 7;
            unsigned n, nn;
            if (!getbits(b, 16, n) || !getbits(b, 16, nn)) return SPNET_PNG_ERR_TRUNCATED;
            if (n != (~nn & 0xffffu)) return SPNET_PNG_ERR_DATA;
            if ((long long)n > o.cap - o.pos) return SPNET_PNG_ERR_SIZE;
            for (unsigned k = 0; k < n; ++k) {
                unsigned v;
                if (!getbits(b, 8, v)) return SPNET_PNG_ERR_TRUNCATED;
                put(o, (uint8_t)v);
            }
            err = SPNET_PNG_OK;
        } else if (type == 1) {
            fixed_tables(t);
            err = codes(b, o, t);
        } else if (type == 2) {
            err = dynamic_tables(b, t);
            if (err == SPNET_PNG_OK) err = codes(b, o, t);
        } else {
            return SPNET_PNG_ERR_DATA;
        }
        if (err != SPNET_PNG_OK) return err;
    } while (!last);
    *produced = o.pos;
    *trailer = b.pos - (b.cnt >> 3);  // whole bytes still in the bit buffer were not consumed
    return SPNET_PNG_OK;
}

// Adler-32 of buf[0 .. n) (RFC 1950), serial; png.cu splits the same sums over a warp.
SPNET_HD uint32_t adler32(const uint8_t* buf, long long n) {
    uint32_t a = 1, s = 0;
    for (long long i = 0; i < n; ++i) {
        a = (a + buf[i]) % 65521u;
        s = (s + a) % 65521u;
    }
    return (s << 16) | a;
}

}  // namespace inflate
