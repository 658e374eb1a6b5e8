// Host build of spnet_b200/csrc/inflate.cuh for tests/test_png_host.py, compiled with -fsanitize=address,undefined.
//
//   inflate_harness <cases> <results> <window bytes>
//
// cases: records of (uint64 stream length, uint64 output capacity, stream bytes). Each stream and each output buffer is
// its own heap block of exactly that size, so any read or write past either is a sanitizer report. results: per case
// (int32 status, uint64 bytes produced, the bytes). The status follows the kernel's rules (csrc/png.cu): the inflate
// core's, then SPNET_PNG_ERR_ADLER unless exactly the four trailer bytes follow the last block and match.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../spnet_b200/csrc/inflate.cuh"

int main(int argc, char** argv) {
    if (argc != 4) return 2;
    FILE* in = fopen(argv[1], "rb");
    FILE* res = fopen(argv[2], "wb");
    const unsigned win_size = (unsigned)atoi(argv[3]);
    if (!in || !res || win_size == 0 || (win_size & (win_size - 1))) return 2;
    inflate::Tables* tables = (inflate::Tables*)malloc(sizeof(inflate::Tables));
    uint8_t* win = (uint8_t*)malloc(win_size);
    uint64_t hdr[2];
    while (fread(hdr, sizeof(hdr), 1, in) == 1) {
        uint8_t* stream = (uint8_t*)malloc(hdr[0] ? hdr[0] : 1);
        uint8_t* out = (uint8_t*)malloc(hdr[1] ? hdr[1] : 1);
        if (hdr[0] && fread(stream, hdr[0], 1, in) != 1) return 2;
        long long produced = 0, trailer = 0;
        int st = inflate::inflate_zlib(stream, (long long)hdr[0], out, (long long)hdr[1], *tables, win, win_size, &produced,
                                       &trailer);
        if (st == SPNET_PNG_OK) {
            const uint8_t* t = stream + trailer;
            if (trailer + 4 != (long long)hdr[0] ||
                inflate::adler32(out, produced) != ((uint32_t)t[0] << 24 | (uint32_t)t[1] << 16 | (uint32_t)t[2] << 8 | t[3]))
                st = SPNET_PNG_ERR_ADLER;
        }
        const int32_t s32 = st;
        const uint64_t n = st == SPNET_PNG_OK ? (uint64_t)produced : 0;
        fwrite(&s32, sizeof(s32), 1, res);
        fwrite(&n, sizeof(n), 1, res);
        if (n) fwrite(out, n, 1, res);
        free(stream);
        free(out);
    }
    free(win);
    free(tables);
    fclose(in);
    fclose(res);
    return 0;
}
