// PNG pixel data on the device: the concatenated IDAT payload of each frame (one zlib stream of filtered scanlines)
// -> channel 0 of the frame as uint8, the bytes Pillow decodes (np.asarray(Image.open(f).convert("RGB"))[:, :, 0]) for
// 8-bit, non-interlaced, non-palette PNGs. spnet_b200/png.py parses the container and sends every other file to Pillow.
//
// One warp per frame, frames independent:
//   1. lane 0 inflates the stream into the frame's scratch slice (inflate.cuh; Huffman tables and an 8 KB window of
//      recent output in the warp's shared memory);
//   2. the warp checks the Adler-32 trailer, the two sums split over the lanes and combined by a warp reduction;
//   3. the warp un-filters row by row. At bit depth 8 every PNG filter predicts a byte from the same channel of the
//      pixel to the left and the byte above, so channel 0 is reconstructed alone: None and Up lane-parallel, Sub as a
//      warp prefix sum mod 256, Average and Paeth serially on lane 0. The previous row's channel 0 lives in the window.
// Parallelism comes from the number of frames per launch.
#include "common.cuh"
#include "inflate.cuh"

namespace {

// Power of two; also the widest frame (the un-filter keeps one row in it). 8 KB keeps a CTA near 11 KB of shared memory,
// so a 2,048-frame launch runs in one wave on 148 SMs; with 16 KB it took two (67.7 -> 42.7 ms per launch on a B200 at 1000 W),
// and 2 or 4 KB gained nothing more. Back-references further than the window read the output in global memory.
constexpr unsigned kWindow = 8192;
constexpr size_t kPngSmem = sizeof(inflate::Tables) + kWindow;  // under the 48 KB that needs no opt-in

__device__ __forceinline__ int paeth(int a, int b, int c) {
    const int p = a + b - c;
    const int pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
    return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}

__global__ void __launch_bounds__(32) png_decode_u8_kernel(const unsigned char* __restrict__ streams, long long stream_bytes,
                                                           const long long* __restrict__ offsets, int H, int W, int bpp,
                                                           unsigned char* scratch, unsigned char* __restrict__ out,
                                                           int* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char smem[];
    inflate::Tables& tables = *reinterpret_cast<inflate::Tables*>(smem);
    unsigned char* win = smem + sizeof(inflate::Tables);
    const int frame = blockIdx.x, lane = threadIdx.x;
    const long long lo = min(max(offsets[frame], 0ll), stream_bytes);
    const long long hi = min(max(offsets[frame + 1], lo), stream_bytes);
    const unsigned char* in = streams + lo;
    const long long len = hi - lo;
    const long long stride = 1 + (long long)W * bpp, total = stride * H;
    unsigned char* raw = scratch + (long long)frame * total;  // written by lane 0, read by the warp: no read-only loads

    int st = SPNET_PNG_OK;
    long long trailer = 0;
    if (lane == 0) {
        long long produced = 0;
        st = inflate::inflate_zlib(in, len, raw, total, tables, win, kWindow, &produced, &trailer);
        if (st == SPNET_PNG_OK && produced != total) st = SPNET_PNG_ERR_SIZE;
        if (st == SPNET_PNG_OK && trailer + 4 != len) st = SPNET_PNG_ERR_ADLER;
    }
    st = __shfl_sync(0xffffffffu, st, 0);
    trailer = __shfl_sync(0xffffffffu, trailer, 0);
    __syncwarp();  // lane 0's scratch writes are visible to the warp

    if (st == SPNET_PNG_OK) {
        // adler = (b << 16) | a, a = 1 + sum d_i, b = total + sum (total - i) d_i, both mod 65521
        unsigned long long sa = 0, sb = 0;
        for (long long i = lane; i < total; i += 32) {
            const unsigned d = raw[i];
            sa += d;
            sb += (unsigned long long)((total - i) % 65521) * d;
        }
        unsigned a = (unsigned)(sa % 65521), b = (unsigned)(sb % 65521);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        a = (1 + a) % 65521;
        b = (unsigned)((total % 65521 + b) % 65521);
        const unsigned want = ((unsigned)__ldg(in + trailer) << 24) | ((unsigned)__ldg(in + trailer + 1) << 16) |
                              ((unsigned)__ldg(in + trailer + 2) << 8) | (unsigned)__ldg(in + trailer + 3);
        if (((b << 16) | a) != want) st = SPNET_PNG_ERR_ADLER;
    }

    if (st == SPNET_PNG_OK) {
        unsigned char* above = win;  // channel 0 of the row above; zeros above the first row
        for (int x = lane; x < W; x += 32) above[x] = 0;
        __syncwarp();
        unsigned char* dst = out + (long long)frame * H * W;
        for (int y = 0; y < H; ++y, dst += W) {
            const unsigned char* r = raw + y * stride;
            const int ft = r[0];
            if (ft > 4) {
                st = SPNET_PNG_ERR_FILTER;
                break;
            }
            ++r;
            if (ft == 0 || ft == 2) {  // None, Up
                for (int x = lane; x < W; x += 32) {
                    const unsigned char v = (unsigned char)(r[(long long)x * bpp] + (ft == 2 ? above[x] : 0));
                    above[x] = v;
                    dst[x] = v;
                }
            } else if (ft == 1) {  // Sub: a running sum along the row
                int carry = 0;
                for (int x0 = 0; x0 < W; x0 += 32) {
                    const int x = x0 + lane;
                    int v = x < W ? r[(long long)x * bpp] : 0;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int u = __shfl_up_sync(0xffffffffu, v, o);
                        if (lane >= o) v += u;
                    }
                    v += carry;
                    carry = __shfl_sync(0xffffffffu, v, 31) & 255;
                    if (x < W) {
                        above[x] = (unsigned char)v;
                        dst[x] = (unsigned char)v;
                    }
                }
            } else if (lane == 0) {  // Average, Paeth
                int left = 0, upleft = 0;
                for (int x = 0; x < W; ++x) {
                    const int up = above[x];
                    const int pred = ft == 3 ? (left + up) >> 1 : paeth(left, up, upleft);
                    const int v = (r[(long long)x * bpp] + pred) & 255;
                    above[x] = (unsigned char)v;
                    dst[x] = (unsigned char)v;
                    left = v;
                    upleft = up;
                }
            }
            __syncwarp();
        }
    }
    if (lane == 0) status[frame] = st;
}

}  // namespace

extern "C" {

int spnet_png_decode_u8(const unsigned char* streams, long long stream_bytes, const long long* offsets, int n, int H, int W,
                        int bpp, unsigned char* scratch, long long scratch_bytes, unsigned char* out, int* status,
                        cudaStream_t stream) {
    SPNET_REQUIRE(streams && offsets && scratch && out && status, "png_decode_u8: null pointer");
    SPNET_REQUIRE(n > 0 && H > 0 && H <= (1 << 20) && W > 0 && W <= (int)kWindow && bpp >= 1 && bpp <= 4 && stream_bytes >= 0,
                  "png_decode_u8: bad shape n=%d H=%d W=%d (at most %u) bpp=%d stream_bytes=%lld", n, H, W, kWindow, bpp,
                  stream_bytes);
    const long long per = (long long)H * (1 + (long long)W * bpp);
    SPNET_REQUIRE(scratch_bytes >= 0 && n <= scratch_bytes / per,
                  "png_decode_u8: scratch holds %lld bytes, %d frames need %lld each", scratch_bytes, n, per);
    png_decode_u8_kernel<<<n, 32, kPngSmem, stream>>>(streams, stream_bytes, offsets, H, W, bpp, scratch, out, status);
    return spnet_check_launch("png_decode_u8");
}

}  // extern "C"
