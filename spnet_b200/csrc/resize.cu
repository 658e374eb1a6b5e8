// LANCZOS resize of uint8 frames, bit-identical to Pillow's Image.resize(..., Image.LANCZOS) on 8-bit images
// (libImaging/Resample.c), fused with the (v/255 - 0.5)*2 normalisation of spnet/utils.py:340-342.
//
// Pillow resamples separably: a horizontal pass whose result is clipped to uint8, then a vertical pass over that
// uint8 image. Each output byte is clamp((2^21 + sum_k src[xmin + k] * coeff[k]) >> 22, 0, 255) in int32, with
// coefficient tables that depend only on (in size, out size). The host computes the tables exactly as Pillow does
// (spnet_b200/ops.py lanczos_tables), so the kernel is pure integer arithmetic and its bytes are Pillow's.
//
// One CTA per (frame, band of output rows): the horizontal pass of every input row the band reads goes to shared
// memory as uint8, then the vertical pass writes lut[byte] as fp32. Rows read by two bands are computed by both (the
// same bytes), so no CTA waits for another.
#include "common.cuh"

namespace {

constexpr int kResizeThreads = 256;
constexpr int kMaxBand = 32;                 // output rows per CTA
constexpr size_t kResizeSmemMax = 200 * 1024;

__device__ __forceinline__ unsigned char clip8(int acc) {
    const int v = acc >> 22;  // Pillow's PRECISION_BITS = 32 - 8 - 2
    return (unsigned char)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// Taps of one output index, clamped to what the source span holds: for tables from lanczos_tables the clamps change
// nothing; for any other table they keep every read in bounds.
__device__ __forceinline__ void taps(const int* __restrict__ bounds, int i, int lo, int span, int k, int& first, int& count) {
    first = min(max(__ldg(bounds + 2 * i) - lo, 0), span);
    count = max(min(min(__ldg(bounds + 2 * i + 1), k), span - first), 0);
}

__global__ void __launch_bounds__(kResizeThreads) resize_lanczos_u8_kernel(
    const unsigned char* __restrict__ in, int H, int W, const int* __restrict__ xbounds, const int* __restrict__ xcoeffs,
    int kx, const int* __restrict__ ybounds, const int* __restrict__ ycoeffs, int ky, const float* __restrict__ lut,
    float* __restrict__ out, int OH, int OW, int band, int cap) {
    extern __shared__ unsigned char mid[];   // [rows][OW] horizontal-pass bytes of input rows y0 .. y0 + rows - 1
    __shared__ float sl[256];
    sl[threadIdx.x] = lut[threadIdx.x];
    const int frame = blockIdx.y;
    const int oy0 = blockIdx.x * band, oy1 = min(oy0 + band, OH);
    const int y0 = min(max(__ldg(ybounds + 2 * oy0), 0), H - 1);
    const int rows = min(max(__ldg(ybounds + 2 * (oy1 - 1)) + __ldg(ybounds + 2 * (oy1 - 1) + 1) - y0, 1), min(cap, H - y0));
    const unsigned char* src = in + ((size_t)frame * H + y0) * W;

    for (int i = threadIdx.x; i < rows * OW; i += kResizeThreads) {
        const int r = i / OW, ox = i - r * OW;
        int xmin, count;
        taps(xbounds, ox, 0, W, kx, xmin, count);
        const unsigned char* s = src + (size_t)r * W + xmin;
        const int* k = xcoeffs + (size_t)ox * kx;
        int acc = 1 << 21;
        for (int t = 0; t < count; ++t) acc += (int)__ldg(s + t) * __ldg(k + t);
        mid[i] = clip8(acc);
    }
    __syncthreads();

    float* dst = out + ((size_t)frame * OH + oy0) * OW;
    for (int i = threadIdx.x; i < (oy1 - oy0) * OW; i += kResizeThreads) {
        const int r = i / OW, ox = i - r * OW;
        int first, count;
        taps(ybounds, oy0 + r, y0, rows, ky, first, count);
        const unsigned char* s = mid + first * OW + ox;
        const int* k = ycoeffs + (size_t)(oy0 + r) * ky;
        int acc = 1 << 21;
        for (int t = 0; t < count; ++t) acc += (int)s[t * OW] * __ldg(k + t);
        dst[i] = sl[clip8(acc)];
    }
}

}  // namespace

extern "C" {

// in uint8 [n, H, W]; xbounds int32 [OW, 2] / ybounds [OH, 2] = (first input index, tap count); xcoeffs int32
// [OW, kx] / ycoeffs [OH, ky] in units of 2^-22 (ops.lanczos_tables); lut fp32 [256] (spnet_normalize_u8's table);
// out fp32 [n, OH, OW].
int spnet_resize_lanczos_u8(const unsigned char* in, int n, int H, int W, const int* xbounds, const int* xcoeffs, int kx,
                            const int* ybounds, const int* ycoeffs, int ky, const float* lut, float* out, int OH, int OW,
                            cudaStream_t stream) {
    SPNET_REQUIRE(in && xbounds && xcoeffs && ybounds && ycoeffs && lut && out, "resize_lanczos_u8: null pointer");
    SPNET_REQUIRE(n > 0 && n <= 65535 && H > 0 && W > 0 && OH > 0 && OW > 0 && kx > 0 && ky > 0,
                  "resize_lanczos_u8: bad shape n=%d %dx%d -> %dx%d, kx=%d ky=%d", n, H, W, OH, OW, kx, ky);
    // Input rows one band reads, for Pillow's tables: from center(oy0) - support to center(oy0 + band - 1) + support,
    // i.e. fewer than (band - 1) * H / OH + 2 * support + 2 <= (band - 1) * H / OH + ky + 1.
    int band = kMaxBand, cap = 0;
    for (;; band >>= 1) {
        const long long need = (long long)(band - 1) * H / OH + ky + 1;
        cap = need < H ? (int)need : H;
        if ((size_t)cap * OW <= kResizeSmemMax || band == 1) break;
    }
    const size_t smem = (size_t)cap * OW;
    SPNET_REQUIRE(smem <= kResizeSmemMax, "resize_lanczos_u8: %d input rows of %d bytes do not fit shared memory", cap, OW);
    static bool configured[64] = {};
    const int rc = spnet_smem_optin(configured, resize_lanczos_u8_kernel, kResizeSmemMax, "resize_lanczos_u8");
    if (rc) return rc;
    const dim3 grid((unsigned)ceil_div(OH, band), (unsigned)n);
    resize_lanczos_u8_kernel<<<grid, kResizeThreads, smem, stream>>>(in, H, W, xbounds, xcoeffs, kx, ybounds, ycoeffs, ky, lut,
                                                                      out, OH, OW, band, cap);
    return spnet_check_launch("resize_lanczos_u8");
}

}  // extern "C"
