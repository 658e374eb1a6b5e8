// spnet_b200 — shared device/host helpers for the sm_100a kernels.
// Conventions (SURVEY.md §8b): caller owns all memory, every entry point is
// asynchronous on the given stream, returns 0 or a negative error code and
// records a per-thread message readable through spnet_last_error().
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/spnet_b200.h"

#define SPNET_OK 0

#define SPNET_F32 0
#define SPNET_BF16 1

void spnet_set_error(const char* fmt, ...);
int spnet_check_launch(const char* what);

#define SPNET_REQUIRE(cond, ...)                                   \
    do {                                                           \
        if (!(cond)) {                                             \
            spnet_set_error(__VA_ARGS__);                          \
            return SPNET_ERR_ARG;                                  \
        }                                                          \
    } while (0)

typedef __nv_bfloat16 bf16;

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------
// 16-byte vector access: 4 floats or 8 bf16, always widened to fp32 registers.
// ---------------------------------------------------------------------------
template <typename T> struct VecN;
template <> struct VecN<float> { static constexpr int N = 4; };
template <> struct VecN<bf16> { static constexpr int N = 8; };

__device__ __forceinline__ void load_vec(const float* p, float (&v)[4]) {
    float4 r = *reinterpret_cast<const float4*>(p);
    v[0] = r.x; v[1] = r.y; v[2] = r.z; v[3] = r.w;
}
__device__ __forceinline__ void load_vec(const bf16* p, float (&v)[8]) {
    uint4 r = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[2 * i] = __uint_as_float(w[i] << 16);
        v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}
__device__ __forceinline__ void store_vec(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void store_vec(bf16* p, const float (&v)[8]) {
    uint4 r;
    r.x = pack_bf16x2(v[0], v[1]);
    r.y = pack_bf16x2(v[2], v[3]);
    r.z = pack_bf16x2(v[4], v[5]);
    r.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(p) = r;
}

__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(bf16 x) { return __bfloat162float(x); }
template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float x) { return __float2bfloat16_rn(x); }
// value as it will read back after being stored as T
template <typename T> __device__ __forceinline__ float round_to(float x) { return to_f32(from_f32<T>(x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Column sums of a 32x32 block held one row per lane (v[j] = element (lane, j)): after the
// butterfly lane L holds sum_rows element(row, L). 31 shuffles instead of 32*5. Destroys v.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
            const float send = upper ? v[i] : v[i + off];
            const float keep = upper ? v[i + off] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0];
}

// ---- order-independent accumulators for cross-CTA sums (BatchNorm statistics, loss terms) -----
// A sum that many CTAs contribute to must not depend on the order in which they arrive, or two runs of
// the same step differ in the last bits and the network amplifies that (3e-5 at the MobileNet head).
// Floating-point atomics are not associative; 64-bit integer atomics are. Every contribution is split
// into two fixed-point limbs  v = (hi * 2^32 + lo) * 2^-56  (quantum 2^-56 = 1.4e-17, |v| < 2^39) and
// added with integer atomics: exact for any fp32 partial of magnitude >= 2^-32, rounded down to the
// quantum below that, and bit-identical for every arrival order. Entry i occupies words [2i, 2i+1] of
// a zero-initialised int64 buffer; stat_get() reassembles the double.
__device__ __forceinline__ void stat_add(long long* acc, long long i, double v) {
    const double t = v * 16777216.0;  // units of 2^-24
    const double fh = floor(t);
    const long long hi = __double2ll_rd(t);
    const unsigned long long lo = __double2ull_rz((t - fh) * 4294967296.0);  // [0, 2^32)
    unsigned long long* p = reinterpret_cast<unsigned long long*>(acc) + 2 * i;
    atomicAdd(p, (unsigned long long)hi);
    if (lo) atomicAdd(p + 1, lo);
}
__device__ __forceinline__ double stat_get(const long long* acc, long long i) {
    const long long hi = acc[2 * i];
    const unsigned long long lo = (unsigned long long)acc[2 * i + 1];
    return ((double)hi + (double)lo * (1.0 / 4294967296.0)) * (1.0 / 16777216.0);
}
__device__ __forceinline__ void stat_clear(long long* acc, long long i) { acc[2 * i] = 0; acc[2 * i + 1] = 0; }

// cudaFuncSetAttribute (the dynamic shared-memory opt-in) is per DEVICE: one flag per device for a launcher's
// "configured once" state. Returns true the first time it is called for the current device with these flags.
static inline bool spnet_first_use_on_device(bool (&flags)[64]) {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if (flags[dev]) return false;
    flags[dev] = true;
    return true;
}

// SM count of the current device (148 on B200), cached per device: persistent grids are sized from it.
static inline int spnet_num_sms() {
    static int cached[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// dispatch on activation dtype code
#define SPNET_DISPATCH_DTYPE(dtype, ...)                                   \
    do {                                                                   \
        if ((dtype) == SPNET_F32) { typedef float T; __VA_ARGS__; }        \
        else if ((dtype) == SPNET_BF16) { typedef bf16 T; __VA_ARGS__; }   \
        else { spnet_set_error("bad dtype code %d", (int)(dtype)); return SPNET_ERR_ARG; } \
    } while (0)
