// Stem glue kernels (the small-channel convolutions themselves are in smallconv.cu).
//
//  * SPNet stem (spnet/models.py:319-340): Conv2D(3,3x3,same,no bias) -> AveragePooling2D(2)
//    -> BN -> LeakyReLU(0.1) -> Conv2D(3) -> BN -> LeakyReLU(0.1) -> Conv2D(3) -> BN
//    -> Add(AveragePooling2D(2)(input)) -> Dropout(0.1).
//    conv+avgpool is evaluated as the equivalent 4x4 stride-2 convolution (pad 1) whose
//    kernel is the 2x2 box average of the shifted 3x3 kernel, at a quarter of the work.
//  * keras.applications.Xception block1_conv1 (3x3, stride 2, valid, 3->32).
//
// All kernels are HBM/latency-bound (<1 % of the model's FLOPs); one thread per pixel,
// weights in shared memory, BatchNorm statistics reduced in the epilogue.
#include "common.cuh"

namespace {

// N contiguous elements <-> fp32 registers, 16-byte vectors when N allows it
template <typename T, int N>
__device__ __forceinline__ void load_row(const T* p, float (&v)[N]) {
    constexpr int V = VecN<T>::N;
    if constexpr (N % V == 0) {
#pragma unroll
        for (int c = 0; c < N / V; ++c) {
            float t[V];
            load_vec(p + c * V, t);
#pragma unroll
            for (int i = 0; i < V; ++i) v[c * V + i] = t[i];
        }
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = to_f32(p[i]);
    }
}
template <typename T, int N>
__device__ __forceinline__ void store_row(T* p, const float (&v)[N]) {
    constexpr int V = VecN<T>::N;
    if constexpr (N % V == 0) {
#pragma unroll
        for (int c = 0; c < N / V; ++c) {
            float t[V];
#pragma unroll
            for (int i = 0; i < V; ++i) t[i] = v[c * V + i];
            store_vec(p + c * V, t);
        }
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) p[i] = from_f32<T>(v[i]);
    }
}

__device__ __forceinline__ float apply_act(float y, int act) {
    if (act == 1) return fmaxf(y, 0.f);
    if (act == 2) return y > 0.f ? y : 0.1f * y;
    return y;
}

// ---- stem kernel folding: K4 = 2x2 box average of shifted K3; and its adjoint ----
__global__ void stem_k3_to_k4_kernel(const float* __restrict__ k3, float* __restrict__ k4, int cout) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // over 16*cout
    if (i >= 16 * cout) return;
    const int co = i % cout, kw = (i / cout) % 4, kh = i / (4 * cout);
    float s = 0.f;
    for (int dy = 0; dy < 2; ++dy)
        for (int dx = 0; dx < 2; ++dx) {
            const int a = kh - dy, b = kw - dx;
            if (a >= 0 && a < 3 && b >= 0 && b < 3) s += k3[(a * 3 + b) * cout + co];
        }
    k4[i] = 0.25f * s;
}
__global__ void stem_k4grad_to_k3grad_kernel(const float* __restrict__ g4, float* __restrict__ g3, int cout) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // over 9*cout
    if (i >= 9 * cout) return;
    const int co = i % cout, b = (i / cout) % 3, a = i / (3 * cout);
    float s = 0.f;
    for (int dy = 0; dy < 2; ++dy)
        for (int dx = 0; dx < 2; ++dx) s += g4[((a + dy) * 4 + (b + dx)) * cout + co];
    g3[i] += 0.25f * s;
}

// ---- stem output: d = dropout(a*c3 + b + skip)  (C = 3, skip has 1 channel) ----
__device__ __forceinline__ uint32_t mix32(unsigned long long x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return (uint32_t)x;
}
__device__ __forceinline__ bool dropout_keep(unsigned long long seed, long long elem, float rate) {
    const uint32_t r = mix32(seed * 0x9E3779B97F4A7C15ULL + (unsigned long long)elem);
    return (float)(r >> 8) * (1.0f / 16777216.0f) >= rate;
}

// The 3-channel tensors of the stem are walked as flat arrays, G pixels (= 3 sixteen-byte vectors: 24 bf16 or 12 fp32
// elements) per thread and step: element e of a group belongs to channel e % 3 and pixel e / 3 whatever the group, so
// the per-channel coefficients index statically and every access is a full 16-byte vector. (One thread per pixel with
// three 2-byte accesses ran these passes at 1.5 TB/s.) The pixels past the last full group are handled one by one.
template <typename T> struct Tri { static constexpr int G = VecN<T>::N, E = 3 * VecN<T>::N; };

template <typename T> __device__ __forceinline__ void load_tri(const T* __restrict__ p, float (&v)[Tri<T>::E]) {
    constexpr int V = VecN<T>::N;
    float t[V];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        load_vec(p + k * V, t);
#pragma unroll
        for (int i = 0; i < V; ++i) v[k * V + i] = t[i];
    }
}
template <typename T> __device__ __forceinline__ void store_tri(T* __restrict__ p, const float (&v)[Tri<T>::E]) {
    constexpr int V = VecN<T>::N;
    float t[V];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
        for (int i = 0; i < V; ++i) t[i] = v[k * V + i];
        store_vec(p + k * V, t);
    }
}

template <typename T>
__global__ void __launch_bounds__(256) stem_out_fwd_kernel(const T* __restrict__ c3, const float* __restrict__ a,
                                                           const float* __restrict__ b, const T* __restrict__ skip,
                                                           T* __restrict__ out, long long pixels, float rate,
                                                           const unsigned long long* __restrict__ seed) {
    constexpr int G = Tri<T>::G, E = Tri<T>::E;
    const unsigned long long sd = seed ? *seed : 0ULL;
    const float scale = 1.0f / (1.0f - rate);
    const float av[3] = {a[0], a[1], a[2]}, bv[3] = {b[0], b[1], b[2]};
    const long long groups = pixels / G;
    for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += (long long)gridDim.x * blockDim.x) {
        float v[E], s[G];
        load_tri(c3 + gi * E, v);
        load_vec(skip + gi * G, s);
#pragma unroll
        for (int e = 0; e < E; ++e) {
            float y = fmaf(v[e], av[e % 3], bv[e % 3]) + s[e / 3];
            if (seed) y = dropout_keep(sd, gi * E + e, rate) ? y * scale : 0.f;
            v[e] = y;
        }
        store_tri(out + gi * E, v);
    }
    if (blockIdx.x == 0) {  // the last pixels % G pixels
        for (long long p = groups * G + threadIdx.x; p < pixels; p += blockDim.x) {
            const float s = to_f32(skip[p]);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float y = fmaf(to_f32(c3[p * 3 + c]), av[c], bv[c]) + s;
                if (seed) y = dropout_keep(sd, p * 3 + c, rate) ? y * scale : 0.f;
                out[p * 3 + c] = from_f32<T>(y);
            }
        }
    }
}
template <typename T>
__global__ void __launch_bounds__(256) stem_out_bwd_kernel(const T* g, T* gout, long long pixels, float rate,
                                                           const unsigned long long* __restrict__ seed) {
    constexpr int G = Tri<T>::G, E = Tri<T>::E;
    const unsigned long long sd = seed ? *seed : 0ULL;
    const float scale = 1.0f / (1.0f - rate);
    const long long groups = pixels / G;
    for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += (long long)gridDim.x * blockDim.x) {
        float v[E];
        load_tri(g + gi * E, v);
        if (seed) {
#pragma unroll
            for (int e = 0; e < E; ++e) v[e] = dropout_keep(sd, gi * E + e, rate) ? v[e] * scale : 0.f;
        }
        store_tri(gout + gi * E, v);
    }
    if (blockIdx.x == 0) {
        for (long long p = groups * G + threadIdx.x; p < pixels; p += blockDim.x) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float v = to_f32(g[p * 3 + c]);
                if (seed) v = dropout_keep(sd, p * 3 + c, rate) ? v * scale : 0.f;
                gout[p * 3 + c] = from_f32<T>(v);
            }
        }
    }
}

// ---- BatchNorm backward for 3-channel tensors ----
template <typename T>
__global__ void __launch_bounds__(256) bn3_bwd_reduce_kernel(const T* __restrict__ g, const T* __restrict__ z,
                                                             const float* __restrict__ mean,
                                                             const float* __restrict__ rstd,
                                                             long long* __restrict__ stats, long long pixels) {
    constexpr int G = Tri<T>::G, E = Tri<T>::E;
    float s[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float mv[3] = {mean[0], mean[1], mean[2]}, rv[3] = {rstd[0], rstd[1], rstd[2]};
    const long long groups = pixels / G;
    for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += (long long)gridDim.x * blockDim.x) {
        float gv[E], zv[E];
        load_tri(g + gi * E, gv);
        load_tri(z + gi * E, zv);
#pragma unroll
        for (int e = 0; e < E; ++e) {
            s[e % 3] += gv[e];
            s[3 + e % 3] = fmaf(gv[e], (zv[e] - mv[e % 3]) * rv[e % 3], s[3 + e % 3]);
        }
    }
    if (blockIdx.x == 0) {
        for (long long p = groups * G + threadIdx.x; p < pixels; p += blockDim.x) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float gv = to_f32(g[p * 3 + c]);
                s[c] += gv;
                s[3 + c] = fmaf(gv, (to_f32(z[p * 3 + c]) - mv[c]) * rv[c], s[3 + c]);
            }
        }
    }
    __shared__ float red[8][6];  // per-warp partials, summed in warp order (run-to-run identical)
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const float v = warp_sum(s[i]);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        float t = 0.f;
        for (int w_ = 0; w_ < (int)(blockDim.x >> 5); ++w_) t += red[w_][threadIdx.x];
        stat_add(stats, threadIdx.x, (double)t);
    }
}
template <typename T>
__global__ void __launch_bounds__(256) bn3_bwd_dz_kernel(const T* g, const T* __restrict__ z, const float* __restrict__ a,
                                                         const float* __restrict__ mean, const float* __restrict__ rstd,
                                                         const float* __restrict__ c1, const float* __restrict__ c2, T* out,
                                                         long long pixels) {
    constexpr int G = Tri<T>::G, E = Tri<T>::E;
    float av[3], mv[3], rv[3], c1v[3], c2v[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) { av[c] = a[c]; mv[c] = mean[c]; rv[c] = rstd[c]; c1v[c] = c1[c]; c2v[c] = c2[c]; }
    const long long groups = pixels / G;
    for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += (long long)gridDim.x * blockDim.x) {
        float gv[E], zv[E];
        load_tri(g + gi * E, gv);
        load_tri(z + gi * E, zv);
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const float xh = (zv[e] - mv[e % 3]) * rv[e % 3];
            gv[e] = av[e % 3] * (gv[e] - c1v[e % 3] - xh * c2v[e % 3]);
        }
        store_tri(out + gi * E, gv);
    }
    if (blockIdx.x == 0) {
        for (long long p = groups * G + threadIdx.x; p < pixels; p += blockDim.x) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float xh = (to_f32(z[p * 3 + c]) - mv[c]) * rv[c];
                out[p * 3 + c] = from_f32<T>(av[c] * (to_f32(g[p * 3 + c]) - c1v[c] - xh * c2v[c]));
            }
        }
    }
}

int persist_grid(long long n) {
    long long g = (n + 255) / 256;
    const long long cap = (long long)spnet_num_sms() * 4;
    return (int)(g < cap ? (g < 1 ? 1 : g) : cap);
}
// one thread per group of 8 (bf16) / 4 (fp32) pixels; at most one resident wave (the kernels stride over the groups)
int tri_grid(long long pixels, int dtype) {
    const long long groups = pixels / (dtype == SPNET_BF16 ? 8 : 4);
    long long g = (groups + 255) / 256;
    const long long cap = (long long)spnet_num_sms() * 8;
    return (int)(g < cap ? (g < 1 ? 1 : g) : cap);
}

}  // namespace

extern "C" {

int spnet_stem_k3_to_k4(const float* k3, float* k4, int cout, cudaStream_t stream) {
    SPNET_REQUIRE(k3 && k4 && cout > 0, "stem_k3_to_k4: bad args");
    stem_k3_to_k4_kernel<<<ceil_div(16 * cout, 64), 64, 0, stream>>>(k3, k4, cout);
    return spnet_check_launch("stem_k3_to_k4");
}
// g3 += fold(g4)
int spnet_stem_k4grad_to_k3grad(const float* g4, float* g3, int cout, cudaStream_t stream) {
    SPNET_REQUIRE(g4 && g3 && cout > 0, "stem_k4grad_to_k3grad: bad args");
    stem_k4grad_to_k3grad_kernel<<<ceil_div(9 * cout, 64), 64, 0, stream>>>(g4, g3, cout);
    return spnet_check_launch("stem_k4grad_to_k3grad");
}

// d = dropout(a*c3 + b + skip);  seed nullable (= inference / rate 0: no dropout)
int spnet_stem_out_fwd(const void* c3, const float* a, const float* b, const void* skip, void* out, int dtype,
                       long long pixels, float rate, const unsigned long long* seed, cudaStream_t stream) {
    SPNET_REQUIRE(c3 && a && b && skip && out && pixels > 0 && rate >= 0.f && rate < 1.f, "stem_out_fwd: bad args");
    SPNET_DISPATCH_DTYPE(dtype, (stem_out_fwd_kernel<T><<<tri_grid(pixels, dtype), 256, 0, stream>>>(
                                    reinterpret_cast<const T*>(c3), a, b, reinterpret_cast<const T*>(skip),
                                    reinterpret_cast<T*>(out), pixels, rate, seed)));
    return spnet_check_launch("stem_out_fwd");
}
int spnet_stem_out_bwd(const void* g, void* gout, int dtype, long long pixels, float rate,
                       const unsigned long long* seed, cudaStream_t stream) {
    SPNET_REQUIRE(g && gout && pixels > 0 && rate >= 0.f && rate < 1.f, "stem_out_bwd: bad args");
    SPNET_DISPATCH_DTYPE(dtype, (stem_out_bwd_kernel<T><<<tri_grid(pixels, dtype), 256, 0, stream>>>(
                                    reinterpret_cast<const T*>(g), reinterpret_cast<T*>(gout), pixels, rate, seed)));
    return spnet_check_launch("stem_out_bwd");
}

int spnet_bn3_bwd_reduce(const void* g, const void* z, const float* save_mean, const float* save_rstd, long long* stats,
                         int dtype, long long pixels, cudaStream_t stream) {
    SPNET_REQUIRE(g && z && save_mean && save_rstd && stats && pixels > 0, "bn3_bwd_reduce: bad args");
    SPNET_DISPATCH_DTYPE(dtype, (bn3_bwd_reduce_kernel<T><<<persist_grid(pixels), 256, 0, stream>>>(
                                    reinterpret_cast<const T*>(g), reinterpret_cast<const T*>(z), save_mean, save_rstd,
                                    stats, pixels)));
    return spnet_check_launch("bn3_bwd_reduce");
}
int spnet_bn3_bwd_dz(const void* g, const void* z, const float* a, const float* save_mean, const float* save_rstd,
                     const float* c1, const float* c2, void* out, int dtype, long long pixels, cudaStream_t stream) {
    SPNET_REQUIRE(g && z && a && save_mean && save_rstd && c1 && c2 && out && pixels > 0, "bn3_bwd_dz: bad args");
    SPNET_DISPATCH_DTYPE(dtype, (bn3_bwd_dz_kernel<T><<<tri_grid(pixels, dtype), 256, 0, stream>>>(
                                    reinterpret_cast<const T*>(g), reinterpret_cast<const T*>(z), a, save_mean, save_rstd,
                                    c1, c2, reinterpret_cast<T*>(out), pixels)));
    return spnet_check_launch("bn3_bwd_dz");
}

}  // extern "C"
