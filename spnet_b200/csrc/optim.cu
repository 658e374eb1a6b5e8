// Optimiser and parameter utilities.
//  * Adam in the Keras 2.1.3 form used by the reference (spnet/models.py:494:
//    Adam(lr=1e-5), beta=(0.9,0.999), eps=K.epsilon()=1e-7):
//        lr_t = lr*sqrt(1-b2^t)/(1-b1^t);  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2
//        p   -= lr_t * m / (sqrt(v) + eps)         <- eps outside the bias correction
//    fused with the L2 regulariser gradient of add_regularization (spnet/models.py:47-71:
//    1e-4*sum(w^2) on 10 kernels -> + 2e-4*w) and with the refresh of the bf16 working copy.
//  * sum of squares (the L2 term of the reported loss), casts, bias fill, column sums.
#include "common.cuh"

namespace {

// params live in one flat fp32 buffer; the L2-regularised tensors occupy [0, n_l2).
// HBM-bound (28 B read+written per parameter + 2 B bf16 copy): 16-byte accesses, two independent
// vectors per thread in flight. Buffers must be 16-byte aligned (8-byte for the bf16 copy).
__device__ __forceinline__ float adam_one(float& p, float g, float& m, float& v, bool reg, float l2x2, float lr_t,
                                          float beta1, float beta2, float eps, float grad_scale) {
    float gi = g * grad_scale;
    if (reg) gi = fmaf(l2x2, p, gi);
    m = beta1 * m + (1.0f - beta1) * gi;
    v = beta2 * v + (1.0f - beta2) * gi * gi;
    p -= lr_t * m / (sqrtf(v) + eps);
    return p;
}

__global__ void __launch_bounds__(256) adam_keras_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                         float* __restrict__ m, float* __restrict__ v,
                                                         long long n, long long n_l2, float l2,
                                                         const float* __restrict__ lr_t_ptr, float beta1,
                                                         float beta2, float eps, float grad_scale,
                                                         bf16* __restrict__ p_bf16,
                                                         const unsigned char* __restrict__ frozen8,
                                                         const bf16* __restrict__ g_bf16) {
    // frozen8 (nullable): one byte per 8 parameters (every tensor is padded to 8), non-zero = the tensor is not
    // trainable (layer.trainable = False, spnet/models.py:361-372): no update, no L2 pull, moments untouched.
    // g_bf16 (nullable): the gradients come from this bf16 buffer (data-parallel all-reduce in bf16) instead of g.
    const float lr_t = *lr_t_ptr;
    const float l2x2 = 2.0f * l2;
    const long long nv = n >> 2;  // float4 vectors
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < nv; i0 += 2 * stride) {
        float4 pv[2], gv[2], mv[2], vv[2];
        bool ok[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const long long i = i0 + u * stride;
            ok[u] = i < nv && !(frozen8 && frozen8[i >> 1]);
            if (ok[u]) {
                pv[u] = reinterpret_cast<const float4*>(p)[i];
                if (g_bf16) {
                    const uint2 w = __ldcs(reinterpret_cast<const uint2*>(g_bf16) + i);
                    gv[u] = make_float4(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xffff0000u),
                                        __uint_as_float(w.y << 16), __uint_as_float(w.y & 0xffff0000u));
                } else {
                    gv[u] = __ldcs(reinterpret_cast<const float4*>(g) + i);  // gradients are dead after this read
                }
                mv[u] = reinterpret_cast<const float4*>(m)[i];
                vv[u] = reinterpret_cast<const float4*>(v)[i];
            }
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            if (!ok[u]) continue;
            const long long i = i0 + u * stride;
            const long long e = 4 * i;
            adam_one(pv[u].x, gv[u].x, mv[u].x, vv[u].x, e < n_l2, l2x2, lr_t, beta1, beta2, eps, grad_scale);
            adam_one(pv[u].y, gv[u].y, mv[u].y, vv[u].y, e + 1 < n_l2, l2x2, lr_t, beta1, beta2, eps, grad_scale);
            adam_one(pv[u].z, gv[u].z, mv[u].z, vv[u].z, e + 2 < n_l2, l2x2, lr_t, beta1, beta2, eps, grad_scale);
            adam_one(pv[u].w, gv[u].w, mv[u].w, vv[u].w, e + 3 < n_l2, l2x2, lr_t, beta1, beta2, eps, grad_scale);
            reinterpret_cast<float4*>(p)[i] = pv[u];
            reinterpret_cast<float4*>(m)[i] = mv[u];
            reinterpret_cast<float4*>(v)[i] = vv[u];
            if (p_bf16)
                reinterpret_cast<uint2*>(p_bf16)[i] = make_uint2(pack_bf16x2(pv[u].x, pv[u].y), pack_bf16x2(pv[u].z, pv[u].w));
        }
    }
    // tail (n not a multiple of 4: never the case for the engine's padded buffers)
    for (long long i = 4 * nv + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (frozen8 && frozen8[i >> 3]) continue;
        float pi = p[i], mi = m[i], vi = v[i];
        adam_one(pi, g_bf16 ? __bfloat162float(g_bf16[i]) : g[i], mi, vi, i < n_l2, l2x2, lr_t, beta1, beta2, eps, grad_scale);
        p[i] = pi; m[i] = mi; v[i] = vi;
        if (p_bf16) p_bf16[i] = __float2bfloat16_rn(pi);
    }
}

__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ p, long long n, float scale,
                                                    long long* __restrict__ out) {
    float s = 0.f;
    const long long nv = n >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
        const float4 q = reinterpret_cast<const float4*>(p)[i];
        s = fmaf(q.x, q.x, s); s = fmaf(q.y, q.y, s); s = fmaf(q.z, q.z, s); s = fmaf(q.w, q.w, s);
    }
    for (long long i = 4 * nv + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x)
        s = fmaf(p[i], p[i], s);
    __shared__ float red[8];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w];
        stat_add(out, 0, (double)t * (double)scale);  // order-independent across CTAs (common.cuh)
    }
}

// out[i] (+)= value of accumulator i (common.cuh stat_get); optionally clears the accumulators for the next step
__global__ void acc_to_f32_kernel(long long* __restrict__ acc, float* __restrict__ out, long long n, int accumulate, int clear) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = (float)stat_get(acc, i);
    out[i] = accumulate ? out[i] + v : v;
    if (clear) stat_clear(acc, i);
}

// out[r, c] = (accumulate ? out[r, c] : 0) + bias[c] + slab_0[r, c] + slab_1[r, c] + ... (that order): the second half
// of a split-K GEMM whose result must not depend on which split finished first (spnet_gemm_bf16 out_mode 3)
__global__ void __launch_bounds__(256) slab_reduce_kernel(const float* __restrict__ slabs, int nslabs, long long slab_stride,
                                                          long long lds, const float* __restrict__ bias, float* __restrict__ out,
                                                          long long ldo, int rows, int cols4, int accumulate) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)rows * cols4) return;
    const int r = (int)(i / cols4), c = (int)(i % cols4) * 4;
    float4 a = accumulate ? *reinterpret_cast<const float4*>(out + r * ldo + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) {
        const float4 b = *reinterpret_cast<const float4*>(bias + c);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
#pragma unroll 8
    for (int s = 0; s < nslabs; ++s) {  // the loads of eight slabs in flight, the adds in slab order
        const float4 v = *reinterpret_cast<const float4*>(slabs + s * slab_stride + r * lds + c);
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    *reinterpret_cast<float4*>(out + r * ldo + c) = a;
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x)
        dst[i] = __float2bfloat16_rn(src[i]);
}

// out[c] = sum_r g[r, c]   (rows small: the Dense bias gradient)
__global__ void colsum_kernel(const float* __restrict__ g, float* __restrict__ out, int rows, int cols) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    float s = 0.f;
    for (int r = 0; r < rows; ++r) s += g[(size_t)r * cols + c];
    out[c] = s;
}

int grid_for(long long n) {
    long long g = (n + 255) / 256;
    const long long cap = (long long)spnet_num_sms() * 8;
    return (int)(g < cap ? (g < 1 ? 1 : g) : cap);
}

}  // namespace

extern "C" {

int spnet_adam_keras_step(float* p, const float* g, float* m, float* v, long long n, long long n_l2, float l2,
                          const float* lr_t_dev, float beta1, float beta2, float eps, float grad_scale,
                          void* p_bf16, const unsigned char* frozen8, const void* g_bf16, cudaStream_t stream) {
    SPNET_REQUIRE(p && (g || g_bf16) && m && v && lr_t_dev && n > 0 && n_l2 >= 0 && n_l2 <= n, "adam_keras_step: bad args");
    SPNET_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0 && ((uintptr_t)p_bf16 & 7) == 0 &&
                      ((uintptr_t)g_bf16 & 7) == 0,
                  "adam_keras_step: buffers must be 16-byte aligned");
    adam_keras_kernel<<<grid_for(n), 256, 0, stream>>>(p, g, m, v, n, n_l2, l2, lr_t_dev, beta1, beta2, eps,
                                                      grad_scale, reinterpret_cast<bf16*>(p_bf16), frozen8,
                                                      reinterpret_cast<const bf16*>(g_bf16));
    return spnet_check_launch("adam_keras_step");
}

// *out += scale * sum(p^2)
int spnet_sumsq(const float* p, long long n, float scale, long long* out, cudaStream_t stream) {
    SPNET_REQUIRE(p && out && n > 0 && ((uintptr_t)p & 15) == 0, "sumsq: bad args (p must be 16-byte aligned)");
    sumsq_kernel<<<grid_for(n), 256, 0, stream>>>(p, n, scale, out);
    return spnet_check_launch("sumsq");
}

int spnet_cast_f32_to_bf16(const float* src, void* dst, long long n, cudaStream_t stream) {
    SPNET_REQUIRE(src && dst && n > 0, "cast_f32_to_bf16: bad args");
    cast_f32_bf16_kernel<<<grid_for(n), 256, 0, stream>>>(src, reinterpret_cast<bf16*>(dst), n);
    return spnet_check_launch("cast_f32_to_bf16");
}

int spnet_colsum(const float* g, float* out, int rows, int cols, cudaStream_t stream) {
    SPNET_REQUIRE(g && out && rows > 0 && cols > 0, "colsum: bad args");
    colsum_kernel<<<ceil_div(cols, 128), 128, 0, stream>>>(g, out, rows, cols);
    return spnet_check_launch("colsum");
}


int spnet_acc_to_f32(long long* acc, float* out, long long n, int accumulate, int clear, cudaStream_t stream) {
    SPNET_REQUIRE(acc && out && n > 0, "acc_to_f32: bad args");
    acc_to_f32_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(acc, out, n, accumulate, clear);
    return spnet_check_launch("acc_to_f32");
}

int spnet_slab_reduce(const float* slabs, int nslabs, long long slab_stride, long long lds, const float* bias, float* out,
                      long long ldo, int rows, int cols, int accumulate, cudaStream_t stream) {
    SPNET_REQUIRE(slabs && out && nslabs > 0 && rows > 0 && cols > 0, "slab_reduce: bad args");
    SPNET_REQUIRE(cols % 4 == 0 && lds % 4 == 0 && ldo % 4 == 0 && slab_stride % 4 == 0, "slab_reduce: cols / strides must be multiples of 4");
    SPNET_REQUIRE(((uintptr_t)slabs % 16 == 0) && ((uintptr_t)out % 16 == 0) && (!bias || (uintptr_t)bias % 16 == 0),
                  "slab_reduce: pointers must be 16-byte aligned");
    slab_reduce_kernel<<<ceil_div((long long)rows * (cols / 4), 256), 256, 0, stream>>>(slabs, nslabs, slab_stride, lds, bias, out,
                                                                                      ldo, rows, cols / 4, accumulate);
    return spnet_check_launch("slab_reduce");
}

}  // extern "C"
