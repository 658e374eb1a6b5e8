// Generic pieces for the dense-convolution backbone (keras.applications.InceptionResNetV2 behind
// spnet/models.py:18,357-359 — BASELINE configs[3]): im2col / col2im for an arbitrary kh x kw, stride
// and TF padding (the GEMM itself is gemm_tc.cu / gemm_simt.cu; Xception's block1_conv2 uses the pair
// too in the fp32 and deterministic modes), 'valid' max-pooling entry points,
// AveragePooling2D(3, 1, 'same'), channel-slice copies for Concatenate, the scaled residual
// `x + scale * (up + bias)` (+ReLU) of the Inception-ResNet blocks, accumulation and column sums.
// All HBM-bound element-wise work on 16-byte channel vectors (C % 8 == 0 for bf16, % 4 for fp32).
#include "common.cuh"

namespace {

constexpr int kT = 256;

template <typename T> __device__ __forceinline__ void zero_vec(float (&v)[VecN<T>::N]) {
#pragma unroll
    for (int i = 0; i < VecN<T>::N; ++i) v[i] = 0.f;
}

// col[(b,oh,ow), (kh*KW+kw)*C + c] = in[b, oh*sh-pt+kh, ow*sw-pl+kw, c]  (zero outside the image)
template <typename T>
__global__ void __launch_bounds__(kT) im2col_kernel(const T* __restrict__ in, T* __restrict__ col, int B, int H, int W,
                                                    int C, int KH, int KW, int sh, int sw, int pt, int pl, int OH,
                                                    int OW, long long n) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    for (long long idx = (long long)blockIdx.x * kT + threadIdx.x; idx < n; idx += (long long)gridDim.x * kT) {
        const int cv = (int)(idx % CV);
        long long r = idx / CV;
        const int kw = (int)(r % KW); r /= KW;
        const int kh = (int)(r % KH); r /= KH;
        const int ow = (int)(r % OW); r /= OW;
        const int oh = (int)(r % OH);
        const int b = (int)(r / OH);
        const int ih = oh * sh - pt + kh, iw = ow * sw - pl + kw;
        float v[V];
        zero_vec<T>(v);
        if (ih >= 0 && ih < H && iw >= 0 && iw < W) load_vec(in + (((size_t)b * H + ih) * W + iw) * C + cv * V, v);
        store_vec(col + idx * V, v);
    }
}

// gin[b,ih,iw,c] (+)= sum over (kh,kw,oh,ow) with oh*sh-pt+kh == ih, ow*sw-pl+kw == iw of gcol[...]
template <typename T>
__global__ void __launch_bounds__(kT) col2im_kernel(const T* __restrict__ gcol, T* __restrict__ gin, int accumulate,
                                                    int B, int H, int W, int C, int KH, int KW, int sh, int sw, int pt,
                                                    int pl, int OH, int OW, long long n) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    const size_t krow = (size_t)KH * KW * C;
    for (long long idx = (long long)blockIdx.x * kT + threadIdx.x; idx < n; idx += (long long)gridDim.x * kT) {
        const int cv = (int)(idx % CV);
        long long r = idx / CV;
        const int iw = (int)(r % W); r /= W;
        const int ih = (int)(r % H);
        const int b = (int)(r / H);
        float acc[V];
        zero_vec<T>(acc);
        if (accumulate) load_vec(gin + idx * V, acc);
        for (int kh = 0; kh < KH; ++kh) {
            const int t = ih + pt - kh;
            if (t < 0 || t % sh != 0) continue;
            const int oh = t / sh;
            if (oh >= OH) continue;
            for (int kw = 0; kw < KW; ++kw) {
                const int u = iw + pl - kw;
                if (u < 0 || u % sw != 0) continue;
                const int ow = u / sw;
                if (ow >= OW) continue;
                float g[V];
                load_vec(gcol + (((size_t)b * OH + oh) * OW + ow) * krow + (size_t)(kh * KW + kw) * C + cv * V, g);
#pragma unroll
                for (int i = 0; i < V; ++i) acc[i] += g[i];
            }
        }
        store_vec(gin + idx * V, acc);
    }
}

// AveragePooling2D(3, strides 1, 'same'): TF divides by the number of in-image cells of the window.
// BWD = false: out = avg3x3(in);  BWD = true: out (+)= sum over the windows containing the pixel of g / count(window)
template <typename T, bool BWD>
__global__ void __launch_bounds__(kT) avgpool3s1_kernel(const T* __restrict__ in, T* __restrict__ out, int accumulate, int B,
                                                        int H, int W, int C, long long n) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    for (long long idx = (long long)blockIdx.x * kT + threadIdx.x; idx < n; idx += (long long)gridDim.x * kT) {
        const int cv = (int)(idx % CV);
        long long r = idx / CV;
        const int w = (int)(r % W); r /= W;
        const int h = (int)(r % H);
        const int b = (int)(r / H);
        float acc[V];
        zero_vec<T>(acc);
        if (BWD && accumulate) load_vec(out + idx * V, acc);
        const int cnt_self = (min(h + 1, H - 1) - max(h - 1, 0) + 1) * (min(w + 1, W - 1) - max(w - 1, 0) + 1);
        float s[V];
        zero_vec<T>(s);
        for (int dh = -1; dh <= 1; ++dh) {
            const int hh = h + dh;
            if (hh < 0 || hh >= H) continue;
            for (int dw = -1; dw <= 1; ++dw) {
                const int ww = w + dw;
                if (ww < 0 || ww >= W) continue;
                float v[V];
                load_vec(in + (((size_t)b * H + hh) * W + ww) * C + cv * V, v);
                float wgt = 1.f;
                if (BWD) {  // the window centred at (hh, ww) divides by ITS cell count
                    const int cnt = (min(hh + 1, H - 1) - max(hh - 1, 0) + 1) * (min(ww + 1, W - 1) - max(ww - 1, 0) + 1);
                    wgt = 1.f / (float)cnt;
                }
#pragma unroll
                for (int i = 0; i < V; ++i) s[i] = fmaf(v[i], wgt, s[i]);
            }
        }
        const float inv = BWD ? 1.f : 1.f / (float)cnt_self;
#pragma unroll
        for (int i = 0; i < V; ++i) acc[i] = fmaf(s[i], inv, acc[i]);
        store_vec(out + idx * V, acc);
    }
}

// dst[r, 0:cols] (+)= src[r, 0:cols] with independent row pitches (Concatenate and its adjoint)
template <typename T>
__global__ void __launch_bounds__(kT) copy2d_kernel(const T* __restrict__ src, long long ld_src, T* __restrict__ dst,
                                                    long long ld_dst, int accumulate, long long rows, int cols) {
    constexpr int V = VecN<T>::N;
    const int CV = cols / V;
    const long long n = rows * CV;
    for (long long idx = (long long)blockIdx.x * kT + threadIdx.x; idx < n; idx += (long long)gridDim.x * kT) {
        const int cv = (int)(idx % CV);
        const long long r = idx / CV;
        float v[V];
        load_vec(src + r * ld_src + cv * V, v);
        if (accumulate) {
            float d[V];
            load_vec(dst + r * ld_dst + cv * V, d);
#pragma unroll
            for (int i = 0; i < V; ++i) v[i] += d[i];
        }
        store_vec(dst + r * ld_dst + cv * V, v);
    }
}

// y = act(x + scale * (u + bias))      (Inception-ResNet block tail; relu = 0/1)
template <typename T>
__global__ void __launch_bounds__(kT) residual_fwd_kernel(const T* __restrict__ x, const T* __restrict__ u,
                                                          const float* __restrict__ bias, float scale, int relu,
                                                          T* __restrict__ y, long long rows, int C) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    const long long n = rows * CV;
    for (long long idx = (long long)blockIdx.x * kT + threadIdx.x; idx < n; idx += (long long)gridDim.x * kT) {
        const int c0 = (int)(idx % CV) * V;
        float xv[V], uv[V];
        load_vec(x + idx * V, xv);
        load_vec(u + idx * V, uv);
#pragma unroll
        for (int i = 0; i < V; ++i) {
            float v = fmaf(scale, uv[i] + (bias ? bias[c0 + i] : 0.f), xv[i]);
            xv[i] = relu ? fmaxf(v, 0.f) : v;
        }
        store_vec(y + idx * V, xv);
    }
}

// gm = gy * (y > 0 if relu);  gx (+)= gm;  gu = scale * gm
template <typename T>
__global__ void __launch_bounds__(kT) residual_bwd_kernel(const T* __restrict__ gy, const T* __restrict__ y, float scale,
                                                          int relu, T* __restrict__ gx, int accumulate_gx,
                                                          T* __restrict__ gu, long long n_vec) {
    constexpr int V = VecN<T>::N;
    for (long long idx = (long long)blockIdx.x * kT + threadIdx.x; idx < n_vec; idx += (long long)gridDim.x * kT) {
        float g[V], yv[V], a[V];
        load_vec(gy + idx * V, g);
        if (relu) {
            load_vec(y + idx * V, yv);
#pragma unroll
            for (int i = 0; i < V; ++i)
                if (!(yv[i] > 0.f)) g[i] = 0.f;
        }
        if (accumulate_gx) {
            load_vec(gx + idx * V, a);
#pragma unroll
            for (int i = 0; i < V; ++i) a[i] += g[i];
        } else {
#pragma unroll
            for (int i = 0; i < V; ++i) a[i] = g[i];
        }
        store_vec(gx + idx * V, a);
#pragma unroll
        for (int i = 0; i < V; ++i) g[i] *= scale;
        store_vec(gu + idx * V, g);
    }
}

// out[c] += sum_r g[r, c]   (bias gradient; out is fp32 and zeroed by the caller)
// blockIdx.y = chunk of cvb channel vectors; thread t -> vector t % cvb of row lane t / cvb
// acc == nullptr: fp32 partial sums per thread, added into out with float atomics (order of the adds not fixed).
// acc != nullptr: every element is split into the fixed-point limbs of the order-independent accumulators
// (common.cuh stat_limbs), summed as integers per thread and added into acc[c] with integer atomics: the result
// does not depend on the order of the rows or of the CTAs (spnet_acc_to_f32 then adds acc into out)
template <typename T>
__global__ void __launch_bounds__(kT) colsum_rows_kernel(const T* __restrict__ g, float* __restrict__ out,
                                                         long long* __restrict__ acc_out, long long rows, int C, int cvb,
                                                         int per) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    const int cv = blockIdx.y * cvb + threadIdx.x % cvb, rl = threadIdx.x / cvb;
    if (rl >= per || cv >= CV) return;
    if (acc_out) {
        long long hi[V];
        unsigned long long lo[V];
#pragma unroll
        for (int i = 0; i < V; ++i) hi[i] = 0, lo[i] = 0;
        for (long long r = (long long)blockIdx.x * per + rl; r < rows; r += (long long)gridDim.x * per) {
            float v[V];
            load_vec(g + r * C + cv * V, v);
#pragma unroll
            for (int i = 0; i < V; ++i) {
                long long h;
                unsigned long long l;
                stat_limbs((double)v[i], h, l);
                hi[i] += h;
                lo[i] += l;
            }
        }
        unsigned long long* p = reinterpret_cast<unsigned long long*>(acc_out) + 2 * (cv * V);
#pragma unroll
        for (int i = 0; i < V; ++i) {
            atomicAdd(p + 2 * i, (unsigned long long)hi[i]);
            if (lo[i]) atomicAdd(p + 2 * i + 1, lo[i]);
        }
        return;
    }
    float acc[V];
    zero_vec<T>(acc);
    for (long long r = (long long)blockIdx.x * per + rl; r < rows; r += (long long)gridDim.x * per) {
        float v[V];
        load_vec(g + r * C + cv * V, v);
#pragma unroll
        for (int i = 0; i < V; ++i) acc[i] += v[i];
    }
#pragma unroll
    for (int i = 0; i < V; ++i) atomicAdd(out + cv * V + i, acc[i]);
}

int grid_for_n(long long n) {
    long long g = (n + kT - 1) / kT;
    const long long cap = (long long)spnet_num_sms() * 16;
    return (int)(g < cap ? (g < 1 ? 1 : g) : cap);
}

int chk(const char* who, int dtype, int C) {
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    SPNET_REQUIRE(C > 0 && C % V == 0, "%s: C=%d must be a multiple of %d", who, C, V);
    return SPNET_OK;
}

}  // namespace

extern "C" {

// out dims: OH = (H + pt + pb - KH)/sh + 1 with TF padding decided by the caller (pt, pl = leading pads;
// trailing pads are implied by OH, OW). col: [B*OH*OW, KH*KW*C].
int spnet_im2col(const void* in, void* col, int dtype, int B, int H, int W, int C, int KH, int KW, int sh, int sw, int pt,
                 int pl, int OH, int OW, cudaStream_t stream) {
    int rc = chk("im2col", dtype, C);
    if (rc) return rc;
    SPNET_REQUIRE(in && col && B > 0 && H > 0 && W > 0 && KH > 0 && KW > 0 && sh > 0 && sw > 0 && OH > 0 && OW > 0,
                  "im2col: bad args");
    const long long n = (long long)B * OH * OW * KH * KW * (C / (dtype == SPNET_BF16 ? 8 : 4));
    SPNET_DISPATCH_DTYPE(dtype, (im2col_kernel<T><<<grid_for_n(n), kT, 0, stream>>>(
                                    reinterpret_cast<const T*>(in), reinterpret_cast<T*>(col), B, H, W, C, KH, KW, sh, sw, pt,
                                    pl, OH, OW, n)));
    return spnet_check_launch("im2col");
}

int spnet_col2im(const void* gcol, void* gin, int accumulate, int dtype, int B, int H, int W, int C, int KH, int KW, int sh,
                 int sw, int pt, int pl, int OH, int OW, cudaStream_t stream) {
    int rc = chk("col2im", dtype, C);
    if (rc) return rc;
    SPNET_REQUIRE(gcol && gin && B > 0 && H > 0 && W > 0 && KH > 0 && KW > 0 && sh > 0 && sw > 0 && OH > 0 && OW > 0,
                  "col2im: bad args");
    const long long n = (long long)B * H * W * (C / (dtype == SPNET_BF16 ? 8 : 4));
    SPNET_DISPATCH_DTYPE(dtype, (col2im_kernel<T><<<grid_for_n(n), kT, 0, stream>>>(
                                    reinterpret_cast<const T*>(gcol), reinterpret_cast<T*>(gin), accumulate, B, H, W, C, KH,
                                    KW, sh, sw, pt, pl, OH, OW, n)));
    return spnet_check_launch("col2im");
}

// AveragePooling2D(3, 1, 'same'), forward (bwd = 0) or backward (bwd = 1: out (+)= adjoint applied to in)
int spnet_avgpool3s1(const void* in, void* out, int bwd, int accumulate, int dtype, int B, int H, int W, int C,
                     cudaStream_t stream) {
    int rc = chk("avgpool3s1", dtype, C);
    if (rc) return rc;
    SPNET_REQUIRE(in && out && B > 0 && H > 0 && W > 0, "avgpool3s1: bad args");
    const long long n = (long long)B * H * W * (C / (dtype == SPNET_BF16 ? 8 : 4));
    if (bwd) {
        SPNET_DISPATCH_DTYPE(dtype, (avgpool3s1_kernel<T, true><<<grid_for_n(n), kT, 0, stream>>>(
                                        reinterpret_cast<const T*>(in), reinterpret_cast<T*>(out), accumulate, B, H, W, C, n)));
    } else {
        SPNET_DISPATCH_DTYPE(dtype, (avgpool3s1_kernel<T, false><<<grid_for_n(n), kT, 0, stream>>>(
                                        reinterpret_cast<const T*>(in), reinterpret_cast<T*>(out), 0, B, H, W, C, n)));
    }
    return spnet_check_launch("avgpool3s1");
}

// dst[r, 0:cols] (+)= src[r, 0:cols];  ld_* in elements (multiples of the 16-byte vector)
int spnet_copy2d(const void* src, long long ld_src, void* dst, long long ld_dst, int accumulate, int dtype, long long rows,
                 int cols, cudaStream_t stream) {
    int rc = chk("copy2d", dtype, cols);
    if (rc) return rc;
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    SPNET_REQUIRE(src && dst && rows > 0 && ld_src % V == 0 && ld_dst % V == 0, "copy2d: bad args");
    const long long n = rows * (cols / V);
    SPNET_DISPATCH_DTYPE(dtype, (copy2d_kernel<T><<<grid_for_n(n), kT, 0, stream>>>(
                                    reinterpret_cast<const T*>(src), ld_src, reinterpret_cast<T*>(dst), ld_dst, accumulate,
                                    rows, cols)));
    return spnet_check_launch("copy2d");
}

int spnet_residual_fwd(const void* x, const void* u, const float* bias, float scale, int relu, void* y, int dtype,
                       long long rows, int C, cudaStream_t stream) {
    int rc = chk("residual_fwd", dtype, C);
    if (rc) return rc;
    SPNET_REQUIRE(x && u && y && rows > 0, "residual_fwd: bad args");
    const long long n = rows * (C / (dtype == SPNET_BF16 ? 8 : 4));
    SPNET_DISPATCH_DTYPE(dtype, (residual_fwd_kernel<T><<<grid_for_n(n), kT, 0, stream>>>(
                                    reinterpret_cast<const T*>(x), reinterpret_cast<const T*>(u), bias, scale, relu,
                                    reinterpret_cast<T*>(y), rows, C)));
    return spnet_check_launch("residual_fwd");
}

int spnet_residual_bwd(const void* gy, const void* y, float scale, int relu, void* gx, int accumulate_gx, void* gu,
                       int dtype, long long rows, int C, cudaStream_t stream) {
    int rc = chk("residual_bwd", dtype, C);
    if (rc) return rc;
    SPNET_REQUIRE(gy && y && gx && gu && rows > 0, "residual_bwd: bad args");
    const long long n = rows * (C / (dtype == SPNET_BF16 ? 8 : 4));
    SPNET_DISPATCH_DTYPE(dtype, (residual_bwd_kernel<T><<<grid_for_n(n), kT, 0, stream>>>(
                                    reinterpret_cast<const T*>(gy), reinterpret_cast<const T*>(y), scale, relu,
                                    reinterpret_cast<T*>(gx), accumulate_gx, reinterpret_cast<T*>(gu), n)));
    return spnet_check_launch("residual_bwd");
}

// out[c] += sum over rows of g[r, c]   (fp32 out, zeroed by the caller). acc (nullable): the sums go to these
// order-independent accumulators instead (C entries, zero; spnet_acc_to_f32 adds them into out and clears them)
int spnet_colsum_rows(const void* g, float* out, long long* acc, int dtype, long long rows, int C, cudaStream_t stream) {
    int rc = chk("colsum_rows", dtype, C);
    if (rc) return rc;
    const int CV = C / (dtype == SPNET_BF16 ? 8 : 4);
    SPNET_REQUIRE(g && out && rows > 0, "colsum_rows: bad args");
    const int chunks = ceil_div(CV, 128);
    const int cvb = ceil_div(CV, chunks);
    const int per = kT / cvb;
    long long gx = (rows + (long long)per * 32 - 1) / ((long long)per * 32);  // >= 32 rows per thread: the float atomics at the
    if (gx > 64) gx = 64;                                                    // end serialise per address (64-deep at most)
    if (gx < 1) gx = 1;
    SPNET_DISPATCH_DTYPE(dtype, (colsum_rows_kernel<T><<<dim3((unsigned)gx, chunks), kT, 0, stream>>>(
                                    reinterpret_cast<const T*>(g), out, acc, rows, C, cvb, per)));
    return spnet_check_launch("colsum_rows");
}

// MaxPooling2D(3, strides 2, 'valid') (Inception-ResNet reductions): the 'same' kernels of pool.cu with zero
// leading padding and OH = (H-3)/2+1 are reached through spnet_maxpool3s2_valid_{fwd,bwd} there.

}  // extern "C"
