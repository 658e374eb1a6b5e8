// BatchNormalization (keras axis=-1, eps 1e-3, momentum 0.99; 43 instances in the
// reference graph: spnet/models.py:326-336 and keras.applications.Xception) split into
// the pieces a fused training step needs:
//   * batch statistics are accumulated (fp64 sum / sum of squares) by the PRODUCING
//     kernel's epilogue (GEMM, small conv); bn_finalize turns them into the per-channel
//     affine  y = a*z + b  that CONSUMERS apply on load, and updates the moving stats;
//   * bn_act / bn_add materialise BN(+activation / +residual) where a tensor has to exist;
//   * backward: bn_bwd_reduce -> bn_bwd_finalize -> bn_bwd_dz.
#include "common.cuh"

namespace {

__global__ void bn_finalize_kernel(long long* __restrict__ stats, double count, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum, int unbiased,
                                   float* __restrict__ a, float* __restrict__ b, float* __restrict__ save_mean,
                                   float* __restrict__ save_rstd, float* __restrict__ moving_mean,
                                   float* __restrict__ moving_var, int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double mean = stat_get(stats, c) / count;
    double var = stat_get(stats, C + c) / count - mean * mean;
    if (var < 0.0) var = 0.0;
    stat_clear(stats, c);
    stat_clear(stats, C + c);
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float g = gamma ? gamma[c] : 1.0f;
    const float aa = g * rstd;
    a[c] = aa;
    b[c] = (beta ? beta[c] : 0.0f) - (float)mean * aa;
    save_mean[c] = (float)mean;
    save_rstd[c] = rstd;
    if (moving_mean) {
        const double uv = (unbiased && count > 1.0) ? var * count / (count - 1.0) : var;
        moving_mean[c] = momentum * moving_mean[c] + (1.0f - momentum) * (float)mean;
        moving_var[c] = momentum * moving_var[c] + (1.0f - momentum) * (float)uv;
    }
}

__global__ void bn_inference_affine_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                           const float* __restrict__ mm, const float* __restrict__ mv, float eps,
                                           float* __restrict__ a, float* __restrict__ b, float* __restrict__ save_mean,
                                           float* __restrict__ save_rstd, int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float aa = (gamma ? gamma[c] : 1.0f) / sqrtf(mv[c] + eps);
    a[c] = aa;
    b[c] = (beta ? beta[c] : 0.0f) - mm[c] * aa;
    if (save_mean) {  // a BatchNorm that normalises with its moving statistics inside a TRAINING step: backward needs them
        save_mean[c] = mm[c];
        save_rstd[c] = 1.0f / sqrtf(mv[c] + eps);
    }
}

// Channel-stationary mapping shared by the element-wise kernels below: a thread keeps one
// 16-byte channel vector (its per-channel coefficients stay in registers as fp32 pairs, fetched
// with 16-byte loads) and walks a contiguous range of rows, UNROLL independent 16-byte loads in
// flight per tensor. Tensor values stay in their raw 16-byte form until they are used and all
// arithmetic is packed fp32 (fma.rn.f32x2), which keeps the kernels at ~64 registers so that a
// whole grid is resident in ONE wave — these launches are short (tens of microseconds), a second
// wave would pay the prologue latency again.
constexpr int UNROLL = 4;

// A 16-byte vector of activations as NP fp32 pairs (bf16: 4 pairs, fp32: 2 pairs).
template <typename T> struct RawVec;
template <> struct RawVec<bf16> {
    static constexpr int NP = 4;
    uint4 r;
    __device__ __forceinline__ float2 get(int i) const {
        const uint32_t w = i == 0 ? r.x : (i == 1 ? r.y : (i == 2 ? r.z : r.w));
        return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
    }
    __device__ __forceinline__ void set(int i, float2 v) {
        const uint32_t w = pack_bf16x2(v.x, v.y);
        if (i == 0) r.x = w; else if (i == 1) r.y = w; else if (i == 2) r.z = w; else r.w = w;
    }
};
template <> struct RawVec<float> {
    static constexpr int NP = 2;
    float4 r;
    __device__ __forceinline__ float2 get(int i) const { return i == 0 ? make_float2(r.x, r.y) : make_float2(r.z, r.w); }
    __device__ __forceinline__ void set(int i, float2 v) {
        if (i == 0) { r.x = v.x; r.y = v.y; } else { r.z = v.x; r.w = v.y; }
    }
};
template <typename T> __device__ __forceinline__ RawVec<T> ld_raw(const T* p) {
    RawVec<T> v;
    v.r = *reinterpret_cast<const decltype(v.r)*>(p);
    return v;
}
template <typename T> __device__ __forceinline__ void st_raw(T* p, const RawVec<T>& v) {
    *reinterpret_cast<decltype(v.r)*>(p) = v.r;
}
// per-channel fp32 coefficients of one channel vector as pairs (c0 is a multiple of 4)
template <int NP> __device__ __forceinline__ void ld_coef(const float* __restrict__ p, int c0, float2 (&v)[NP]) {
#pragma unroll
    for (int i = 0; i < NP; i += 2) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p + c0 + 2 * i));
        v[i] = make_float2(q.x, q.y);
        v[i + 1] = make_float2(q.z, q.w);
    }
}

struct RowRange { long long begin, end; };
__device__ __forceinline__ RowRange cta_rows(long long rows) {
    // each CTA walks a CONTIGUOUS range of rows (sequential DRAM pages)
    const long long per_cta = (rows + gridDim.x - 1) / gridDim.x;
    RowRange r;
    r.begin = (long long)blockIdx.x * per_cta;
    r.end = r.begin + per_cta < rows ? r.begin + per_cta : rows;
    return r;
}

// out = act(a*z + b) [+ x];  act: 0 none, 1 relu, 2 leaky-relu(0.1), 3 relu6
template <typename T>
__global__ void __launch_bounds__(256, 3) bn_apply_kernel(const T* z, const float* __restrict__ a,
                                                          const float* __restrict__ b, int act, const T* x, T* out,
                                                          long long rows, int C, int cvb, int krows) {
    constexpr int V = VecN<T>::N, NP = RawVec<T>::NP;
    const int CV = C / V;
    const int cvl = threadIdx.x % cvb, rl = threadIdx.x / cvb;
    const int cv = blockIdx.y * cvb + cvl;
    if (cv >= CV) return;
    const int c0 = cv * V;
    float2 av[NP], bv[NP];
    ld_coef<NP>(a, c0, av);
    ld_coef<NP>(b, c0, bv);
    const RowRange rr = cta_rows(rows);
    const long long stride = krows;
    for (long long r0 = rr.begin + rl; r0 < rr.end; r0 += stride * UNROLL) {
        RawVec<T> v[UNROLL], xr[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const long long r = r0 + u * stride;
            if (r < rr.end) {
                v[u] = ld_raw(z + r * C + c0);
                if (x) xr[u] = ld_raw(x + r * C + c0);
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const long long r = r0 + u * stride;
            if (r < rr.end) {
#pragma unroll
                for (int i = 0; i < NP; ++i) {
                    float2 y = ffma2(v[u].get(i), av[i], bv[i]);
                    if (act == 1) { y.x = fmaxf(y.x, 0.f); y.y = fmaxf(y.y, 0.f); }
                    else if (act == 2) { y.x = y.x > 0.f ? y.x : 0.1f * y.x; y.y = y.y > 0.f ? y.y : 0.1f * y.y; }
                    else if (act == 3) { y.x = fminf(fmaxf(y.x, 0.f), 6.f); y.y = fminf(fmaxf(y.y, 0.f), 6.f); }
                    if (x) y = fadd2(y, xr[u].get(i));
                    v[u].set(i, y);
                }
                st_raw(out + r * C + c0, v[u]);
            }
        }
    }
}

// stats[c] += sum g, stats[C+c] += sum g*xhat, xhat = (z-mean)*rstd.
// If relu_a is given, g is first masked in place by (relu_a*z+relu_b > 0) (act 1) or scaled
// by the leaky slope (act 2): the gradient of the activation that followed this BN.
template <typename T, bool MASKED>
__global__ void __launch_bounds__(512, 1) bn_bwd_reduce_kernel(T* __restrict__ g, const T* __restrict__ z,
                                                               const float* __restrict__ mean,
                                                               const float* __restrict__ rstd,
                                                               const float* __restrict__ relu_a,
                                                               const float* __restrict__ relu_b, int act,
                                                               long long* __restrict__ stats, long long rows, int C,
                                                               int cvb, int krows) {
    constexpr int V = VecN<T>::N, NP = RawVec<T>::NP;
    const int CV = C / V;
    const int cvl = threadIdx.x % cvb, rl = threadIdx.x / cvb;
    const int cv = blockIdx.y * cvb + cvl;
    const bool active = cv < CV;
    const int c0 = cv * V;
    float2 s1[NP], s2[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) s1[i] = s2[i] = make_float2(0.f, 0.f);
    if (active) {
        float2 rs[NP], nm[NP], ra[NP], rb[NP];  // xhat = z*rs + nm,  nm = -mean*rs
        ld_coef<NP>(rstd, c0, rs);
        ld_coef<NP>(mean, c0, nm);
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            nm[i] = make_float2(-nm[i].x * rs[i].x, -nm[i].y * rs[i].y);
            ra[i] = rb[i] = make_float2(0.f, 0.f);
        }
        if (MASKED) {
            ld_coef<NP>(relu_a, c0, ra);
            ld_coef<NP>(relu_b, c0, rb);
        }
        const RowRange rr = cta_rows(rows);
        const long long stride = krows;
        for (long long r0 = rr.begin + rl; r0 < rr.end; r0 += stride * UNROLL) {
            RawVec<T> gv[UNROLL], zv[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const long long r = r0 + u * stride;
                if (r < rr.end) {
                    gv[u] = ld_raw(g + r * C + c0);
                    zv[u] = ld_raw(z + r * C + c0);
                }
            }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const long long r = r0 + u * stride;
                if (r >= rr.end) continue;
                if (MASKED) {
#pragma unroll
                    for (int i = 0; i < NP; ++i) {
                        const float2 y = ffma2(zv[u].get(i), ra[i], rb[i]);
                        float2 gg = gv[u].get(i);
                        if (act == 3) {  // relu6: open only inside (0, 6)
                            if (!(y.x > 0.f && y.x < 6.f)) gg.x = 0.f;
                            if (!(y.y > 0.f && y.y < 6.f)) gg.y = 0.f;
                        } else {
                            if (!(y.x > 0.f)) gg.x = (act == 2) ? 0.1f * gg.x : 0.f;
                            if (!(y.y > 0.f)) gg.y = (act == 2) ? 0.1f * gg.y : 0.f;
                        }
                        gv[u].set(i, gg);  // re-rounded to T: the sums below use the value as it will be re-read
                    }
                    st_raw(g + r * C + c0, gv[u]);
                }
#pragma unroll
                for (int i = 0; i < NP; ++i) {
                    const float2 gg = gv[u].get(i);
                    s1[i] = fadd2(s1[i], gg);
                    s2[i] = ffma2(gg, ffma2(zv[u].get(i), rs[i], nm[i]), s2[i]);
                }
            }
        }
    }
    __shared__ float red[2][512 * 8];
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        red[0][threadIdx.x * V + 2 * i] = s1[i].x; red[0][threadIdx.x * V + 2 * i + 1] = s1[i].y;
        red[1][threadIdx.x * V + 2 * i] = s2[i].x; red[1][threadIdx.x * V + 2 * i + 1] = s2[i].y;
    }
    __syncthreads();
    if (rl == 0 && active) {
#pragma unroll
        for (int i = 0; i < V; ++i) {
            float t1 = 0.f, t2 = 0.f;
            for (int j = 0; j < krows; ++j) {
                t1 += red[0][(j * cvb + cvl) * V + i];
                t2 += red[1][(j * cvb + cvl) * V + i];
            }
            stat_add(stats, c0 + i, (double)t1);
            stat_add(stats, C + c0 + i, (double)t2);
        }
    }
}

// stats[c] += sum z, stats[C+c] += sum z^2 over the rows (batch statistics of a tensor whose producer
// has no statistics epilogue)
template <typename T>
__global__ void __launch_bounds__(512, 1) colstats_kernel(const T* __restrict__ z, long long* __restrict__ stats,
                                                          long long rows, int C, int cvb, int krows) {
    constexpr int V = VecN<T>::N, NP = RawVec<T>::NP;
    const int CV = C / V;
    const int cvl = threadIdx.x % cvb, rl = threadIdx.x / cvb;
    const int cv = blockIdx.y * cvb + cvl;
    const bool active = cv < CV;
    const int c0 = cv * V;
    float2 s1[NP], s2[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) s1[i] = s2[i] = make_float2(0.f, 0.f);
    if (active) {
        const RowRange rr = cta_rows(rows);
        const long long stride = krows;
        for (long long r0 = rr.begin + rl; r0 < rr.end; r0 += stride * UNROLL) {
            RawVec<T> zv[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const long long r = r0 + u * stride;
                if (r < rr.end) zv[u] = ld_raw(z + r * C + c0);
            }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const long long r = r0 + u * stride;
                if (r >= rr.end) continue;
#pragma unroll
                for (int i = 0; i < NP; ++i) {
                    const float2 v = zv[u].get(i);
                    s1[i] = fadd2(s1[i], v);
                    s2[i] = ffma2(v, v, s2[i]);
                }
            }
        }
    }
    __shared__ float red[2][512 * 8];
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        red[0][threadIdx.x * V + 2 * i] = s1[i].x; red[0][threadIdx.x * V + 2 * i + 1] = s1[i].y;
        red[1][threadIdx.x * V + 2 * i] = s2[i].x; red[1][threadIdx.x * V + 2 * i + 1] = s2[i].y;
    }
    __syncthreads();
    if (rl == 0 && active) {
#pragma unroll
        for (int i = 0; i < V; ++i) {
            float t1 = 0.f, t2 = 0.f;
            for (int j = 0; j < krows; ++j) {
                t1 += red[0][(j * cvb + cvl) * V + i];
                t2 += red[1][(j * cvb + cvl) * V + i];
            }
            stat_add(stats, c0 + i, (double)t1);
            stat_add(stats, C + c0 + i, (double)t2);
        }
    }
}

__global__ void bn_bwd_finalize_kernel(long long* __restrict__ stats, double count, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta, float* __restrict__ c1, float* __restrict__ c2,
                                       int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double sg = stat_get(stats, c), sgx = stat_get(stats, C + c);
    stat_clear(stats, c);
    stat_clear(stats, C + c);
    if (dgamma) dgamma[c] = (float)sgx;
    if (dbeta) dbeta[c] = (float)sg;
    // count <= 0: the BatchNorm normalised with fixed (moving) statistics in this step - no batch-statistics terms
    c1[c] = count > 0.0 ? (float)(sg / count) : 0.f;
    c2[c] = count > 0.0 ? (float)(sgx / count) : 0.f;
}

// out = a * (g - c1 - xhat*c2) = A*g + Bz*z + D with per-channel A = a, Bz = -a*rstd*c2,
// D = a*(rstd*c2*mean - c1)
template <typename T>
__global__ void __launch_bounds__(256, 3) bn_bwd_dz_kernel(const T* g, const T* __restrict__ z,
                                                           const float* __restrict__ a,
                                                           const float* __restrict__ mean,
                                                           const float* __restrict__ rstd,
                                                           const float* __restrict__ c1,
                                                           const float* __restrict__ c2, T* out, long long rows,
                                                           int C, int cvb, int krows) {
    constexpr int V = VecN<T>::N, NP = RawVec<T>::NP;
    const int CV = C / V;
    const int cvl = threadIdx.x % cvb, rl = threadIdx.x / cvb;
    const int cv = blockIdx.y * cvb + cvl;
    if (cv >= CV) return;
    const int c0 = cv * V;
    float2 A[NP], Bz[NP], D[NP];
    {
        float2 mu[NP], rs[NP], k1[NP], k2[NP];
        ld_coef<NP>(a, c0, A);
        ld_coef<NP>(mean, c0, mu);
        ld_coef<NP>(rstd, c0, rs);
        ld_coef<NP>(c1, c0, k1);
        ld_coef<NP>(c2, c0, k2);
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            const float kx = rs[i].x * k2[i].x, ky = rs[i].y * k2[i].y;
            Bz[i] = make_float2(-A[i].x * kx, -A[i].y * ky);
            D[i] = make_float2(A[i].x * (kx * mu[i].x - k1[i].x), A[i].y * (ky * mu[i].y - k1[i].y));
        }
    }
    const RowRange rr = cta_rows(rows);
    const long long stride = krows;
    for (long long r0 = rr.begin + rl; r0 < rr.end; r0 += stride * UNROLL) {
        RawVec<T> gv[UNROLL], zv[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const long long r = r0 + u * stride;
            if (r < rr.end) {
                gv[u] = ld_raw(g + r * C + c0);
                zv[u] = ld_raw(z + r * C + c0);
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const long long r = r0 + u * stride;
            if (r < rr.end) {
#pragma unroll
                for (int i = 0; i < NP; ++i) gv[u].set(i, ffma2(gv[u].get(i), A[i], ffma2(zv[u].get(i), Bz[i], D[i])));
                st_raw(out + r * C + c0, gv[u]);
            }
        }
    }
}

struct ChanGrid { int cvb, krows; dim3 grid; };
static ChanGrid chan_grid(int CV, long long rows, int ctas_per_sm) {
    ChanGrid c;
    const int nchunks = ceil_div(CV, 128);
    c.cvb = ceil_div(CV, nchunks);
    c.krows = 256 / c.cvb;
    if (c.krows < 1) c.krows = 1;
    // one resident wave; at least 2*UNROLL rows per thread so the coefficient prologue is amortised
    long long gx = (rows + (long long)c.krows * 2 * UNROLL - 1) / ((long long)c.krows * 2 * UNROLL);
    const long long cap = ((long long)spnet_num_sms() * ctas_per_sm) / nchunks;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    c.grid = dim3((unsigned)gx, nchunks);
    return c;
}

// Reductions end with fp64 atomics per channel from every CTA, and that tail is serialised per address:
// one fat CTA per SM (up to 512 threads) keeps the chains 148 deep instead of 444 (the 12288 x 728
// reduce took 29 us next to 12 us for the dz kernel that moves more bytes).
static ChanGrid chan_grid_reduce(int CV, long long rows) {
    ChanGrid c;
    const int nchunks = ceil_div(CV, 128);
    c.cvb = ceil_div(CV, nchunks);
    c.krows = 512 / c.cvb;
    if (c.krows < 1) c.krows = 1;
    long long gx = (rows + (long long)c.krows * 2 * UNROLL - 1) / ((long long)c.krows * 2 * UNROLL);
    const long long cap = spnet_num_sms() / nchunks > 0 ? spnet_num_sms() / nchunks : 1;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    c.grid = dim3((unsigned)gx, nchunks);
    return c;
}

int check_rc(const char* who, int dtype, long long rows, int C) {
    SPNET_REQUIRE(rows > 0 && C > 0, "%s: bad shape", who);
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    SPNET_REQUIRE(C % V == 0, "%s: C=%d must be a multiple of %d", who, C, V);
    return SPNET_OK;
}

}  // namespace

extern "C" {

int spnet_bn_finalize(long long* stats, long long count, const float* gamma, const float* beta, float eps,
                      float momentum, int unbiased_moving_var, float* a, float* b, float* save_mean,
                      float* save_rstd, float* moving_mean, float* moving_var, int C, cudaStream_t stream) {
    SPNET_REQUIRE(stats && a && b && save_mean && save_rstd && C > 0 && count > 0, "bn_finalize: bad args");
    SPNET_REQUIRE((moving_mean == nullptr) == (moving_var == nullptr), "bn_finalize: moving stats come in pairs");
    bn_finalize_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(stats, (double)count, gamma, beta, eps, momentum,
                                                             unbiased_moving_var, a, b, save_mean, save_rstd, moving_mean,
                                                             moving_var, C);
    return spnet_check_launch("bn_finalize");
}

int spnet_bn_inference_affine(const float* gamma, const float* beta, const float* moving_mean,
                              const float* moving_var, float eps, float* a, float* b, float* save_mean,
                              float* save_rstd, int C, cudaStream_t stream) {
    SPNET_REQUIRE(moving_mean && moving_var && a && b && C > 0, "bn_inference_affine: bad args");
    SPNET_REQUIRE((save_mean == nullptr) == (save_rstd == nullptr), "bn_inference_affine: save_mean and save_rstd go together");
    bn_inference_affine_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(gamma, beta, moving_mean, moving_var, eps, a,
                                                                     b, save_mean, save_rstd, C);
    return spnet_check_launch("bn_inference_affine");
}

// out = act(a*z+b) [+ x]   (x nullable; out may alias z or x)
int spnet_bn_apply(const void* z, const float* a, const float* b, int act, const void* x, void* out, int dtype,
                   long long rows, int C, cudaStream_t stream) {
    int rc = check_rc("bn_apply", dtype, rows, C);
    if (rc) return rc;
    SPNET_REQUIRE(z && a && b && out && act >= 0 && act <= 3, "bn_apply: bad args");
    const ChanGrid cg = chan_grid(C / (dtype == SPNET_BF16 ? 8 : 4), rows, 3);
    SPNET_DISPATCH_DTYPE(dtype, (bn_apply_kernel<T><<<cg.grid, cg.cvb * cg.krows, 0, stream>>>(
                                    reinterpret_cast<const T*>(z), a, b, act, reinterpret_cast<const T*>(x),
                                    reinterpret_cast<T*>(out), rows, C, cg.cvb, cg.krows)));
    return spnet_check_launch("bn_apply");
}

int spnet_bn_bwd_reduce(void* g, const void* z, const float* save_mean, const float* save_rstd,
                        const float* relu_a, const float* relu_b, int act, long long* stats, int dtype,
                        long long rows, int C, cudaStream_t stream) {
    int rc = check_rc("bn_bwd_reduce", dtype, rows, C);
    if (rc) return rc;
    SPNET_REQUIRE(g && z && save_mean && save_rstd && stats, "bn_bwd_reduce: null pointer");
    SPNET_REQUIRE((relu_a == nullptr) == (relu_b == nullptr), "bn_bwd_reduce: mask affine comes in pairs");
    const ChanGrid cg = chan_grid_reduce(C / (dtype == SPNET_BF16 ? 8 : 4), rows);
    if (relu_a) {
        SPNET_DISPATCH_DTYPE(dtype, (bn_bwd_reduce_kernel<T, true><<<cg.grid, cg.cvb * cg.krows, 0, stream>>>(
                                        reinterpret_cast<T*>(g), reinterpret_cast<const T*>(z), save_mean, save_rstd,
                                        relu_a, relu_b, act, stats, rows, C, cg.cvb, cg.krows)));
    } else {
        SPNET_DISPATCH_DTYPE(dtype, (bn_bwd_reduce_kernel<T, false><<<cg.grid, cg.cvb * cg.krows, 0, stream>>>(
                                        reinterpret_cast<T*>(g), reinterpret_cast<const T*>(z), save_mean, save_rstd,
                                        relu_a, relu_b, act, stats, rows, C, cg.cvb, cg.krows)));
    }
    return spnet_check_launch("bn_bwd_reduce");
}

// stats[2*C] += (sum, sum of squares) per channel of z [rows, C]
int spnet_colstats(const void* z, long long* stats, int dtype, long long rows, int C, cudaStream_t stream) {
    int rc = check_rc("colstats", dtype, rows, C);
    if (rc) return rc;
    SPNET_REQUIRE(z && stats, "colstats: null pointer");
    const ChanGrid cg = chan_grid_reduce(C / (dtype == SPNET_BF16 ? 8 : 4), rows);
    SPNET_DISPATCH_DTYPE(dtype, (colstats_kernel<T><<<cg.grid, cg.cvb * cg.krows, 0, stream>>>(
                                    reinterpret_cast<const T*>(z), stats, rows, C, cg.cvb, cg.krows)));
    return spnet_check_launch("colstats");
}

int spnet_bn_bwd_finalize(long long* stats, long long count, float* dgamma, float* dbeta, float* c1, float* c2,
                          int C, cudaStream_t stream) {
    SPNET_REQUIRE(stats && c1 && c2 && C > 0 && count >= 0, "bn_bwd_finalize: bad args");
    bn_bwd_finalize_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(stats, (double)count, dgamma, dbeta, c1, c2, C);
    return spnet_check_launch("bn_bwd_finalize");
}

// out = a*(g - c1 - xhat*c2)   (out may alias g)
int spnet_bn_bwd_dz(const void* g, const void* z, const float* a, const float* save_mean, const float* save_rstd,
                    const float* c1, const float* c2, void* out, int dtype, long long rows, int C,
                    cudaStream_t stream) {
    int rc = check_rc("bn_bwd_dz", dtype, rows, C);
    if (rc) return rc;
    SPNET_REQUIRE(g && z && a && save_mean && save_rstd && c1 && c2 && out, "bn_bwd_dz: null pointer");
    const ChanGrid cg = chan_grid(C / (dtype == SPNET_BF16 ? 8 : 4), rows, 3);
    SPNET_DISPATCH_DTYPE(dtype, (bn_bwd_dz_kernel<T><<<cg.grid, cg.cvb * cg.krows, 0, stream>>>(
                                    reinterpret_cast<const T*>(g), reinterpret_cast<const T*>(z), a, save_mean, save_rstd,
                                    c1, c2, reinterpret_cast<T*>(out), rows, C, cg.cvb, cg.krows)));
    return spnet_check_launch("bn_bwd_dz");
}

}  // extern "C"
