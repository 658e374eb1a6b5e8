// MaxPooling2D(3, strides 2, 'same') fused with the BatchNorm-apply of both branches and
// the residual add of the Xception entry/exit blocks (keras.applications.Xception blocks
// 2-4 and 13; reference call site spnet/models.py:359), its backward, and the stride-2
// row/column subsample that feeds the 1x1 stride-2 residual convolutions.
//
// TF 'SAME' padding is asymmetric: out = ceil(in/2), pad_total = max((out-1)*2+3-in, 0),
// pad_before = pad_total/2 (even sizes pad only at the end). Padded cells never win the max.
#include "common.cuh"

namespace {

__host__ __device__ inline int same_pad_before(int in) {
    const int out = (in + 1) / 2;
    int total = (out - 1) * 2 + 3 - in;
    if (total < 0) total = 0;
    return total / 2;
}

// per-channel coefficients of one channel vector with 16-byte loads
template <int V> __device__ __forceinline__ void load_coef(const float* __restrict__ p, int c0, float (&v)[V]) {
#pragma unroll
    for (int i = 0; i < V; i += 4) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p + c0 + i));
        v[i] = q.x; v[i + 1] = q.y; v[i + 2] = q.z; v[i + 3] = q.w;
    }
}

// Both pooling kernels: blockIdx.x = one row of the tensor the kernel WRITES (image, output row), the threads
// walk that row's (column, channel vector) items; the image / row split is per CTA and one division per item
// is left (the one-thread-per-item versions spent three 32-bit divisions and eight single-byte argmax stores
// per item and ran at 30-40 % of the HBM roofline).
//
// out = max_{3x3,s2}(a*z+b) + (ra*res+rb);  argmax (optional) = kh*3+kw of the first maximum
template <typename T>
__global__ void __launch_bounds__(256) maxpool_add_fwd_kernel(const T* __restrict__ z, const float* __restrict__ a,
                                                              const float* __restrict__ b,
                                                              const T* __restrict__ res,
                                                              const float* __restrict__ ra,
                                                              const float* __restrict__ rb, T* __restrict__ out,
                                                              unsigned char* __restrict__ argmax, int B, int H,
                                                              int W, int C, int OH, int OW, int pt, int pl) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    const int row = blockIdx.x;  // bi * OH + oh
    const int bi = row / OH, oh = row - bi * OH;
    const int items = OW * CV;
    // the three input rows of this output row (clamped; flagged when they are padding)
    int ihc[3];
    bool okh[3];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
        const int ih = oh * 2 - pt + kh;
        ihc[kh] = min(max(ih, 0), H - 1);
        okh[kh] = ih == ihc[kh];
    }
    for (int it = blockIdx.y * blockDim.x + threadIdx.x; it < items; it += blockDim.x * gridDim.y) {
        const int ow = it / CV, cv = it - ow * CV;
        const int c0 = cv * V;
        const size_t idx = (size_t)row * items + it;
        float av[V], bv[V], best[V];
        int arg[V];
        if (a) {
            load_coef<V>(a, c0, av);
            load_coef<V>(b, c0, bv);
        }
#pragma unroll
        for (int i = 0; i < V; ++i) {
            if (!a) { av[i] = 1.f; bv[i] = 0.f; }
            best[i] = -INFINITY;
            arg[i] = 0;
        }
        // all nine loads are issued before the first compare (clamped addresses + validity flags): the
        // kernel is latency-bound, branches around the loads would serialise them
        float v[9][V];
        bool ok[9];
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
                const int iw = ow * 2 - pl + kw;
                const int iwc = min(max(iw, 0), W - 1);
                ok[kh * 3 + kw] = okh[kh] && iw == iwc;
                load_vec(z + (((size_t)bi * H + ihc[kh]) * W + iwc) * C + c0, v[kh * 3 + kw]);
            }
        }
        float rv[V];
        if (res) load_vec(res + idx * V, rv);
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            if (!ok[t]) continue;
#pragma unroll
            for (int i = 0; i < V; ++i) {
                const float y = fmaf(v[t][i], av[i], bv[i]);
                if (y > best[i]) { best[i] = y; arg[i] = t; }
            }
        }
        if (res) {
            if (ra) {
                float rav[V], rbv[V];
                load_coef<V>(ra, c0, rav);
                load_coef<V>(rb, c0, rbv);
#pragma unroll
                for (int i = 0; i < V; ++i) best[i] += fmaf(rv[i], rav[i], rbv[i]);
            } else {
#pragma unroll
                for (int i = 0; i < V; ++i) best[i] += rv[i];
            }
        }
        store_vec(out + idx * V, best);
        if (argmax) {  // V codes in one store
            uint32_t w[V / 4];
#pragma unroll
            for (int i = 0; i < V / 4; ++i)
                w[i] = (uint32_t)arg[4 * i] | ((uint32_t)arg[4 * i + 1] << 8) | ((uint32_t)arg[4 * i + 2] << 16) |
                       ((uint32_t)arg[4 * i + 3] << 24);
            if (V == 8) *reinterpret_cast<uint2*>(argmax + idx * V) = make_uint2(w[0], w[V / 4 - 1]);
            else *reinterpret_cast<uint32_t*>(argmax + idx * V) = w[0];
        }
    }
}

// bf16 forward: the same result bit for bit with a third of the instructions (the kernel above is issue-bound in
// bf16: 9 taps x 8 channels x (unpack, FMA, compare, two selects)). y = fma(v, a, b) is monotone in v for a fixed
// channel (rounding is monotone), so max_t y_t = fma(max_t v_t, a, b) for a > 0, fma(min_t v_t, a, b) for a < 0 and
// b for a = 0: the window maximum is taken on the raw bf16 pairs with packed max instructions on the KEY
// (v & zmask) ^ smask (sign flipped where a < 0, zero where a = 0), and the affine runs once per output.
// Padding: a padded tap is read from its clamped address, which is another tap of the same window (TF 'SAME'
// pads at most one row / column per side), so it can never change the maximum; it carries the CODE of the tap
// it duplicates, so that the first-maximum scan below lands on a real position. argmax = first tap, in kh*3+kw
// order, whose key equals the maximum (the fp32 kernel compares y instead of v: the two differ only where two
// different bf16 inputs round to the same fp32 y, and then both are maxima of y).
__global__ void __launch_bounds__(256) maxpool_add_fwd_bf16_kernel(const bf16* __restrict__ z, const float* __restrict__ a,
                                                                   const float* __restrict__ b,
                                                                   const bf16* __restrict__ res,
                                                                   const float* __restrict__ ra,
                                                                   const float* __restrict__ rb, bf16* __restrict__ out,
                                                                   unsigned char* __restrict__ argmax, int B, int H,
                                                                   int W, int C, int OH, int OW, int pt, int pl) {
    constexpr int V = 8;
    const int CV = C / V;
    const int row = blockIdx.x;  // bi * OH + oh
    const int bi = row / OH, oh = row - bi * OH;
    const int items = OW * CV;
    int ihc[3];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) ihc[kh] = min(max(oh * 2 - pt + kh, 0), H - 1);
    const int ih0 = oh * 2 - pt;
    for (int it = blockIdx.y * blockDim.x + threadIdx.x; it < items; it += blockDim.x * gridDim.y) {
        const int ow = it / CV, cv = it - ow * CV;
        const int c0 = cv * V;
        const size_t idx = (size_t)row * items + it;
        const int iw0 = ow * 2 - pl;
        uint4 raw[9];
        uint32_t code[9];  // kh*3+kw of the position actually read, in both halves of the word
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
                const int iwc = min(max(iw0 + kw, 0), W - 1);
                raw[kh * 3 + kw] = *reinterpret_cast<const uint4*>(z + (((size_t)bi * H + ihc[kh]) * W + iwc) * C + c0);
                code[kh * 3 + kw] = (uint32_t)((ihc[kh] - ih0) * 3 + (iwc - iw0)) * 0x00010001u;
            }
        }
        float av[V], bv[V];
        uint32_t zm[4], sm[4];
        if (a) {
            load_coef<V>(a, c0, av);
            load_coef<V>(b, c0, bv);
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                zm[p] = (av[2 * p] != 0.f ? 0x0000ffffu : 0u) | (av[2 * p + 1] != 0.f ? 0xffff0000u : 0u);
                sm[p] = (av[2 * p] < 0.f ? 0x00008000u : 0u) | (av[2 * p + 1] < 0.f ? 0x80000000u : 0u);
            }
        } else {
#pragma unroll
            for (int p = 0; p < 4; ++p) { zm[p] = 0xffffffffu; sm[p] = 0u; }
#pragma unroll
            for (int i = 0; i < V; ++i) { av[i] = 1.f; bv[i] = 0.f; }
        }
        uint32_t key[9][4], best[4], arg[4];
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const uint32_t w[4] = {raw[t].x, raw[t].y, raw[t].z, raw[t].w};
#pragma unroll
            for (int p = 0; p < 4; ++p) key[t][p] = (w[p] & zm[p]) ^ sm[p];
        }
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            __nv_bfloat162 m = *reinterpret_cast<const __nv_bfloat162*>(&key[0][p]);
#pragma unroll
            for (int t = 1; t < 9; ++t) m = __hmax2(m, *reinterpret_cast<const __nv_bfloat162*>(&key[t][p]));
            best[p] = *reinterpret_cast<const uint32_t*>(&m);
            arg[p] = 0u;
#pragma unroll
            for (int t = 8; t >= 0; --t) {  // last write wins = the first tap that holds the maximum
                const uint32_t eq = __heq2_mask(*reinterpret_cast<const __nv_bfloat162*>(&key[t][p]), m);
                arg[p] = (arg[p] & ~eq) | (code[t] & eq);
            }
        }
        float y[V];
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            const uint32_t v = best[p] ^ sm[p];
            y[2 * p] = fmaf(__uint_as_float(v << 16), av[2 * p], bv[2 * p]);
            y[2 * p + 1] = fmaf(__uint_as_float(v & 0xffff0000u), av[2 * p + 1], bv[2 * p + 1]);
        }
        if (res) {
            float rv[V];
            load_vec(res + idx * V, rv);
            if (ra) {
                float rav[V], rbv[V];
                load_coef<V>(ra, c0, rav);
                load_coef<V>(rb, c0, rbv);
#pragma unroll
                for (int i = 0; i < V; ++i) y[i] += fmaf(rv[i], rav[i], rbv[i]);
            } else {
#pragma unroll
                for (int i = 0; i < V; ++i) y[i] += rv[i];
            }
        }
        store_vec(out + idx * V, y);
        if (argmax) {
            const uint32_t w0 = (arg[0] & 0xffu) | ((arg[0] >> 8) & 0xff00u) | ((arg[1] & 0xffu) << 16) | ((arg[1] << 8) & 0xff000000u);
            const uint32_t w1 = (arg[2] & 0xffu) | ((arg[2] >> 8) & 0xff00u) | ((arg[3] & 0xffu) << 16) | ((arg[3] << 8) & 0xff000000u);
            *reinterpret_cast<uint2*>(argmax + idx * V) = make_uint2(w0, w1);
        }
    }
}

// gin[b,h,w,c] = sum over the (<= 2x2) windows containing (h,w) whose argmax is (h,w).
// One item = a 2 x 2 block of input positions (rows 2j-pt, 2j-pt+1; columns 2i-pl, 2i-pl+1) x one channel vector:
// the block lies inside window (j, i) - taps (0..1, 0..1) - and its first row / column are taps 2 of windows
// j-1 / i-1, so FOUR (gout, argmax) loads serve four outputs (one item per input position needed four loads
// each, 7 of every 16 of them for windows that cannot contain the position). The sums run in the order
// (j,i), (j,i-1), (j-1,i), (j-1,i-1). a[k] = gradient of block position k = 2*(row - r0) + (column - q0).
template <typename T, int V>
__device__ __forceinline__ void maxpool_bwd_item(const T* __restrict__ gout, const unsigned char* __restrict__ argmax,
                                                 int bi, int j, int i, int c0, int C, int OH, int OW, float (&a)[4][V]) {
    const bool okj0 = j < OH, okj1 = j >= 1 && j - 1 < OH;  // windows j and j-1 exist
    const bool oki0 = i < OW, oki1 = i >= 1 && i - 1 < OW;
    // windows in summation order: (j,i) (j,i-1) (j-1,i) (j-1,i-1)
    const bool okw[4] = {okj0 && oki0, okj0 && oki1, okj1 && oki0, okj1 && oki1};
    float g[4][V];
    uint32_t am[4][2];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int oh = (k < 2) ? (okj0 ? j : 0) : (okj1 ? j - 1 : 0);
        const int ow = (k & 1) ? (oki1 ? i - 1 : 0) : (oki0 ? i : 0);
        const size_t o = (((size_t)bi * OH + oh) * OW + ow) * C + c0;
        load_vec(gout + o, g[k]);
        if (V == 8) {
            const uint2 q = *reinterpret_cast<const uint2*>(argmax + o);
            am[k][0] = q.x; am[k][1] = q.y;
        } else {
            am[k][0] = *reinterpret_cast<const uint32_t*>(argmax + o); am[k][1] = 0;
        }
        if (!okw[k]) { am[k][0] = 0xffffffffu; am[k][1] = 0xffffffffu; }  // code 255: matches no tap
    }
#pragma unroll
    for (int e = 0; e < V; ++e) {
        const int sh = 8 * (e & 3), wd = e >> 2;
        const uint32_t k0 = (am[0][wd] >> sh) & 0xffu, k1 = (am[1][wd] >> sh) & 0xffu;
        const uint32_t k2 = (am[2][wd] >> sh) & 0xffu, k3 = (am[3][wd] >> sh) & 0xffu;
        float s = 0.f;
        if (k0 == 0u) s += g[0][e];
        if (k1 == 2u) s += g[1][e];
        if (k2 == 6u) s += g[2][e];
        if (k3 == 8u) s += g[3][e];
        a[0][e] = s;
        s = 0.f;
        if (k0 == 1u) s += g[0][e];
        if (k2 == 7u) s += g[2][e];
        a[1][e] = s;
        s = 0.f;
        if (k0 == 3u) s += g[0][e];
        if (k1 == 5u) s += g[1][e];
        a[2][e] = s;
        a[3][e] = (k0 == 4u) ? g[0][e] : 0.f;
    }
}

template <typename T>
__global__ void __launch_bounds__(256) maxpool_bwd_kernel(const T* __restrict__ gout,
                                                          const unsigned char* __restrict__ argmax,
                                                          T* __restrict__ gin, int B, int H, int W, int C, int OH,
                                                          int OW, int pt, int pl, int HP, int WP) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    const int row = blockIdx.x;  // bi * HP + j
    const int bi = row / HP, j = row - bi * HP;
    const int items = WP * CV;
    const int r0 = 2 * j - pt, r1 = r0 + 1;
    const bool okr0 = r0 >= 0, okr1 = r1 < H;             // r0 < H and r1 >= 0 by construction of HP
    for (int it = blockIdx.y * blockDim.x + threadIdx.x; it < items; it += blockDim.x * gridDim.y) {
        const int i = it / CV, cv = it - i * CV;
        const int c0 = cv * V;
        const int q0 = 2 * i - pl, q1 = q0 + 1;
        const bool okq0 = q0 >= 0, okq1 = q1 < W;
        float a[4][V];
        maxpool_bwd_item<T, V>(gout, argmax, bi, j, i, c0, C, OH, OW, a);
        T* base = gin + (((size_t)bi * H + r0) * W + q0) * C + c0;
        if (okr0 && okq0) store_vec(base, a[0]);
        if (okr0 && okq1) store_vec(base + C, a[1]);
        if (okr1 && okq0) store_vec(base + (size_t)W * C, a[2]);
        if (okr1 && okq1) store_vec(base + (size_t)W * C + C, a[3]);
    }
}

// The same gin, plus the BatchNorm-backward sums of the BN that produced the pooled tensor (z = its raw input):
//   stats[c] += sum gin,  stats[C+c] += sum gin * xhat,  xhat = z*rstd - mean*rstd  (as bn_bwd_reduce_kernel),
// over gin as stored. Channel-stationary: a thread keeps one channel vector and walks the items of its CTA's
// contiguous range, its partial sums in registers; one CTA per SM and ONE flush per CTA, so that the per-address
// fp64-atomic chains stay ~148 deep (a flush per tensor row would build chains thousands deep).
template <typename T>
__global__ void __launch_bounds__(512, 1) maxpool_bwd_stats_kernel(const T* __restrict__ gout,
                                                                   const unsigned char* __restrict__ argmax,
                                                                   T* __restrict__ gin, const T* __restrict__ z,
                                                                   const float* __restrict__ mean,
                                                                   const float* __restrict__ rstd,
                                                                   long long* __restrict__ stats, int B, int H, int W,
                                                                   int C, int OH, int OW, int pt, int pl, int HP, int WP,
                                                                   int cvb, int krows) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    const int cvl = threadIdx.x % cvb, rl = threadIdx.x / cvb;
    const int cv = blockIdx.y * cvb + cvl;
    const bool active = cv < CV;
    const int c0 = cv * V;
    float s1[V], s2[V];
#pragma unroll
    for (int e = 0; e < V; ++e) s1[e] = s2[e] = 0.f;
    if (active) {
        float rs[V], nm[V];
        load_coef<V>(rstd, c0, rs);
        load_coef<V>(mean, c0, nm);
#pragma unroll
        for (int e = 0; e < V; ++e) nm[e] = -nm[e] * rs[e];
        const int items = B * HP * WP;  // < 2^31: check_pool bounds B*H*W*C
        const int per_cta = (items + gridDim.x - 1) / gridDim.x;
        const int begin = blockIdx.x * per_cta, end = min(begin + per_cta, items);
        for (int p = begin + rl; p < end; p += krows) {
            const int bj = p / WP, i = p - bj * WP;
            const int bi = bj / HP, j = bj - bi * HP;
            const int r0 = 2 * j - pt, q0 = 2 * i - pl;
            const bool ok[4] = {r0 >= 0 && q0 >= 0, r0 >= 0 && q0 + 1 < W, r0 + 1 < H && q0 >= 0, r0 + 1 < H && q0 + 1 < W};
            // z of the four positions (clamped addresses, flagged by ok) is in flight with the gradient loads
            const int rc0 = max(r0, 0), rc1 = min(r0 + 1, H - 1), qc0 = max(q0, 0), qc1 = min(q0 + 1, W - 1);
            const T* zb = z + ((size_t)bi * H) * W * C + c0;
            float zv[4][V];
            load_vec(zb + ((size_t)rc0 * W + qc0) * C, zv[0]);
            load_vec(zb + ((size_t)rc0 * W + qc1) * C, zv[1]);
            load_vec(zb + ((size_t)rc1 * W + qc0) * C, zv[2]);
            load_vec(zb + ((size_t)rc1 * W + qc1) * C, zv[3]);
            float a[4][V];
            maxpool_bwd_item<T, V>(gout, argmax, bi, j, i, c0, C, OH, OW, a);
            T* base = gin + (((size_t)bi * H + r0) * W + q0) * C + c0;
            const size_t off[4] = {0, (size_t)C, (size_t)W * C, (size_t)W * C + C};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (!ok[k]) continue;
                store_vec(base + off[k], a[k]);
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    const float v = round_to<T>(a[k][e]);
                    s1[e] += v;
                    s2[e] = fmaf(v, fmaf(zv[k][e], rs[e], nm[e]), s2[e]);
                }
            }
        }
    }
    __shared__ float red[2][512 * 8];
#pragma unroll
    for (int e = 0; e < V; ++e) {
        red[0][threadIdx.x * V + e] = s1[e];
        red[1][threadIdx.x * V + e] = s2[e];
    }
    __syncthreads();
    if (rl == 0 && active) {
#pragma unroll
        for (int e = 0; e < V; ++e) {
            float t1 = 0.f, t2 = 0.f;
            for (int r = 0; r < krows; ++r) {
                t1 += red[0][(r * cvb + cvl) * V + e];
                t2 += red[1][(r * cvb + cvl) * V + e];
            }
            stat_add(stats, c0 + e, (double)t1);
            stat_add(stats, C + c0 + e, (double)t2);
        }
    }
}

// out[b,oh,ow,:] = in[b,2oh+off_h,2ow+off_w,:]   (off 0: what a 1x1 stride-2 'same' convolution reads, and a 3x3
// stride-2 'same' convolution on an ODD-sized dimension = its stride-1 result at even positions; off 1: the
// same on an EVEN-sized dimension = the stride-1 result at odd positions, because TF pads only at the end)
template <typename T>
__global__ void __launch_bounds__(256) gather_s2_kernel(const T* __restrict__ in, T* __restrict__ out, int B, int H,
                                                        int W, int C, int OH, int OW, int off_h, int off_w) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    const long long n = (long long)B * OH * OW * CV;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const unsigned uidx = (unsigned)idx;  // host guarantees < 2^31 items: 32-bit div/mod only
    const int cv = (int)(uidx % CV);
    unsigned r = uidx / CV;
    const int ow = (int)(r % OW);
    r /= OW;
    const int oh = (int)(r % OH);
    const int bi = (int)(r / OH);
    float v[V];
    load_vec(in + (((size_t)bi * H + 2 * oh + off_h) * W + 2 * ow + off_w) * C + cv * V, v);
    store_vec(out + idx * V, v);
}

// adjoint of gather_s2: out[b,h,w,:] = in[b,(h-off)/2,(w-off)/2,:] where both are integral, else 0
template <typename T>
__global__ void __launch_bounds__(256) scatter_s2_kernel(const T* __restrict__ in, T* __restrict__ out, int B, int H,
                                                         int W, int C, int OH, int OW, int off_h, int off_w) {
    constexpr int V = VecN<T>::N;
    const int CV = C / V;
    const long long n = (long long)B * H * W * CV;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const unsigned uidx = (unsigned)idx;
    const int cv = (int)(uidx % CV);
    unsigned r = uidx / CV;
    const int w = (int)(r % W);
    r /= W;
    const int h = (int)(r % H);
    const int bi = (int)(r / H);
    float v[V];
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] = 0.f;
    const int th = h - off_h, tw = w - off_w;
    if (th >= 0 && tw >= 0 && !(th & 1) && !(tw & 1) && (th >> 1) < OH && (tw >> 1) < OW)
        load_vec(in + (((size_t)bi * OH + (th >> 1)) * OW + (tw >> 1)) * C + cv * V, v);
    store_vec(out + idx * V, v);
}

// grid of the row-per-CTA pooling kernels: x = rows, y = chunks of a row so that a thread handles ~2 items
dim3 row_grid(int rows, int items) {
    int gy = (items + 511) / 512;
    if (gy < 1) gy = 1;
    if (gy > 16) gy = 16;
    return dim3((unsigned)rows, (unsigned)gy);
}

int check_pool(const char* who, int dtype, int B, int H, int W, int C) {
    SPNET_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0, "%s: bad shape", who);
    SPNET_REQUIRE((long long)B * H * W * C < 0x7fffffffLL, "%s: tensor too large for 32-bit indexing", who);
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    SPNET_REQUIRE(C % V == 0, "%s: C=%d must be a multiple of %d", who, C, V);
    return SPNET_OK;
}

}  // namespace

extern "C" {

int spnet_maxpool3s2_add_fwd(const void* z, const float* a, const float* b, const void* res, const float* ra,
                             const float* rb, void* out, unsigned char* argmax, int dtype, int B, int H, int W,
                             int C, cudaStream_t stream) {
    int rc = check_pool("maxpool3s2_add_fwd", dtype, B, H, W, C);
    if (rc) return rc;
    SPNET_REQUIRE(z && out, "maxpool3s2_add_fwd: null pointer");
    SPNET_REQUIRE((a == nullptr) == (b == nullptr) && (ra == nullptr) == (rb == nullptr),
                  "maxpool3s2_add_fwd: affine parameters come in pairs");
    const int OH = (H + 1) / 2, OW = (W + 1) / 2;
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    if (dtype == SPNET_BF16)
        maxpool_add_fwd_bf16_kernel<<<row_grid(B * OH, OW * (C / V)), 256, 0, stream>>>(
            reinterpret_cast<const bf16*>(z), a, b, reinterpret_cast<const bf16*>(res), ra, rb, reinterpret_cast<bf16*>(out),
            argmax, B, H, W, C, OH, OW, same_pad_before(H), same_pad_before(W));
    else
        maxpool_add_fwd_kernel<float><<<row_grid(B * OH, OW * (C / V)), 256, 0, stream>>>(
            reinterpret_cast<const float*>(z), a, b, reinterpret_cast<const float*>(res), ra, rb,
            reinterpret_cast<float*>(out), argmax, B, H, W, C, OH, OW, same_pad_before(H), same_pad_before(W));
    return spnet_check_launch("maxpool3s2_add_fwd");
}

// z, mean, rstd, stats (all or none): also stats[2*C] += (sum gin, sum gin*xhat), xhat = (z-mean)*rstd, over gin as
// stored, the BatchNorm-backward sums of the BN whose output was pooled (z = its raw input, [B,H,W,C] like gin)
int spnet_maxpool3s2_bwd(const void* gout, const unsigned char* argmax, void* gin, int dtype, int B, int H, int W,
                         int C, const void* z, const float* mean, const float* rstd, long long* stats,
                         cudaStream_t stream) {
    int rc = check_pool("maxpool3s2_bwd", dtype, B, H, W, C);
    if (rc) return rc;
    SPNET_REQUIRE(gout && argmax && gin, "maxpool3s2_bwd: null pointer");
    SPNET_REQUIRE((z == nullptr) == (stats == nullptr) && (z == nullptr) == (mean == nullptr) &&
                      (z == nullptr) == (rstd == nullptr), "maxpool3s2_bwd: z, mean, rstd and stats come together");
    const int OH = (H + 1) / 2, OW = (W + 1) / 2;
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    const int pt = same_pad_before(H), pl = same_pad_before(W);
    const int HP = (H - 1 + pt) / 2 + 1, WP = (W - 1 + pl) / 2 + 1;  // 2 x 2 blocks of input positions
    if (z) {
        // up to 128 channel vectors per CTA, the rest of 512 threads on items; one CTA per SM
        const int CV = C / V, nchunks = ceil_div(CV, 128);
        const int cvb = ceil_div(CV, nchunks), krows = 512 / cvb > 0 ? 512 / cvb : 1;
        long long gx = ceil_div((long long)B * HP * WP, krows);
        const long long cap = spnet_num_sms() / nchunks > 0 ? spnet_num_sms() / nchunks : 1;
        if (gx > cap) gx = cap;
        SPNET_DISPATCH_DTYPE(dtype, (maxpool_bwd_stats_kernel<T><<<dim3((unsigned)gx, nchunks), cvb * krows, 0, stream>>>(
                                        reinterpret_cast<const T*>(gout), argmax, reinterpret_cast<T*>(gin),
                                        reinterpret_cast<const T*>(z), mean, rstd, stats, B, H, W, C, OH, OW, pt, pl, HP,
                                        WP, cvb, krows)));
        return spnet_check_launch("maxpool3s2_bwd_stats");
    }
    SPNET_DISPATCH_DTYPE(dtype, (maxpool_bwd_kernel<T><<<row_grid(B * HP, WP * (C / V)), 256, 0, stream>>>(
                                    reinterpret_cast<const T*>(gout), argmax, reinterpret_cast<T*>(gin), B, H, W, C,
                                    OH, OW, pt, pl, HP, WP)));
    return spnet_check_launch("maxpool3s2_bwd");
}

// MaxPooling2D(3, strides 2, 'valid') (Inception-ResNet stem / reductions): the same kernels with no
// padding and OH = (H-3)/2+1. out [B,OH,OW,C]; argmax nullable (inference).
int spnet_maxpool3s2_valid_fwd(const void* z, void* out, unsigned char* argmax, int dtype, int B, int H, int W, int C,
                               cudaStream_t stream) {
    int rc = check_pool("maxpool3s2_valid_fwd", dtype, B, H, W, C);
    if (rc) return rc;
    SPNET_REQUIRE(z && out && H >= 3 && W >= 3, "maxpool3s2_valid_fwd: bad args");
    const int OH = (H - 3) / 2 + 1, OW = (W - 3) / 2 + 1;
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    if (dtype == SPNET_BF16)
        maxpool_add_fwd_bf16_kernel<<<row_grid(B * OH, OW * (C / V)), 256, 0, stream>>>(
            reinterpret_cast<const bf16*>(z), nullptr, nullptr, nullptr, nullptr, nullptr, reinterpret_cast<bf16*>(out), argmax,
            B, H, W, C, OH, OW, 0, 0);
    else
        maxpool_add_fwd_kernel<float><<<row_grid(B * OH, OW * (C / V)), 256, 0, stream>>>(
            reinterpret_cast<const float*>(z), nullptr, nullptr, nullptr, nullptr, nullptr, reinterpret_cast<float*>(out),
            argmax, B, H, W, C, OH, OW, 0, 0);
    return spnet_check_launch("maxpool3s2_valid_fwd");
}

int spnet_maxpool3s2_valid_bwd(const void* gout, const unsigned char* argmax, void* gin, int dtype, int B, int H, int W,
                               int C, cudaStream_t stream) {
    int rc = check_pool("maxpool3s2_valid_bwd", dtype, B, H, W, C);
    if (rc) return rc;
    SPNET_REQUIRE(gout && argmax && gin && H >= 3 && W >= 3, "maxpool3s2_valid_bwd: bad args");
    const int OH = (H - 3) / 2 + 1, OW = (W - 3) / 2 + 1;
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    const int HP = (H - 1) / 2 + 1, WP = (W - 1) / 2 + 1;
    SPNET_DISPATCH_DTYPE(dtype, (maxpool_bwd_kernel<T><<<row_grid(B * HP, WP * (C / V)), 256, 0, stream>>>(
                                    reinterpret_cast<const T*>(gout), argmax, reinterpret_cast<T*>(gin), B, H, W, C, OH, OW,
                                    0, 0, HP, WP)));
    return spnet_check_launch("maxpool3s2_valid_bwd");
}

// per dimension: off = 0 takes positions 0,2,4,... (ceil(n/2) of them), off = 1 takes 1,3,5,... (n/2 of them)
int spnet_gather_s2(const void* in, void* out, int dtype, int B, int H, int W, int C, int off_h, int off_w,
                    cudaStream_t stream) {
    int rc = check_pool("gather_s2", dtype, B, H, W, C);
    if (rc) return rc;
    SPNET_REQUIRE(in && out && (off_h == 0 || off_h == 1) && (off_w == 0 || off_w == 1), "gather_s2: bad args");
    const int OH = (H + 1 - off_h) / 2, OW = (W + 1 - off_w) / 2;
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    const long long n = (long long)B * OH * OW * (C / V);
    SPNET_DISPATCH_DTYPE(dtype, (gather_s2_kernel<T><<<ceil_div(n, 256), 256, 0, stream>>>(
                                    reinterpret_cast<const T*>(in), reinterpret_cast<T*>(out), B, H, W, C, OH, OW, off_h, off_w)));
    return spnet_check_launch("gather_s2");
}

// adjoint of spnet_gather_s2: in [B,OH,OW,C] (OH, OW as above) -> out [B,H,W,C], zero elsewhere
int spnet_scatter_s2(const void* in, void* out, int dtype, int B, int H, int W, int C, int off_h, int off_w,
                     cudaStream_t stream) {
    int rc = check_pool("scatter_s2", dtype, B, H, W, C);
    if (rc) return rc;
    SPNET_REQUIRE(in && out && (off_h == 0 || off_h == 1) && (off_w == 0 || off_w == 1), "scatter_s2: bad args");
    const int OH = (H + 1 - off_h) / 2, OW = (W + 1 - off_w) / 2;
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    const long long n = (long long)B * H * W * (C / V);
    SPNET_DISPATCH_DTYPE(dtype, (scatter_s2_kernel<T><<<ceil_div(n, 256), 256, 0, stream>>>(
                                    reinterpret_cast<const T*>(in), reinterpret_cast<T*>(out), B, H, W, C, OH, OW, off_h, off_w)));
    return spnet_check_launch("scatter_s2");
}

}  // extern "C"
