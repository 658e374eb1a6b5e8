// Small-channel direct convolutions of the SPNet stem and of Xception's block1_conv1
// (spnet/models.py:319-340; keras.applications.Xception block1_conv1): Cin <= 3, so there is no
// tensor-core shape for them and they are HBM/latency-bound (<1 % of the model's FLOPs).
//
//   which 0 : stem conv1 folded with AveragePooling2D(2): 4x4 stride-2 (pad 1), 1 -> 3, fp32 input
//   which 1 : stem conv2 / conv3: 3x3 'same', 3 -> 3, BN + LeakyReLU(0.1) applied on load
//   which 2 : block1_conv1: 3x3 stride 2 'valid', 3 -> 32
//
// All kernels share one structure: a persistent CTA walks output tiles; the input window of a tile
// is loaded cooperatively (contiguous, coalesced element loads), transformed ONCE (BN affine +
// activation, zero padding applied after it) and parked in shared memory as fp32, so the
// per-pixel work is conflict-free LDS + FMA with no address arithmetic; 3-channel outputs go back
// through shared memory so that global stores are contiguous too. BatchNorm statistics and weight
// gradients are accumulated in registers across all tiles of a CTA and reduced once at the end.
#include "common.cuh"

namespace {

__device__ __forceinline__ float apply_act(float y, int act) {
    if (act == 1) return fmaxf(y, 0.f);
    if (act == 2) return y > 0.f ? y : 0.1f * y;
    return y;
}

constexpr int kThreads = 256;

// Input window of an output tile -> fp32 shared memory sm[r][c*CIN + ci] (row pitch ROWP, the same
// interleaved order as global memory), transformed by act(a*v+b); out-of-image elements are zero
// (padding follows the activation). Two phases so that the global loads of the NEXT tile are in
// flight while the current tile is computed: fetch() = coalesced element loads into registers,
// commit() = transform + park in smem. Warp w owns rows w, w+8, ..., a lane owns every 32nd element
// of a row, so no per-element division is needed and all predicates are compares.
template <typename TI, int CIN, int IH_T, int IW_T>
struct Window {
    static constexpr int ROW_E = IW_T * CIN, ROWP = ROW_E + 1;
    static constexpr int RPW = (IH_T + 7) / 8, EPL = (ROW_E + 31) / 32;
    TI raw[RPW * EPL];
    __device__ __forceinline__ void fetch(const TI* __restrict__ img, int H, int W, int ih0, int iw0) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        const int e_lo = max(0, -iw0) * CIN, e_hi = min(IW_T, W - iw0) * CIN;
#pragma unroll
        for (int i = 0; i < RPW; ++i) {
            const int r = warp + 8 * i, ih = ih0 + r;
            const bool rowok = r < IH_T && ih >= 0 && ih < H;
            const TI* rowp = img + ((long long)ih * W + iw0) * CIN;
#pragma unroll
            for (int j = 0; j < EPL; ++j) {
                const int e = lane + 32 * j;
                if (rowok && e >= e_lo && e < e_hi) raw[i * EPL + j] = rowp[e];
            }
        }
    }
    __device__ __forceinline__ void commit(float* __restrict__ sm, const float* sab, bool affine, int act, int H, int W,
                                           int ih0, int iw0) const {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        const int e_lo = max(0, -iw0) * CIN, e_hi = min(IW_T, W - iw0) * CIN;
        const int l3 = lane % CIN;
#pragma unroll
        for (int i = 0; i < RPW; ++i) {
            const int r = warp + 8 * i, ih = ih0 + r;
            if (r >= IH_T) break;
            const bool rowok = ih >= 0 && ih < H;
#pragma unroll
            for (int j = 0; j < EPL; ++j) {
                const int e = lane + 32 * j;
                if (e >= ROW_E) break;
                int ci = l3 + (32 * j) % CIN;
                if (ci >= CIN) ci -= CIN;
                float v = 0.f;
                if (rowok && e >= e_lo && e < e_hi) {
                    v = to_f32(raw[i * EPL + j]);
                    if (affine) v = apply_act(fmaf(v, sab[ci], sab[CIN + ci]), act);
                }
                sm[r * ROWP + e] = v;
            }
        }
    }
};

// rows of a tile -> global memory: warp w copies rows w, w+8, ... (row_e contiguous elements each)
template <typename T>
__device__ __forceinline__ void copy_rows_out(T* __restrict__ dst, long long dst_pitch, const T* __restrict__ src, int src_pitch,
                                              int rows, int row_e) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = warp; r < rows; r += 8)
        for (int e = lane; e < row_e; e += 32) dst[r * dst_pitch + e] = src[r * src_pitch + e];
}

struct TileXY { int b, r0, c0; };
__device__ __forceinline__ TileXY tile_xy(int tile, int tiles_h, int tiles_w, int TH, int TW) {
    TileXY t;
    const int tw = tile % tiles_w, q = tile / tiles_w;
    t.c0 = tw * TW;
    t.r0 = (q % tiles_h) * TH;
    t.b = q / tiles_h;
    return t;
}

// =================================================================================================
// Forward-type pass, 3 output channels (which 0, which 1, and the data gradient of which 1, which
// is the same convolution with the flipped + transposed kernel followed by the activation mask).
// Tile = 16 x 64 output pixels, thread = 4 pixels (rows ty, ty+4, ty+8, ty+12).
//   MODE 0: plain   MODE 1: + skip = mean of the 2x2 centre taps (which 0)   MODE 2: data gradient
// =================================================================================================
constexpr int C3_TH = 16, C3_TW = 64;
constexpr int C3W_TH = 8;  // weight-gradient tiles: 81 partial sums + the prefetch stage must fit 128 registers

template <typename TI, typename TO, int CIN, int KS, int S, int MODE>
__global__ void __launch_bounds__(kThreads, 2) conv3out_kernel(const TI* __restrict__ in, const float* __restrict__ w,
                                                               const float* __restrict__ in_a,
                                                               const float* __restrict__ in_b, int act,
                                                               TO* __restrict__ out, TO* __restrict__ skip,
                                                               long long* __restrict__ stats,
                                                               const TO* __restrict__ mask_z,
                                                               const float* __restrict__ mask_a,
                                                               const float* __restrict__ mask_b, int B, int H, int W,
                                                               int OH, int OW, int pt, int pl, int tiles_h, int tiles_w) {
    constexpr int COUT = 3, TH = C3_TH, TW = C3_TW;
    constexpr int IH_T = (TH - 1) * S + KS, IW_T = (TW - 1) * S + KS;
    typedef Window<TI, CIN, IH_T, IW_T> Win;
    constexpr int ROWP = Win::ROWP;
    constexpr int NW = KS * KS * CIN * COUT;
    __shared__ float s_in[IH_T * ROWP];
    __shared__ __align__(16) float ws[KS * KS * CIN * 4];  // [tap][ci][co padded to 4]
    __shared__ float sab[2 * CIN + 2 * COUT];
    __shared__ TO s_out[TH * TW * COUT];
    __shared__ TO s_skip[MODE == 1 ? TH * TW : 1];
    __shared__ float sred[(kThreads / 32) * 2 * COUT];  // per-warp partials, summed in warp order (run-to-run identical)
    for (int i = threadIdx.x; i < NW; i += kThreads) {
        const int t = i / (CIN * COUT), rem = i % (CIN * COUT);
        const int cin_here = rem / COUT, cout_here = rem % COUT;
        // data gradient: out channel = forward ci, in channel = forward co, taps flipped
        ws[(t * CIN + cin_here) * 4 + cout_here] =
            MODE == 2 ? w[((KS * KS - 1 - t) * COUT + cout_here) * CIN + cin_here] : w[i];
    }
    if (threadIdx.x < CIN) {
        sab[threadIdx.x] = in_a ? in_a[threadIdx.x] : 1.f;
        sab[CIN + threadIdx.x] = in_a ? in_b[threadIdx.x] : 0.f;
    }
    if (MODE == 2 && threadIdx.x < COUT) {
        sab[2 * CIN + threadIdx.x] = mask_z ? mask_a[threadIdx.x] : 1.f;
        sab[2 * CIN + COUT + threadIdx.x] = mask_z ? mask_b[threadIdx.x] : 0.f;
    }
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    float ssum[COUT] = {0.f, 0.f, 0.f}, ssq[COUT] = {0.f, 0.f, 0.f};
    const int n_tiles = B * tiles_h * tiles_w;
    Win win;
    if ((int)blockIdx.x < n_tiles) {
        const TileXY t = tile_xy(blockIdx.x, tiles_h, tiles_w, TH, TW);
        win.fetch(in + (size_t)t.b * H * W * CIN, H, W, t.r0 * S - pt, t.c0 * S - pl);
    }
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TileXY tc = tile_xy(tile, tiles_h, tiles_w, TH, TW);
        const int oh0 = tc.r0, ow0 = tc.c0, b = tc.b;
        __syncthreads();  // previous tile: compute is done with s_in, copy-out is done with s_out
        win.commit(s_in, sab, in_a != nullptr, act, H, W, oh0 * S - pt, ow0 * S - pl);
        __syncthreads();
        if (tile + (int)gridDim.x < n_tiles) {  // next tile's loads fly during this tile's compute
            const TileXY t = tile_xy(tile + gridDim.x, tiles_h, tiles_w, TH, TW);
            win.fetch(in + (size_t)t.b * H * W * CIN, H, W, t.r0 * S - pt, t.c0 * S - pl);
        }
        // 4 pixels per thread (rows ty + 4*pp) share every weight triple: one LDS.128 per (tap, ci)
        constexpr int PP = TH / 4;
        float acc[PP][COUT], centre[PP];
#pragma unroll
        for (int pp = 0; pp < PP; ++pp) {
            centre[pp] = 0.f;
#pragma unroll
            for (int co = 0; co < COUT; ++co) acc[pp][co] = 0.f;
        }
#pragma unroll 1
        for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
            for (int kh = 0; kh < KS; ++kh)
#pragma unroll
                for (int kw = 0; kw < KS; ++kw) {
                    const float4 wv = *reinterpret_cast<const float4*>(&ws[((kh * KS + kw) * CIN + ci) * 4]);
#pragma unroll
                    for (int pp = 0; pp < PP; ++pp) {
                        const float v = s_in[((ty + 4 * pp) * S + kh) * ROWP + (tx * S + kw) * CIN + ci];
                        if (MODE == 1 && (kh == 1 || kh == 2) && (kw == 1 || kw == 2)) centre[pp] += v;
                        acc[pp][0] = fmaf(v, wv.x, acc[pp][0]);
                        acc[pp][1] = fmaf(v, wv.y, acc[pp][1]);
                        acc[pp][2] = fmaf(v, wv.z, acc[pp][2]);
                    }
                }
#pragma unroll
        for (int pp = 0; pp < PP; ++pp) {
            const int r = ty + 4 * pp;
            const int oh = oh0 + r, ow = ow0 + tx;
            const bool valid = oh < OH && ow < OW;
            if (MODE == 2 && mask_z && valid) {
                const TO* mz = mask_z + (((size_t)b * OH + oh) * OW + ow) * COUT;
#pragma unroll
                for (int co = 0; co < COUT; ++co) {
                    const float pre = fmaf(to_f32(mz[co]), sab[2 * CIN + co], sab[2 * CIN + COUT + co]);
                    if (!(pre > 0.f)) acc[pp][co] = (act == 2) ? 0.1f * acc[pp][co] : (act == 1 ? 0.f : acc[pp][co]);
                }
            }
#pragma unroll
            for (int co = 0; co < COUT; ++co) {
                const TO o = from_f32<TO>(acc[pp][co]);
                s_out[(r * TW + tx) * COUT + co] = o;
                if (valid) {
                    const float rr = to_f32(o);
                    ssum[co] += rr;
                    ssq[co] = fmaf(rr, rr, ssq[co]);
                }
            }
            if (MODE == 1) s_skip[r * TW + tx] = from_f32<TO>(0.25f * centre[pp]);
        }
        __syncthreads();
        // contiguous row segments of the output tile
        const int vw = min(TW, OW - ow0), vh = min(TH, OH - oh0);
        copy_rows_out(out + (((size_t)b * OH + oh0) * OW + ow0) * COUT, (long long)OW * COUT, s_out, TW * COUT, vh, vw * COUT);
        if (MODE == 1) copy_rows_out(skip + ((size_t)b * OH + oh0) * OW + ow0, (long long)OW, s_skip, TW, vh, vw);
    }
    if (stats) {
        __syncthreads();
#pragma unroll
        for (int co = 0; co < COUT; ++co) {
            const float s = warp_sum(ssum[co]), q = warp_sum(ssq[co]);
            if ((threadIdx.x & 31) == 0) {
                sred[(threadIdx.x >> 5) * 2 * COUT + co] = s;
                sred[(threadIdx.x >> 5) * 2 * COUT + COUT + co] = q;
            }
        }
        __syncthreads();
        if (threadIdx.x < 2 * COUT) {
            float t = 0.f;
            for (int w_ = 0; w_ < kThreads / 32; ++w_) t += sred[w_ * 2 * COUT + threadIdx.x];
            stat_add(stats, threadIdx.x, (double)t);
        }
    }
}

// =================================================================================================
// block1_conv1 forward: 3x3 stride 2 valid, 3 -> 32. Tile = 4 x 64 output pixels, thread = pixel,
// 32 accumulators per thread, weights read from shared memory as float4.
// =================================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads, 2) conv_b1c1_fwd_kernel(const T* __restrict__ in, const float* __restrict__ w,
                                                                    const float* __restrict__ in_a,
                                                                    const float* __restrict__ in_b, int act,
                                                                    T* __restrict__ out, long long* __restrict__ stats,
                                                                    int B, int H, int W, int OH, int OW, int pt, int pl,
                                                                    int tiles_h, int tiles_w) {
    constexpr int CIN = 3, COUT = 32, KS = 3, S = 2, TH = 4, TW = 64;
    constexpr int IH_T = (TH - 1) * S + KS, IW_T = (TW - 1) * S + KS;
    typedef Window<T, CIN, IH_T, IW_T> Win;
    constexpr int ROWP = Win::ROWP;
    __shared__ float s_in[IH_T * ROWP];
    __shared__ __align__(16) float ws[KS * KS * CIN * COUT];
    __shared__ float sab[2 * CIN];
    __shared__ float sred[(kThreads / 32) * 2 * COUT];  // per-warp partials, summed in warp order
    for (int i = threadIdx.x; i < KS * KS * CIN * COUT; i += kThreads) ws[i] = w[i];
    if (threadIdx.x < CIN) {
        sab[threadIdx.x] = in_a ? in_a[threadIdx.x] : 1.f;
        sab[CIN + threadIdx.x] = in_a ? in_b[threadIdx.x] : 0.f;
    }
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6, lane = threadIdx.x & 31;
    float cs = 0.f, cq = 0.f;  // running per-channel sums: channel = lane
    const int n_tiles = B * tiles_h * tiles_w;
    Win win;
    if ((int)blockIdx.x < n_tiles) {
        const TileXY t = tile_xy(blockIdx.x, tiles_h, tiles_w, TH, TW);
        win.fetch(in + (size_t)t.b * H * W * CIN, H, W, t.r0 * S - pt, t.c0 * S - pl);
    }
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TileXY tc = tile_xy(tile, tiles_h, tiles_w, TH, TW);
        const int oh0 = tc.r0, ow0 = tc.c0, b = tc.b;
        __syncthreads();  // previous tile's readers are done with s_in
        win.commit(s_in, sab, in_a != nullptr, act, H, W, oh0 * S - pt, ow0 * S - pl);
        __syncthreads();
        if (tile + (int)gridDim.x < n_tiles) {
            const TileXY t = tile_xy(tile + gridDim.x, tiles_h, tiles_w, TH, TW);
            win.fetch(in + (size_t)t.b * H * W * CIN, H, W, t.r0 * S - pt, t.c0 * S - pl);
        }
        const int oh = oh0 + ty, ow = ow0 + tx;
        const bool valid = oh < OH && ow < OW;
        float acc[COUT];
#pragma unroll
        for (int co = 0; co < COUT; ++co) acc[co] = 0.f;
#pragma unroll
        for (int kh = 0; kh < KS; ++kh)
#pragma unroll
            for (int kw = 0; kw < KS; ++kw)
#pragma unroll
                for (int ci = 0; ci < CIN; ++ci) {
                    const float v = s_in[(ty * S + kh) * ROWP + (tx * S + kw) * CIN + ci];
                    const float4* wr = reinterpret_cast<const float4*>(&ws[((kh * KS + kw) * CIN + ci) * COUT]);
#pragma unroll
                    for (int c4 = 0; c4 < COUT / 4; ++c4) {
                        const float4 ww = wr[c4];
                        acc[4 * c4 + 0] = fmaf(v, ww.x, acc[4 * c4 + 0]);
                        acc[4 * c4 + 1] = fmaf(v, ww.y, acc[4 * c4 + 1]);
                        acc[4 * c4 + 2] = fmaf(v, ww.z, acc[4 * c4 + 2]);
                        acc[4 * c4 + 3] = fmaf(v, ww.w, acc[4 * c4 + 3]);
                    }
                }
        if (valid) {
            T* o = out + (((size_t)b * OH + oh) * OW + ow) * COUT;
            if constexpr (sizeof(T) == 2) {
#pragma unroll
                for (int g = 0; g < 4; ++g)
                    *reinterpret_cast<uint4*>(o + 8 * g) =
                        make_uint4(pack_bf16x2(acc[8 * g], acc[8 * g + 1]), pack_bf16x2(acc[8 * g + 2], acc[8 * g + 3]),
                                   pack_bf16x2(acc[8 * g + 4], acc[8 * g + 5]), pack_bf16x2(acc[8 * g + 6], acc[8 * g + 7]));
            } else {
#pragma unroll
                for (int g = 0; g < 8; ++g)
                    *reinterpret_cast<float4*>(o + 4 * g) = make_float4(acc[4 * g], acc[4 * g + 1], acc[4 * g + 2], acc[4 * g + 3]);
            }
        }
        if (stats) {
            // lane = pixel, 32 channels per lane: the butterfly leaves channel `lane`'s sum over the warp's pixels
            float sq[32];
#pragma unroll
            for (int co = 0; co < 32; ++co) {
                acc[co] = valid ? round_to<T>(acc[co]) : 0.f;
                sq[co] = acc[co] * acc[co];
            }
            cs += warp_colsum32(acc, lane);
            cq += warp_colsum32(sq, lane);
        }
    }
    if (stats) {
        __syncthreads();
        sred[(threadIdx.x >> 5) * 2 * COUT + lane] = cs;
        sred[(threadIdx.x >> 5) * 2 * COUT + COUT + lane] = cq;
        __syncthreads();
        if (threadIdx.x < 2 * COUT) {
            float t = 0.f;
            for (int w_ = 0; w_ < kThreads / 32; ++w_) t += sred[w_ * 2 * COUT + threadIdx.x];
            stat_add(stats, threadIdx.x, (double)t);
        }
    }
}

// 4 consecutive channels of a gradient pixel, widened to fp32, with a register prefetch stage
template <typename T> struct G4;
template <> struct G4<bf16> {
    uint2 r;
    __device__ __forceinline__ void load(const bf16* p) { r = *reinterpret_cast<const uint2*>(p); }
    __device__ __forceinline__ void zero() { r = make_uint2(0u, 0u); }
    __device__ __forceinline__ float4 get() const {
        return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16),
                           __uint_as_float(r.y & 0xffff0000u));
    }
};
template <> struct G4<float> {
    float4 r;
    __device__ __forceinline__ void load(const float* p) { r = *reinterpret_cast<const float4*>(p); }
    __device__ __forceinline__ void zero() { r = make_float4(0.f, 0.f, 0.f, 0.f); }
    __device__ __forceinline__ float4 get() const { return r; }
};

// =================================================================================================
// block1_conv1 / MobileNet conv1 data gradient: gin[ih,iw,ci] = sum_{kh,kw,co} g[(ih+pt-kh)/2, (iw+pl-kw)/2, co] w[kh,kw,ci,co]
// over the taps whose (ih+pt-kh, iw+pl-kw) are even and inside the output (pt, pl = leading padding, 0 or 1). Tile = 8 x 64 INPUT pixels;
// warp = one row, lane = column pair (2*lane, 2*lane+1) processed one parity at a time, so that
// the set of contributing taps is warp-uniform.
// =================================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads, 2) conv_b1c1_dgrad_kernel(const T* __restrict__ g, const float* __restrict__ w,
                                                                      T* __restrict__ gin, int B, int H, int W, int OH,
                                                                      int OW, int pt, int pl, int tiles_h, int tiles_w) {
    constexpr int CIN = 3, COUT = 32, KS = 3, TH = 8, TW = 64;
    constexpr int GH_T = TH / 2 + 2, GW_T = TW / 2 + 2, GP = COUT + 4;  // padded pixel pitch: conflict-free LDS.128
    constexpr int NV = GH_T * GW_T * (COUT / 4), PER = (NV + kThreads - 1) / kThreads;
    __shared__ __align__(16) float s_g[GH_T * GW_T * GP];
    __shared__ __align__(16) float ws[KS * KS * CIN * COUT];
    __shared__ T s_out[TH * TW * CIN];
    for (int i = threadIdx.x; i < KS * KS * CIN * COUT; i += kThreads) ws[i] = w[i];
    const int lane = threadIdx.x & 31, row = threadIdx.x >> 5;
    const int n_tiles = B * tiles_h * tiles_w;
    G4<T> pre[PER];
    auto fetch = [&](int tile) {
        const TileXY t = tile_xy(tile, tiles_h, tiles_w, TH, TW);
        // g window: oh in [ih0/2 - 1, ih0/2 + TH/2] (oh = (ih + pt - kh)/2, pt in {0,1}), ow likewise (ih0, iw0 even)
        const int goh0 = t.r0 / 2 - 1, gow0 = t.c0 / 2 - 1;
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            const int idx = threadIdx.x + k * kThreads;
            const int v4 = idx % (COUT / 4), p = idx / (COUT / 4);
            const int gr = p / GW_T, gc = p - gr * GW_T;
            const int oh = goh0 + gr, ow = gow0 + gc;
            pre[k].zero();
            if (idx < NV && oh >= 0 && oh < OH && ow >= 0 && ow < OW)
                pre[k].load(g + (((size_t)t.b * OH + oh) * OW + ow) * COUT + 4 * v4);
        }
    };
    if ((int)blockIdx.x < n_tiles) fetch(blockIdx.x);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TileXY tc = tile_xy(tile, tiles_h, tiles_w, TH, TW);
        const int ih0 = tc.r0, iw0 = tc.c0, b = tc.b;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            const int idx = threadIdx.x + k * kThreads;
            if (idx < NV) *reinterpret_cast<float4*>(&s_g[(idx / (COUT / 4)) * GP + 4 * (idx % (COUT / 4))]) = pre[k].get();
        }
        __syncthreads();
        if (tile + (int)gridDim.x < n_tiles) fetch(tile + gridDim.x);
#pragma unroll
        for (int pw = 0; pw < 2; ++pw) {
            const int cl = 2 * lane + pw;  // column inside the tile
            float acc[CIN] = {0.f, 0.f, 0.f};
#pragma unroll
            for (int kh = 0; kh < KS; ++kh) {
                if (((row + pt - kh) & 1) != 0) continue;  // ih0 even: parity of ih+pt-kh = parity of row+pt-kh (warp-uniform)
                const int gr = (row + pt - kh + 2) / 2;     // (ih + pt - kh)/2 - goh0
#pragma unroll
                for (int kw = 0; kw < KS; ++kw) {
                    if (((pw + pl - kw) & 1) != 0) continue;  // warp-uniform
                    const int gc = (cl + pl - kw + 2) / 2;
                    const float4* gp = reinterpret_cast<const float4*>(&s_g[(gr * GW_T + gc) * GP]);
                    const float4* wp = reinterpret_cast<const float4*>(&ws[(kh * KS + kw) * CIN * COUT]);
#pragma unroll
                    for (int c4 = 0; c4 < COUT / 4; ++c4) {
                        const float4 gv = gp[c4];
#pragma unroll
                        for (int ci = 0; ci < CIN; ++ci) {
                            const float4 ww = wp[ci * (COUT / 4) + c4];
                            acc[ci] = fmaf(gv.x, ww.x, acc[ci]);
                            acc[ci] = fmaf(gv.y, ww.y, acc[ci]);
                            acc[ci] = fmaf(gv.z, ww.z, acc[ci]);
                            acc[ci] = fmaf(gv.w, ww.w, acc[ci]);
                        }
                    }
                }
            }
#pragma unroll
            for (int ci = 0; ci < CIN; ++ci) s_out[(row * TW + cl) * CIN + ci] = from_f32<T>(acc[ci]);
        }
        __syncthreads();
        const int vw = min(TW, W - iw0), vh = min(TH, H - ih0);
        copy_rows_out(gin + (((size_t)b * H + ih0) * W + iw0) * CIN, (long long)W * CIN, s_out, TW * CIN, vh, vw * CIN);
    }
}

// =================================================================================================
// Weight gradients with 3 output channels (which 0: 48 weights, which 1: 81 weights): thread = pixel,
// all weight partial sums in registers across the CTA's tiles, one reduction at the end.
// =================================================================================================
template <typename TI, typename TG, int CIN, int KS, int S>
__global__ void __launch_bounds__(kThreads, 2) conv3out_wgrad_kernel(const TI* __restrict__ in,
                                                                     const float* __restrict__ in_a,
                                                                     const float* __restrict__ in_b, int act,
                                                                     const TG* __restrict__ g, float* __restrict__ dw,
                                                                     long long* __restrict__ dw_acc,
                                                                     int B, int H, int W, int OH, int OW, int pt,
                                                                     int pl, int tiles_h, int tiles_w) {
    constexpr int COUT = 3, TH = C3W_TH, TW = C3_TW;
    constexpr int IH_T = (TH - 1) * S + KS, IW_T = (TW - 1) * S + KS;
    typedef Window<TI, CIN, IH_T, IW_T> Win;
    constexpr int ROWP = Win::ROWP;
    constexpr int NW = KS * KS * CIN * COUT;
    constexpr int GROW = TW * COUT, GPITCH = GROW + 1, GEPL = GROW / 32;  // gradient tile: one row per warp (TH == 8)
    static_assert(TH == 8 && GROW % 32 == 0, "gradient tile mapping");
    __shared__ float s_in[IH_T * ROWP];
    __shared__ float s_g[TH * GPITCH];
    __shared__ float sab[2 * CIN];
    __shared__ float sacc[NW];
    if (threadIdx.x < CIN) {
        sab[threadIdx.x] = in_a ? in_a[threadIdx.x] : 1.f;
        sab[CIN + threadIdx.x] = in_a ? in_b[threadIdx.x] : 0.f;
    }
    for (int i = threadIdx.x; i < NW; i += kThreads) sacc[i] = 0.f;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float acc[NW];
#pragma unroll
    for (int i = 0; i < NW; ++i) acc[i] = 0.f;
    const int n_tiles = B * tiles_h * tiles_w;
    Win win;
    TG graw[GEPL];
    auto fetch = [&](int tile) {
        const TileXY t = tile_xy(tile, tiles_h, tiles_w, TH, TW);
        win.fetch(in + (size_t)t.b * H * W * CIN, H, W, t.r0 * S - pt, t.c0 * S - pl);
        const int oh = t.r0 + warp;  // gradient row of this warp
        const int e_hi = min(TW, OW - t.c0) * COUT;
        const TG* rowp = g + (((size_t)t.b * OH + oh) * OW + t.c0) * COUT;
#pragma unroll
        for (int j = 0; j < GEPL; ++j) {
            const int e = lane + 32 * j;
            graw[j] = from_f32<TG>(0.f);
            if (oh < OH && e < e_hi) graw[j] = rowp[e];
        }
    };
    if ((int)blockIdx.x < n_tiles) fetch(blockIdx.x);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TileXY tc = tile_xy(tile, tiles_h, tiles_w, TH, TW);
        __syncthreads();
        win.commit(s_in, sab, in_a != nullptr, act, H, W, tc.r0 * S - pt, tc.c0 * S - pl);
#pragma unroll
        for (int j = 0; j < GEPL; ++j) s_g[warp * GPITCH + lane + 32 * j] = to_f32(graw[j]);  // zero outside the output
        __syncthreads();
        if (tile + (int)gridDim.x < n_tiles) fetch(tile + gridDim.x);
#pragma unroll 1
        for (int pp = 0; pp < TH / 4; ++pp) {
            const int r = ty + 4 * pp;
            float gv[COUT];
#pragma unroll
            for (int co = 0; co < COUT; ++co) gv[co] = s_g[r * GPITCH + tx * COUT + co];
#pragma unroll
            for (int kh = 0; kh < KS; ++kh)
#pragma unroll
                for (int kw = 0; kw < KS; ++kw)
#pragma unroll
                    for (int ci = 0; ci < CIN; ++ci) {
                        const float v = s_in[(r * S + kh) * ROWP + (tx * S + kw) * CIN + ci];
#pragma unroll
                        for (int co = 0; co < COUT; ++co)
                            acc[((kh * KS + kw) * CIN + ci) * COUT + co] =
                                fmaf(v, gv[co], acc[((kh * KS + kw) * CIN + ci) * COUT + co]);
                    }
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NW; ++i) acc[i] = warp_sum(acc[i]);
    // the warps add their sums one after the other (fixed order: the CTA's partial is the same in every run)
    for (int w_ = 0; w_ < kThreads / 32; ++w_) {
        if ((threadIdx.x >> 5) == w_ && (threadIdx.x & 31) == 0) {
#pragma unroll
            for (int i = 0; i < NW; ++i) sacc[i] += acc[i];
        }
        __syncthreads();
    }
    // across CTAs: fp32 atomics (fast, order of the adds not fixed) or the order-independent accumulators
    for (int i = threadIdx.x; i < NW; i += kThreads) {
        if (dw_acc) stat_add(dw_acc, i, (double)sacc[i]);
        else atomicAdd(dw + i, sacc[i]);
    }
}

// =================================================================================================
// block1_conv1 weight gradient (3x3 s2 valid, 3 -> 32; 864 weights): a warp covers 4 output pixels x
// 8 groups of 4 output channels; a thread keeps 27 x 4 partial sums in registers.
// =================================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads, 1) conv_b1c1_wgrad_kernel(const T* __restrict__ in,
                                                                      const float* __restrict__ in_a,
                                                                      const float* __restrict__ in_b, int act,
                                                                      const T* __restrict__ g, float* __restrict__ dw,
                                                                      long long* __restrict__ dw_acc,
                                                                      int B, int H, int W, int OH, int OW, int pt, int pl,
                                                                      int tiles_h, int tiles_w) {
    constexpr int CIN = 3, COUT = 32, KS = 3, S = 2, TH = 4, TW = 32;
    constexpr int IH_T = (TH - 1) * S + KS, IW_T = (TW - 1) * S + KS;
    typedef Window<T, CIN, IH_T, IW_T> Win;
    constexpr int ROWP = Win::ROWP;
    constexpr int GP = COUT + 4;
    constexpr int NT = KS * KS * CIN;  // 27
    constexpr int NV = TH * TW * (COUT / 4), GPER = NV / kThreads;
    __shared__ float s_in[IH_T * ROWP];
    __shared__ __align__(16) float s_g[TH * TW * GP];
    __shared__ float sab[2 * CIN];
    __shared__ float sacc[NT * COUT];
    if (threadIdx.x < CIN) {
        sab[threadIdx.x] = in_a ? in_a[threadIdx.x] : 1.f;
        sab[CIN + threadIdx.x] = in_a ? in_b[threadIdx.x] : 0.f;
    }
    for (int i = threadIdx.x; i < NT * COUT; i += kThreads) sacc[i] = 0.f;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int cg = lane & 7, ps = lane >> 3;  // channel group (4 channels), pixel slot within the warp
    float acc[NT][4];
#pragma unroll
    for (int t = 0; t < NT; ++t)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[t][j] = 0.f;
    const int n_tiles = B * tiles_h * tiles_w;
    Win win;
    G4<T> graw[GPER];
    auto fetch = [&](int tile) {
        const TileXY t = tile_xy(tile, tiles_h, tiles_w, TH, TW);
        win.fetch(in + (size_t)t.b * H * W * CIN, H, W, t.r0 * S - pt, t.c0 * S - pl);
#pragma unroll
        for (int k = 0; k < GPER; ++k) {
            const int idx = threadIdx.x + k * kThreads;
            const int v4 = idx % (COUT / 4), p = idx / (COUT / 4);
            const int r = p / TW, c = p - r * TW;
            const int oh = t.r0 + r, ow = t.c0 + c;
            graw[k].zero();
            if (oh < OH && ow < OW) graw[k].load(g + (((size_t)t.b * OH + oh) * OW + ow) * COUT + 4 * v4);
        }
    };
    if ((int)blockIdx.x < n_tiles) fetch(blockIdx.x);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TileXY tc = tile_xy(tile, tiles_h, tiles_w, TH, TW);
        __syncthreads();
        win.commit(s_in, sab, in_a != nullptr, act, H, W, tc.r0 * S - pt, tc.c0 * S - pl);
#pragma unroll
        for (int k = 0; k < GPER; ++k) {
            const int idx = threadIdx.x + k * kThreads;
            *reinterpret_cast<float4*>(&s_g[(idx / (COUT / 4)) * GP + 4 * (idx % (COUT / 4))]) = graw[k].get();
        }
        __syncthreads();
        if (tile + (int)gridDim.x < n_tiles) fetch(tile + gridDim.x);
        // 128 pixels per tile, 32 per pass (8 warps x 4 slots)
#pragma unroll 1
        for (int pass = 0; pass < TH * TW / 32; ++pass) {
            const int p = pass * 32 + warp * 4 + ps;
            const int r = p / TW, c = p - r * TW;
            const float4 gv = *reinterpret_cast<const float4*>(&s_g[p * GP + 4 * cg]);
#pragma unroll
            for (int kh = 0; kh < KS; ++kh)
#pragma unroll
                for (int kw = 0; kw < KS; ++kw)
#pragma unroll
                    for (int ci = 0; ci < CIN; ++ci) {
                        const float v = s_in[(r * S + kh) * ROWP + (c * S + kw) * CIN + ci];
                        const int t = (kh * KS + kw) * CIN + ci;
                        acc[t][0] = fmaf(v, gv.x, acc[t][0]);
                        acc[t][1] = fmaf(v, gv.y, acc[t][1]);
                        acc[t][2] = fmaf(v, gv.z, acc[t][2]);
                        acc[t][3] = fmaf(v, gv.w, acc[t][3]);
                    }
        }
    }
    __syncthreads();
    // reduce the 4 pixel slots of a warp, then the 8 warps through shared memory, one warp after the other (fixed
    // order: the CTA's partial is the same in every run)
#pragma unroll
    for (int t = 0; t < NT; ++t)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float s = acc[t][j];
            s += __shfl_xor_sync(0xffffffffu, s, 8);
            s += __shfl_xor_sync(0xffffffffu, s, 16);
            acc[t][j] = s;
        }
    for (int w_ = 0; w_ < kThreads / 32; ++w_) {
        if (warp == w_ && ps == 0) {
#pragma unroll
            for (int t = 0; t < NT; ++t)
#pragma unroll
                for (int j = 0; j < 4; ++j) sacc[t * COUT + 4 * cg + j] += acc[t][j];
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < NT * COUT; i += kThreads) {
        if (dw_acc) stat_add(dw_acc, i, (double)sacc[i]);
        else atomicAdd(dw + i, sacc[i]);
    }
}

// =================================================================================================
// Strip kernels for the 3 -> 3, 3x3 'same' stem convolutions (which 1) when W % 8 == 0: a thread owns a strip of
// 8 consecutive output pixels of one row. The kernels above read one shared-memory word per multiply-add operand
// (27 input reads + weight reads for 81 FMAs: bound by the shared-memory pipe, 15-25 % of the FP32 peak); here a
// thread reads the 10-pixel x 3-channel input run of its strip once per filter row with eight 16-byte loads and
// keeps it in registers: 24 loads for 648 FMAs. Same arithmetic (fp32 FMA in (ky, kx, ci) order per output) and
// same results as the pixel-per-thread kernels.
//   tile = 16 rows x 128 pixels, 256 threads = 16 rows x 16 strips; window = 18 rows x 130 pixels x 3, fp32,
//   pixel x0-1 at float 0 of a row so that strip j starts at float 24*j (16-byte aligned)
// Global memory is moved in aligned 16-byte chunks (W % 8 == 0 makes every row 16-byte aligned and every chunk
// entirely inside or outside its row); the next tile's chunks are in flight while the current tile is computed.
// =================================================================================================
constexpr int SK_TH = 16, SK_TW = 128, SK_WR = SK_TH + 2, SK_WE = (SK_TW + 2) * 3, SK_RP = 392;

template <typename T>
struct StripWindow {
    static constexpr int EPC = 16 / (int)sizeof(T);          // elements per 16-byte chunk
    static constexpr int NCH = 3 * SK_TW / EPC + 2;           // chunks per window row (one before, one after the tile's 384)
    static constexpr int PER = (SK_WR * NCH + kThreads - 1) / kThreads;
    static constexpr int STAGE_BYTES = SK_WR * NCH * 16;      // raw window of one tile
    static constexpr int STAGES = sizeof(T) == 2 ? 3 : 2;     // tiles in flight (cp.async groups)
    static __device__ __forceinline__ bool inside(int idx, int H, int W, int y0, int x0, int* y, int* e0) {
        const int wr = idx / NCH, m = idx - wr * NCH;
        *y = y0 - 1 + wr;
        *e0 = 3 * x0 + (m - 1) * EPC;
        return idx < SK_WR * NCH && *y >= 0 && *y < H && *e0 >= 0 && *e0 + EPC <= 3 * W;
    }
    // raw 16-byte chunks of one tile's window, global -> shared, asynchronously (one cp.async group per call)
    static __device__ __forceinline__ void issue(uint32_t stage, const T* __restrict__ img, int H, int W, int y0, int x0) {
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            const int idx = threadIdx.x + k * kThreads;
            int y, e0;
            if (inside(idx, H, W, y0, x0, &y, &e0))
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(stage + (uint32_t)idx * 16u),
                             "l"(img + ((size_t)y * W) * 3 + e0)
                             : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    // the thread's own chunks (same index map as issue(): visible after its cp.async.wait_group) -> affine +
    // activation (zero outside the image: padding follows the activation) -> fp32 window
    static __device__ __forceinline__ void transform(const uint8_t* __restrict__ stage, float* __restrict__ sm, const float* sab,
                                                     bool affine, int act, int H, int W, int y0, int x0) {
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            const int idx = threadIdx.x + k * kThreads;
            if (idx >= SK_WR * NCH) break;
            int y, e0;
            const bool live = inside(idx, H, W, y0, x0, &y, &e0);
            const int wr = idx / NCH, m = idx - wr * NCH;
            const int w0 = (m - 1) * EPC + 3;      // window float index of the chunk's first element
            int ch = ((m + 2) * EPC) % 3;          // channel of the chunk's first element (x0 * 3 is a multiple of 3)
            float v[EPC];
            const uint4 raw = live ? *reinterpret_cast<const uint4*>(stage + (size_t)idx * 16) : make_uint4(0u, 0u, 0u, 0u);
            if (sizeof(T) == 2) {
                const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    v[(2 * i) % EPC] = __uint_as_float(w[i] << 16);
                    v[(2 * i + 1) % EPC] = __uint_as_float(w[i] & 0xffff0000u);
                }
            } else {
                v[0] = __uint_as_float(raw.x); v[1 % EPC] = __uint_as_float(raw.y);
                v[2 % EPC] = __uint_as_float(raw.z); v[3 % EPC] = __uint_as_float(raw.w);
            }
#pragma unroll
            for (int i = 0; i < EPC; ++i) {
                float x = 0.f;
                if (live) {
                    x = v[i];
                    if (affine) x = apply_act(fmaf(x, sab[ch], sab[3 + ch]), act);
                }
                const int wi = w0 + i;
                if (wi >= 0 && wi < SK_WE) sm[wr * SK_RP + wi] = x;
                ch = ch == 2 ? 0 : ch + 1;
            }
        }
    }
    static constexpr size_t smem_bytes() { return (size_t)SK_WR * SK_RP * 4 + (size_t)STAGES * STAGE_BYTES; }
};
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// 24 consecutive elements (8 pixels x 3 channels) of a 16-byte aligned strip <-> fp32 registers
template <typename T> __device__ __forceinline__ void load_strip(const T* p, float (&v)[24]) {
    if (sizeof(T) == 2) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const uint4 r = reinterpret_cast<const uint4*>(p)[q];
            const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                v[8 * q + 2 * i] = __uint_as_float(w[i] << 16);
                v[8 * q + 2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
            }
        }
    } else {
#pragma unroll
        for (int q = 0; q < 6; ++q) {
            const float4 r = reinterpret_cast<const float4*>(p)[q];
            v[4 * q] = r.x; v[4 * q + 1] = r.y; v[4 * q + 2] = r.z; v[4 * q + 3] = r.w;
        }
    }
}
template <typename T> __device__ __forceinline__ void store_strip(T* p, const float (&v)[24]) {
    if (sizeof(T) == 2) {
#pragma unroll
        for (int q = 0; q < 3; ++q)
            reinterpret_cast<uint4*>(p)[q] = make_uint4(pack_bf16x2(v[8 * q], v[8 * q + 1]), pack_bf16x2(v[8 * q + 2], v[8 * q + 3]),
                                                        pack_bf16x2(v[8 * q + 4], v[8 * q + 5]), pack_bf16x2(v[8 * q + 6], v[8 * q + 7]));
    } else {
#pragma unroll
        for (int q = 0; q < 6; ++q)
            reinterpret_cast<float4*>(p)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    }
}

// MODE 0: forward (+ BatchNorm statistics of the output as stored)   MODE 2: data gradient (flipped, transposed
// kernel; times act'(mask_a * mask_z + mask_b) when mask_z is given)
template <typename T, int MODE>
__global__ void __launch_bounds__(kThreads, 2) conv3c3_strip_kernel(const T* __restrict__ in, const float* __restrict__ w,
                                                                    const float* __restrict__ in_a,
                                                                    const float* __restrict__ in_b, int act,
                                                                    T* __restrict__ out, long long* __restrict__ stats,
                                                                    const T* __restrict__ mask_z,
                                                                    const float* __restrict__ mask_a,
                                                                    const float* __restrict__ mask_b, int B, int H, int W,
                                                                    int tiles_h, int tiles_w) {
    typedef StripWindow<T> Win;
    extern __shared__ __align__(16) uint8_t sk_smem[];
    float* s_in = reinterpret_cast<float*>(sk_smem);
    uint8_t* stages = sk_smem + (size_t)SK_WR * SK_RP * 4;
    __shared__ __align__(16) float ws[27 * 4];  // [tap][ci][co padded to 4]
    __shared__ float sab[12];
    __shared__ float sred[(kThreads / 32) * 6];
    for (int i = threadIdx.x; i < 81; i += kThreads) {
        const int t = i / 9, rem = i % 9, ci = rem / 3, co = rem % 3;
        ws[(t * 3 + ci) * 4 + co] = MODE == 2 ? w[((8 - t) * 3 + co) * 3 + ci] : w[i];
    }
    if (threadIdx.x < 3) {
        sab[threadIdx.x] = in_a ? in_a[threadIdx.x] : 1.f;
        sab[3 + threadIdx.x] = in_a ? in_b[threadIdx.x] : 0.f;
        sab[6 + threadIdx.x] = (MODE == 2 && mask_z) ? mask_a[threadIdx.x] : 1.f;
        sab[9 + threadIdx.x] = (MODE == 2 && mask_z) ? mask_b[threadIdx.x] : 0.f;
    }
    const int j = threadIdx.x & 15, r = threadIdx.x >> 4;
    float ssum[3] = {0.f, 0.f, 0.f}, ssq[3] = {0.f, 0.f, 0.f};
    const int n_tiles = B * tiles_h * tiles_w;
    const uint32_t stage0 = (uint32_t)__cvta_generic_to_shared(stages);
    // STAGES - 1 tiles ahead: one cp.async group per tile slot (empty groups past the end keep the count uniform)
    auto issue = [&](int tile, int slot) {
        if (tile < n_tiles) {
            const TileXY t = tile_xy(tile, tiles_h, tiles_w, SK_TH, SK_TW);
            Win::issue(stage0 + (uint32_t)slot * Win::STAGE_BYTES, in + (size_t)t.b * H * W * 3, H, W, t.r0, t.c0);
        } else {
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
    };
#pragma unroll
    for (int p = 0; p < Win::STAGES - 1; ++p) issue(blockIdx.x + p * gridDim.x, p);
    int slot = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TileXY tc = tile_xy(tile, tiles_h, tiles_w, SK_TH, SK_TW);
        cp_async_wait<Win::STAGES - 2>();  // this thread's chunks of `tile` have landed
        __syncthreads();                   // the previous tile's readers are done with s_in
        Win::transform(stages + (size_t)slot * Win::STAGE_BYTES, s_in, sab, in_a != nullptr, act, H, W, tc.r0, tc.c0);
        __syncthreads();
        {   // refill the slot the PREVIOUS iteration consumed (every thread is past that transform)
            int ps = slot + Win::STAGES - 1;
            if (ps >= Win::STAGES) ps -= Win::STAGES;
            issue(tile + (Win::STAGES - 1) * (int)gridDim.x, ps);
        }
        if (++slot == Win::STAGES) slot = 0;
        const int y = tc.r0 + r, x = tc.c0 + 8 * j;
        if (y >= H || x >= W) continue;  // whole strip outside (W % 8 == 0): nothing to compute or count
        float acc[24];
#pragma unroll
        for (int i = 0; i < 24; ++i) acc[i] = 0.f;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            float xin[32];
            const float4* rp = reinterpret_cast<const float4*>(&s_in[(r + ky) * SK_RP + 24 * j]);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 t4 = rp[q];
                xin[4 * q] = t4.x; xin[4 * q + 1] = t4.y; xin[4 * q + 2] = t4.z; xin[4 * q + 3] = t4.w;
            }
#pragma unroll
            for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                for (int ci = 0; ci < 3; ++ci) {
                    const float4 wv = *reinterpret_cast<const float4*>(&ws[((ky * 3 + kx) * 3 + ci) * 4]);
#pragma unroll
                    for (int px = 0; px < 8; ++px) {
                        const float v = xin[3 * (px + kx) + ci];
                        acc[3 * px] = fmaf(v, wv.x, acc[3 * px]);
                        acc[3 * px + 1] = fmaf(v, wv.y, acc[3 * px + 1]);
                        acc[3 * px + 2] = fmaf(v, wv.z, acc[3 * px + 2]);
                    }
                }
        }
        const size_t o = (((size_t)tc.b * H + y) * W + x) * 3;
        if (MODE == 2 && mask_z) {
            float mz[24];
            load_strip(mask_z + o, mz);
#pragma unroll
            for (int i = 0; i < 24; ++i) {
                const float pre = fmaf(mz[i], sab[6 + i % 3], sab[9 + i % 3]);
                if (!(pre > 0.f)) acc[i] = (act == 2) ? 0.1f * acc[i] : (act == 1 ? 0.f : acc[i]);
            }
        }
        store_strip(out + o, acc);
        if (MODE == 0 && stats) {
#pragma unroll
            for (int i = 0; i < 24; ++i) {
                const float rr = round_to<T>(acc[i]);
                ssum[i % 3] += rr;
                ssq[i % 3] = fmaf(rr, rr, ssq[i % 3]);
            }
        }
    }
    if (MODE == 0 && stats) {
        __syncthreads();
#pragma unroll
        for (int co = 0; co < 3; ++co) {
            const float s_ = warp_sum(ssum[co]), q_ = warp_sum(ssq[co]);
            if ((threadIdx.x & 31) == 0) {
                sred[(threadIdx.x >> 5) * 6 + co] = s_;
                sred[(threadIdx.x >> 5) * 6 + 3 + co] = q_;
            }
        }
        __syncthreads();
        if (threadIdx.x < 6) {
            float t = 0.f;
            for (int w_ = 0; w_ < kThreads / 32; ++w_) t += sred[w_ * 6 + threadIdx.x];
            stat_add(stats, threadIdx.x, (double)t);
        }
    }
}

// weight gradient of the same convolution: 81 partial sums per thread, the strip's input run from shared memory
// (8 x 16-byte loads per filter row), its 8 x 3 output gradients straight from global memory
template <typename T>
__global__ void __launch_bounds__(kThreads, 1) conv3c3_wgrad_strip_kernel(const T* __restrict__ in,
                                                                          const float* __restrict__ in_a,
                                                                          const float* __restrict__ in_b, int act,
                                                                          const T* __restrict__ g, float* __restrict__ dw,
                                                                          long long* __restrict__ dw_acc, int B, int H,
                                                                          int W, int tiles_h, int tiles_w) {
    typedef StripWindow<T> Win;
    extern __shared__ __align__(16) uint8_t sk_smem[];
    float* s_in = reinterpret_cast<float*>(sk_smem);
    uint8_t* stages = sk_smem + (size_t)SK_WR * SK_RP * 4;
    __shared__ float sab[6];
    __shared__ float sacc[81];
    if (threadIdx.x < 3) {
        sab[threadIdx.x] = in_a ? in_a[threadIdx.x] : 1.f;
        sab[3 + threadIdx.x] = in_a ? in_b[threadIdx.x] : 0.f;
    }
    for (int i = threadIdx.x; i < 81; i += kThreads) sacc[i] = 0.f;
    const int j = threadIdx.x & 15, r = threadIdx.x >> 4;
    float acc[81];
#pragma unroll
    for (int i = 0; i < 81; ++i) acc[i] = 0.f;
    const int n_tiles = B * tiles_h * tiles_w;
    const uint32_t stage0 = (uint32_t)__cvta_generic_to_shared(stages);
    float gv[24];
    auto issue = [&](int tile, int slot) {
        if (tile < n_tiles) {
            const TileXY t = tile_xy(tile, tiles_h, tiles_w, SK_TH, SK_TW);
            Win::issue(stage0 + (uint32_t)slot * Win::STAGE_BYTES, in + (size_t)t.b * H * W * 3, H, W, t.r0, t.c0);
        } else {
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
    };
#pragma unroll
    for (int p = 0; p < Win::STAGES - 1; ++p) issue(blockIdx.x + p * gridDim.x, p);
    int slot = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TileXY tc = tile_xy(tile, tiles_h, tiles_w, SK_TH, SK_TW);
        const int y = tc.r0 + r, x = tc.c0 + 8 * j;
        const bool live = y < H && x < W;
        if (live) load_strip(g + (((size_t)tc.b * H + y) * W + x) * 3, gv);  // in flight across the two barriers
        cp_async_wait<Win::STAGES - 2>();
        __syncthreads();
        Win::transform(stages + (size_t)slot * Win::STAGE_BYTES, s_in, sab, in_a != nullptr, act, H, W, tc.r0, tc.c0);
        __syncthreads();
        {
            int ps = slot + Win::STAGES - 1;
            if (ps >= Win::STAGES) ps -= Win::STAGES;
            issue(tile + (Win::STAGES - 1) * (int)gridDim.x, ps);
        }
        if (++slot == Win::STAGES) slot = 0;
        if (!live) continue;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            float xin[32];
            const float4* rp = reinterpret_cast<const float4*>(&s_in[(r + ky) * SK_RP + 24 * j]);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 t4 = rp[q];
                xin[4 * q] = t4.x; xin[4 * q + 1] = t4.y; xin[4 * q + 2] = t4.z; xin[4 * q + 3] = t4.w;
            }
#pragma unroll
            for (int px = 0; px < 8; ++px)   // pixels in order: every partial sum adds its pixels left to right
#pragma unroll
                for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                    for (int ci = 0; ci < 3; ++ci) {
                        const float v = xin[3 * (px + kx) + ci];
#pragma unroll
                        for (int co = 0; co < 3; ++co)
                            acc[((ky * 3 + kx) * 3 + ci) * 3 + co] = fmaf(v, gv[3 * px + co], acc[((ky * 3 + kx) * 3 + ci) * 3 + co]);
                    }
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 81; ++i) acc[i] = warp_sum(acc[i]);
    // the warps add their sums one after the other (fixed order: the CTA's partial is the same in every run)
    for (int w_ = 0; w_ < kThreads / 32; ++w_) {
        if ((threadIdx.x >> 5) == w_ && (threadIdx.x & 31) == 0) {
#pragma unroll
            for (int i = 0; i < 81; ++i) sacc[i] += acc[i];
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < 81; i += kThreads) {
        if (dw_acc) stat_add(dw_acc, i, (double)sacc[i]);
        else atomicAdd(dw + i, sacc[i]);
    }
}

int persist_grid_tiles(long long n_tiles, int ctas_per_sm) {
    const long long cap = (long long)spnet_num_sms() * ctas_per_sm;
    return (int)(n_tiles < cap ? n_tiles : cap);
}

// dynamic shared memory above 48 KB is a per-device opt-in of each kernel: one flag array per kernel (the kernels
// share one function-pointer type, so the kernel itself is the template argument)
template <auto kern> int strip_smem_optin(size_t bytes, const char* who) {
    static bool configured[64] = {};
    return spnet_smem_optin(configured, kern, bytes, who);
}

}  // namespace

extern "C" {

// which: 0 = stem conv1 folded with AveragePooling2D(2): x0 fp32 [B,H,W,1] -> out [B,H/2,W/2,3], skip [B,H/2,W/2,1]
//            (w = K4 [4,4,1,3] from spnet_stem_k3_to_k4)
//        1 = stem conv 3->3, 3x3 same            [B,H,W,3] -> [B,H,W,3]
//        2 = block1_conv1 3->32, 3x3 s2 valid    [B,H,W,3] -> [B,(H-3)/2+1,(W-3)/2+1,32]
//        3 = MobileNet conv1 3->32, 3x3 s2 'same' (TF: no leading pad for an even size, one for an odd size)
//            -> [B,ceil(H/2),ceil(W/2),32]
// in_a/in_b (nullable) + act (0 none, 1 relu, 2 leaky 0.1) transform the input on load.
// stats (nullable): fp64 [2*Cout] batch-norm accumulators.
int spnet_conv_small_fwd(int which, const void* in, const float* w, const float* in_a, const float* in_b, int act,
                         void* out, void* skip, long long* stats, int dtype, int B, int H, int W, cudaStream_t stream) {
    SPNET_REQUIRE(in && w && out && B > 0 && H > 2 && W > 2, "conv_small_fwd: bad args");
    SPNET_REQUIRE((in_a == nullptr) == (in_b == nullptr), "conv_small_fwd: affine parameters come in pairs");
    if (which == 0) {
        SPNET_REQUIRE(skip, "conv_small_fwd(0): needs the skip output");
        const int OH = H / 2, OW = W / 2;
        const int th = ceil_div(OH, C3_TH), tw = ceil_div(OW, C3_TW);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, (conv3out_kernel<float, T, 1, 4, 2, 1><<<grid, kThreads, 0, stream>>>(
                                        reinterpret_cast<const float*>(in), w, in_a, in_b, act, reinterpret_cast<T*>(out),
                                        reinterpret_cast<T*>(skip), stats, nullptr, nullptr, nullptr, B, H, W, OH, OW, 1,
                                        1, th, tw)));
    } else if (which == 1 && W % 8 == 0) {
        const int th = ceil_div(H, SK_TH), tw = ceil_div(W, SK_TW);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, const size_t smem = StripWindow<T>::smem_bytes();
                                    if (int rc = strip_smem_optin<conv3c3_strip_kernel<T, 0>>(smem, "conv_small_fwd")) return rc;
                                    conv3c3_strip_kernel<T, 0><<<grid, kThreads, smem, stream>>>(
                                        reinterpret_cast<const T*>(in), w, in_a, in_b, act, reinterpret_cast<T*>(out), stats,
                                        nullptr, nullptr, nullptr, B, H, W, th, tw));
    } else if (which == 1) {
        const int th = ceil_div(H, C3_TH), tw = ceil_div(W, C3_TW);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, (conv3out_kernel<T, T, 3, 3, 1, 0><<<grid, kThreads, 0, stream>>>(
                                        reinterpret_cast<const T*>(in), w, in_a, in_b, act, reinterpret_cast<T*>(out),
                                        nullptr, stats, nullptr, nullptr, nullptr, B, H, W, H, W, 1, 1, th, tw)));
    } else if (which == 2 || which == 3) {
        // 'same' stride 2 (which 3): out = ceil(n/2); TF pads (k - s)=1 at the end for even n, 1 + 1 for odd n
        const int OH = which == 2 ? (H - 3) / 2 + 1 : (H + 1) / 2, OW = which == 2 ? (W - 3) / 2 + 1 : (W + 1) / 2;
        const int pt = which == 3 ? (H & 1) : 0, pl = which == 3 ? (W & 1) : 0;
        const int th = ceil_div(OH, 4), tw = ceil_div(OW, 64);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, (conv_b1c1_fwd_kernel<T><<<grid, kThreads, 0, stream>>>(
                                        reinterpret_cast<const T*>(in), w, in_a, in_b, act, reinterpret_cast<T*>(out),
                                        stats, B, H, W, OH, OW, pt, pl, th, tw)));
    } else {
        spnet_set_error("conv_small_fwd: unknown conv id %d", which);
        return SPNET_ERR_ARG;
    }
    return spnet_check_launch("conv_small_fwd");
}

// dw += weight gradient of the same three convolutions (dw zeroed by the caller).
// For which == 0, dw is the K4 gradient [4,4,1,3]; fold it with spnet_stem_k4grad_to_k3grad.
// dw_acc (nullable): order-independent accumulators (one entry per weight, spnet_acc_to_f32 adds them into dw): the
// cross-CTA sums are then bit-identical run to run instead of fp32 atomics whose order is not fixed
int spnet_conv_small_wgrad(int which, const void* in, const float* in_a, const float* in_b, int act, const void* g,
                           float* dw, long long* dw_acc, int dtype, int B, int H, int W, cudaStream_t stream) {
    SPNET_REQUIRE(in && g && dw && B > 0 && H > 2 && W > 2, "conv_small_wgrad: bad args");
    SPNET_REQUIRE((in_a == nullptr) == (in_b == nullptr), "conv_small_wgrad: affine parameters come in pairs");
    if (which == 0) {
        const int OH = H / 2, OW = W / 2;
        const int th = ceil_div(OH, C3W_TH), tw = ceil_div(OW, C3_TW);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, (conv3out_wgrad_kernel<float, T, 1, 4, 2><<<grid, kThreads, 0, stream>>>(
                                        reinterpret_cast<const float*>(in), in_a, in_b, act, reinterpret_cast<const T*>(g),
                                        dw, dw_acc, B, H, W, OH, OW, 1, 1, th, tw)));
    } else if (which == 1 && W % 8 == 0) {
        const int th = ceil_div(H, SK_TH), tw = ceil_div(W, SK_TW);
        const int grid = persist_grid_tiles((long long)B * th * tw, 1);
        SPNET_DISPATCH_DTYPE(dtype, const size_t smem = StripWindow<T>::smem_bytes();
                                    if (int rc = strip_smem_optin<conv3c3_wgrad_strip_kernel<T>>(smem, "conv_small_wgrad")) return rc;
                                    conv3c3_wgrad_strip_kernel<T><<<grid, kThreads, smem, stream>>>(
                                        reinterpret_cast<const T*>(in), in_a, in_b, act, reinterpret_cast<const T*>(g), dw,
                                        dw_acc, B, H, W, th, tw));
    } else if (which == 1) {
        const int th = ceil_div(H, C3W_TH), tw = ceil_div(W, C3_TW);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, (conv3out_wgrad_kernel<T, T, 3, 3, 1><<<grid, kThreads, 0, stream>>>(
                                        reinterpret_cast<const T*>(in), in_a, in_b, act, reinterpret_cast<const T*>(g), dw,
                                        dw_acc, B, H, W, H, W, 1, 1, th, tw)));
    } else if (which == 2 || which == 3) {
        const int OH = which == 2 ? (H - 3) / 2 + 1 : (H + 1) / 2, OW = which == 2 ? (W - 3) / 2 + 1 : (W + 1) / 2;
        const int pt = which == 3 ? (H & 1) : 0, pl = which == 3 ? (W & 1) : 0;
        const int th = ceil_div(OH, 4), tw = ceil_div(OW, 32);
        const int grid = persist_grid_tiles((long long)B * th * tw, 1);  // 134 registers x 256 threads: one CTA per SM
        SPNET_DISPATCH_DTYPE(dtype, (conv_b1c1_wgrad_kernel<T><<<grid, kThreads, 0, stream>>>(
                                        reinterpret_cast<const T*>(in), in_a, in_b, act, reinterpret_cast<const T*>(g), dw,
                                        dw_acc, B, H, W, OH, OW, pt, pl, th, tw)));
    } else {
        spnet_set_error("conv_small_wgrad: unknown conv id %d", which);
        return SPNET_ERR_ARG;
    }
    return spnet_check_launch("conv_small_wgrad");
}

// gin = data gradient (which = 1 or 2; conv 0 reads the network input, which has no gradient),
// multiplied by act'(mask_a*mask_z+mask_b) when mask_z is given. H, W are the INPUT dims.
int spnet_conv_small_dgrad(int which, const void* g, const float* w, const void* mask_z, const float* mask_a,
                           const float* mask_b, int act, void* gin, int dtype, int B, int H, int W,
                           cudaStream_t stream) {
    SPNET_REQUIRE(g && w && gin && B > 0 && H > 2 && W > 2, "conv_small_dgrad: bad args");
    SPNET_REQUIRE(!mask_z || (mask_a && mask_b), "conv_small_dgrad: mask needs its affine");
    if (which == 1 && W % 8 == 0) {
        const int th = ceil_div(H, SK_TH), tw = ceil_div(W, SK_TW);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, const size_t smem = StripWindow<T>::smem_bytes();
                                    if (int rc = strip_smem_optin<conv3c3_strip_kernel<T, 2>>(smem, "conv_small_dgrad")) return rc;
                                    conv3c3_strip_kernel<T, 2><<<grid, kThreads, smem, stream>>>(
                                        reinterpret_cast<const T*>(g), w, nullptr, nullptr, act, reinterpret_cast<T*>(gin),
                                        nullptr, reinterpret_cast<const T*>(mask_z), mask_a, mask_b, B, H, W, th, tw));
    } else if (which == 1) {
        // 'same' 3x3 stride 1: the data gradient is the convolution of g with the flipped, transposed kernel
        const int th = ceil_div(H, C3_TH), tw = ceil_div(W, C3_TW);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, (conv3out_kernel<T, T, 3, 3, 1, 2><<<grid, kThreads, 0, stream>>>(
                                        reinterpret_cast<const T*>(g), w, nullptr, nullptr, act, reinterpret_cast<T*>(gin),
                                        nullptr, nullptr, reinterpret_cast<const T*>(mask_z), mask_a, mask_b, B, H, W, H, W,
                                        1, 1, th, tw)));
    } else if (which == 2 || which == 3) {
        SPNET_REQUIRE(!mask_z, "conv_small_dgrad(2|3): these convolutions read the stem output directly (no activation mask)");
        const int OH = which == 2 ? (H - 3) / 2 + 1 : (H + 1) / 2, OW = which == 2 ? (W - 3) / 2 + 1 : (W + 1) / 2;
        const int pt = which == 3 ? (H & 1) : 0, pl = which == 3 ? (W & 1) : 0;
        const int th = ceil_div(H, 8), tw = ceil_div(W, 64);
        const int grid = persist_grid_tiles((long long)B * th * tw, 2);
        SPNET_DISPATCH_DTYPE(dtype, (conv_b1c1_dgrad_kernel<T><<<grid, kThreads, 0, stream>>>(
                                        reinterpret_cast<const T*>(g), w, reinterpret_cast<T*>(gin), B, H, W, OH, OW, pt, pl,
                                        th, tw)));
    } else {
        spnet_set_error("conv_small_dgrad: unknown conv id %d", which);
        return SPNET_ERR_ARG;
    }
    return spnet_check_launch("conv_small_dgrad");
}

}  // extern "C"
