// Depthwise 3x3 (stride 1, 'same', NHWC) forward and fused backward, the depthwise half of keras
// SeparableConv2D as used by keras.applications.Xception (reference call site spnet/models.py:359).
//
// HBM-bound by nature (18 FLOP per 4 bytes moved), so the design goal is to keep the instruction
// issue rate out of the way of the memory system:
//   * lane = one channel PAIR (a 32-bit bf16x2 word, or a float2): a warp covers the 64 channels
//     of one pixel with one conflict-free 128-byte shared-memory access, all per-pixel predicates
//     (row / column inside the image) are warp-uniform, and all arithmetic is packed fp32
//     (fma.rn.f32x2 — one issue slot per two FMAs, fp32 accumulation);
//   * a warp owns NC adjacent columns and slides down the rows of a tile, so every staged input
//     is widened / BN-transformed once per row and reused by three running accumulators;
//   * tiles INCLUDING their halo arrive by TMA (one 4-D box per tile, the out-of-image halo is
//     filled by the TMA unit) into an S-stage full/empty mbarrier ring (lane 0 of warp 0 issues
//     the loads S-1 tiles ahead), so the next tiles stream in while the warps compute and no
//     CTA-wide barrier sits in the loop.
// Xception is pre-activation (ReLU -> sepconv -> BN) and in training the producer's BatchNorm can
// only be applied once its batch statistics exist, so BN-apply (per-channel affine) + ReLU are
// fused on the LOAD side here. TF applies zero padding AFTER that transform: with AFFINE+RELU the
// TMA map fills the halo with NaN, which the affine keeps and fmaxf(NaN, 0) turns into the exact
// zero the padding needs — no per-element masking in the hot loop.
#include "tma.cuh"

namespace {

constexpr int CB = 64;        // channels per CTA: 32 lanes x one channel pair
constexpr int MAX_STAGES = 6;

// ---- packed fp32 pair arithmetic (FFMA2 / FMUL2 / FADD2) ---------------------------------------
__device__ __forceinline__ uint64_t pk(float2 v) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(v.x), "f"(v.y));
    return r;
}
__device__ __forceinline__ float2 upk(uint64_t r) {
    float2 v;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(v.x), "=f"(v.y) : "l"(r));
    return v;
}
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)), "l"(pk(c)));
    return upk(d);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)));
    return upk(d);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk(a)), "l"(pk(b)));
    return upk(d);
}
__device__ __forceinline__ float2 relu2(float2 v) { return make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f)); }
// activation applied on load: RELU = 0 none, 1 ReLU (Xception), 2 ReLU6 (MobileNet). NaN (the padding fill) maps to 0.
template <int RELU> __device__ __forceinline__ float2 act2(float2 v) {
    if (RELU == 1) return relu2(v);
    if (RELU == 2) return make_float2(fminf(fmaxf(v.x, 0.f), 6.f), fminf(fmaxf(v.y, 0.f), 6.f));
    return v;
}
template <int RELU> __device__ __forceinline__ bool act_open(float pre) {  // derivative of the activation is 1
    if (RELU == 1) return pre > 0.f;
    if (RELU == 2) return pre > 0.f && pre < 6.f;
    return true;
}

// ---- one channel pair of one pixel: raw (as stored) and widened (fp32) forms --------------------
template <typename T> struct PairOf;
template <> struct PairOf<bf16> { typedef uint32_t raw; static constexpr uint32_t bytes = 4; };
template <> struct PairOf<float> { typedef float2 raw; static constexpr uint32_t bytes = 8; };

__device__ __forceinline__ uint32_t lds_raw(uint32_t addr, const bf16*) {
    uint32_t w;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(addr));
    return w;
}
__device__ __forceinline__ float2 lds_raw(uint32_t addr, const float*) {
    float2 w;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(w.x), "=f"(w.y) : "r"(addr));
    return w;
}
__device__ __forceinline__ uint32_t ldg_raw(const bf16* p) { return __ldg(reinterpret_cast<const uint32_t*>(p)); }
__device__ __forceinline__ float2 ldg_raw(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
__device__ __forceinline__ float2 widen(uint32_t w) {
    return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ float2 widen(float2 w) { return w; }
__device__ __forceinline__ void stg_pair(bf16* p, float2 v) { *reinterpret_cast<uint32_t*>(p) = pack_bf16x2(v.x, v.y); }
__device__ __forceinline__ void stg_pair(float* p, float2 v) { *reinterpret_cast<float2*>(p) = v; }
// the pair as it will read back after being stored as T
__device__ __forceinline__ float2 round_pair(float2 v, const bf16*) { return widen(pack_bf16x2(v.x, v.y)); }
__device__ __forceinline__ float2 round_pair(float2 v, const float*) { return v; }

__device__ __forceinline__ void mbar_arrive_cta(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void consumer_bar_sync(int nthreads) {
    asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

struct TileCoord { int b, h0, w0; };
__device__ __forceinline__ TileCoord tile_coord(int tile, int tiles_w, int tiles_h, int TH, int TW) {
    TileCoord t;
    const int tw = tile % tiles_w;
    const int q = tile / tiles_w;
    t.w0 = tw * TW;
    t.h0 = (q % tiles_h) * TH;
    t.b = q / tiles_h;
    return t;
}

// =================================================================================================
// Forward:  out = dw3x3(act(in)),  act(v) = relu?(in_a*v + in_b)
// CTA = TW/NC warps; blockIdx.y = 64-channel chunk, blockIdx.x walks
// (image, row-tile, col-tile) tiles round-robin.
// =================================================================================================
// one lane of a converged warp, always the same one, in a form the compiler treats as a single thread
__device__ __forceinline__ uint32_t elect_one_lane() {
    uint32_t leader;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));
    return leader;
}

template <typename T, int NC, bool AFFINE, int RELU>
__global__ void __launch_bounds__(256, 2)
dw3x3_fwd_packed_kernel(const __grid_constant__ CUtensorMap tm_in, const float* __restrict__ k,
                        const float* __restrict__ in_a, const float* __restrict__ in_b, T* __restrict__ out, int B,
                        int H, int W, int C, int TH, int TW, int tiles_h, int tiles_w, int S) {
    constexpr uint32_t PB = PairOf<T>::bytes, PIX = 32 * PB;  // bytes of one pixel's 64-channel slice
    constexpr bool MASK = AFFINE && RELU == 0;                // explicit padding mask (no NaN trick without ReLU)
    typedef typename PairOf<T>::raw raw_t;
    extern __shared__ uint8_t dwp_smem[];
    __shared__ __align__(8) uint64_t bars[2 * MAX_STAGES];
    const uint32_t sbase = (smem_u32(dwp_smem) + 127u) & ~127u;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[MAX_STAGES]);
    // through a shuffle so that the compiler knows the warp index is warp-uniform (uniform-datapath address math,
    // no ELECT / R2UR loops around the TMA issue)
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int ncons = blockDim.x >> 5;
    const int cbase = blockIdx.y * CB;
    const int TWH = TW + 2;
    const uint32_t row_bytes = (uint32_t)TWH * PIX;
    const uint32_t stage_bytes = (uint32_t)(TH + 2) * row_bytes;
    const int n_tiles = B * tiles_h * tiles_w;

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, ncons);
        }
        mbar_fence_init();
    }
    __syncthreads();

    // Producer duty: lane 0 of warp 0 keeps S-1 tiles in flight. Stage (it-1)%S is refilled at the
    // start of tile `it`, once every warp has released it (empty barrier).
    auto issue = [&](int tile, int s) {
        const TileCoord t = tile_coord(tile, tiles_w, tiles_h, TH, TW);
        mbar_expect_tx(full0 + 8 * s, stage_bytes);
        tma_load_4d(sbase + s * stage_bytes, &tm_in, full0 + 8 * s, cbase, t.w0 - 1, t.h0 - 1, t.b);
    };
    if (threadIdx.x == 0)
        for (int i = 0; i < S - 1; ++i)
            if ((int)blockIdx.x + i * (int)gridDim.x < n_tiles) issue(blockIdx.x + i * gridDim.x, i);

    // ---------------- consumers ----------------
    const int c0 = cbase + lane * 2;
    const bool c_ok = c0 < C;  // C is even, so a pair is valid or invalid as a whole
    float2 wt[9], av, bv;
#pragma unroll
    for (int t = 0; t < 9; ++t) wt[t] = c_ok ? make_float2(k[t * C + c0], k[t * C + c0 + 1]) : make_float2(0.f, 0.f);
    av = (AFFINE && c_ok) ? make_float2(in_a[c0], in_a[c0 + 1]) : make_float2(1.f, 1.f);
    bv = (AFFINE && c_ok) ? make_float2(in_b[c0], in_b[c0 + 1]) : make_float2(0.f, 0.f);
    const int col0 = warp * NC;
    const size_t rowC = (size_t)W * C;
    float2 A_[NC], B_[NC], C_[NC];
#pragma unroll
    for (int oc = 0; oc < NC; ++oc) A_[oc] = B_[oc] = C_[oc] = make_float2(0.f, 0.f);

    // Producer duty rotates over the warps (tile i of this CTA is refilled by warp i % ncons): the refill has to
    // wait until EVERY warp has released the stage and then costs a few hundred cycles of coordinate decode + TMA
    // issue; pinned to warp 0 that made warp 0 the last one through every tile and the pace of the whole CTA.
    const uint32_t issuer_lane = elect_one_lane();
    int s = 0, n = 0, duty = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (warp == duty) {  // warp-uniform
            const int nt = tile + (S - 1) * (int)gridDim.x;
            if (nt < n_tiles) {
                const int sp = s == 0 ? S - 1 : s - 1;  // the stage the previous tile used
                if (tile != (int)blockIdx.x) mbar_wait(empty0 + 8 * sp, (uint32_t)(s == 0 ? n - 1 : n) & 1u);
                if (issuer_lane) issue(nt, sp);
            }
        }
        if (++duty == ncons) duty = 0;
        const TileCoord tc = tile_coord(tile, tiles_w, tiles_h, TH, TW);
        const int h0 = tc.h0, w0 = tc.w0;
        mbar_wait(full0 + 8 * s, (uint32_t)n & 1u);
        if (w0 + col0 < W) {  // warp-uniform: this warp owns at least one image column of the tile
            const int rows = min(TH, H - h0) + 2;
            bool stv[NC], colok[NC + 2];
#pragma unroll
            for (int oc = 0; oc < NC; ++oc) stv[oc] = c_ok && (w0 + col0 + oc) < W;
#pragma unroll
            for (int j = 0; j < NC + 2; ++j) {
                const int iw = w0 - 1 + col0 + j;
                colok[j] = iw >= 0 && iw < W;
            }
            uint32_t s_row = sbase + s * stage_bytes + (uint32_t)(col0 * 32 + lane) * PB;
            T* o_ptr = out + ((size_t)tc.b * H + h0) * rowC + (size_t)(w0 + col0) * C + c0;
            raw_t cur[NC + 2];
#pragma unroll
            for (int j = 0; j < NC + 2; ++j) cur[j] = lds_raw(s_row + j * PIX, (const T*)nullptr);
            int r = 0;
            auto step = [&](float2 (&P)[NC], float2 (&Q)[NC], float2 (&R)[NC]) {
                float2 x[NC + 2];
                const bool rowok = MASK ? ((h0 - 1 + r) >= 0 && (h0 - 1 + r) < H) : true;
#pragma unroll
                for (int j = 0; j < NC + 2; ++j) {
                    float2 v = widen(cur[j]);
                    if (AFFINE) v = ffma2(v, av, bv);
                    v = act2<RELU>(v);
                    if (MASK && !(rowok && colok[j])) v = make_float2(0.f, 0.f);
                    x[j] = v;
                }
                if (r + 1 < rows) {  // next row's raw words are in flight while this row is computed
                    s_row += row_bytes;
#pragma unroll
                    for (int j = 0; j < NC + 2; ++j) cur[j] = lds_raw(s_row + j * PIX, (const T*)nullptr);
                }
#pragma unroll
                for (int oc = 0; oc < NC; ++oc) {
                    R[oc] = fmul2(x[oc], wt[0]);  // R starts here: no accumulator zeroing anywhere
#pragma unroll
                    for (int kw = 0; kw < 3; ++kw) {
                        P[oc] = ffma2(x[oc + kw], wt[6 + kw], P[oc]);
                        Q[oc] = ffma2(x[oc + kw], wt[3 + kw], Q[oc]);
                        if (kw) R[oc] = ffma2(x[oc + kw], wt[kw], R[oc]);
                    }
                }
                if (r >= 2) {  // P now holds output row h0 + r - 2
#pragma unroll
                    for (int oc = 0; oc < NC; ++oc)
                        if (stv[oc]) stg_pair(o_ptr + (size_t)oc * C, P[oc]);
                    o_ptr += rowC;
                }
                ++r;
            };
            while (r + 3 <= rows) { step(A_, B_, C_); step(B_, C_, A_); step(C_, A_, B_); }
            if (r < rows) { step(A_, B_, C_); if (r < rows) step(B_, C_, A_); }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_cta(empty0 + 8 * s);
        if (++s == S) { s = 0; ++n; }
    }
}

// =================================================================================================
// Fused backward of the depthwise stage: ONE pass over (gout, in) produces
//   gin   = dw3x3^T(gout) * relu'(in_a*in+in_b)  [+ add_src] [+ add_strided at even (h,w)]
//   dk   += sum act(in)[h+kh-1, w+kw-1] * gout[h, w]                      (weight gradient)
//   stats += (sum gin, sum gin * xhat),  xhat = (in - mean)*rstd          (BatchNorm-backward sums of
//            the BN that produced `in`; only when stats != nullptr)
// Both gradients use the SAME 3x3 neighbourhood G of gout around a pixel p:
//   gin[p] = sum_n G_n * kflip_n,   dkflip_n += act(in)[p] * G_n
// so a thread keeps a 3-row window of the gradient in registers and runs both from it.
// Stage = gout tile with halo (zero-filled) + in tile (+ add_src tile), one mbarrier.
// EPI: 0 none, 1 add_src (TMA-staged), 2 add_strided (global loads at even rows/columns).
// =================================================================================================
template <typename T, bool AFFINE, int RELU, int EPI>
__global__ void __launch_bounds__(512, 1)
dw3x3_bwd_packed_kernel(const __grid_constant__ CUtensorMap tm_g, const __grid_constant__ CUtensorMap tm_x,
                        const __grid_constant__ CUtensorMap tm_add, const float* __restrict__ k,
                        const float* __restrict__ in_a, const float* __restrict__ in_b,
                        const float* __restrict__ bn_mean, const float* __restrict__ bn_rstd, long long* __restrict__ stats,
                        const T* __restrict__ add_strided, T* __restrict__ gin, float* __restrict__ dk,
                        long long* __restrict__ dk_acc, int B, int H, int W, int C, int TH, int TW, int tiles_h, int tiles_w, int S) {
    constexpr int NC = 2;
    constexpr uint32_t PB = PairOf<T>::bytes, PIX = 32 * PB;
    typedef typename PairOf<T>::raw raw_t;
    extern __shared__ uint8_t dwp_smem[];
    __shared__ __align__(8) uint64_t bars[2 * MAX_STAGES];
    const uint32_t sbase = (smem_u32(dwp_smem) + 127u) & ~127u;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[MAX_STAGES]);
    // through a shuffle so that the compiler knows the warp index is warp-uniform (uniform-datapath address math,
    // no ELECT / R2UR loops around the TMA issue)
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int ncons = blockDim.x >> 5;
    const int cbase = blockIdx.y * CB;
    const int TWH = TW + 2;
    const uint32_t grow_bytes = (uint32_t)TWH * PIX;           // gradient tile row (with halo)
    const uint32_t g_bytes = (uint32_t)(TH + 2) * grow_bytes;
    const uint32_t xrow_bytes = (uint32_t)TW * PIX;            // input / add tile row
    const uint32_t x_bytes = (uint32_t)TH * xrow_bytes;
    const uint32_t stage_bytes = g_bytes + x_bytes * (EPI == 1 ? 2u : 1u);
    const int n_tiles = B * tiles_h * tiles_w;

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, ncons);
        }
        mbar_fence_init();
    }
    __syncthreads();

    auto issue = [&](int tile, int s) {
        const TileCoord t = tile_coord(tile, tiles_w, tiles_h, TH, TW);
        const uint32_t dst = sbase + s * stage_bytes, bar = full0 + 8 * s;
        mbar_expect_tx(bar, stage_bytes);
        tma_load_4d(dst, &tm_g, bar, cbase, t.w0 - 1, t.h0 - 1, t.b);
        tma_load_4d(dst + g_bytes, &tm_x, bar, cbase, t.w0, t.h0, t.b);
        if (EPI == 1) tma_load_4d(dst + g_bytes + x_bytes, &tm_add, bar, cbase, t.w0, t.h0, t.b);
    };
    if (threadIdx.x == 0)
        for (int i = 0; i < S - 1; ++i)
            if ((int)blockIdx.x + i * (int)gridDim.x < n_tiles) issue(blockIdx.x + i * gridDim.x, i);

    // ---------------- consumers ----------------
    const int c0 = cbase + lane * 2;
    const bool c_ok = c0 < C;
    float2 kf[9], dkf[9], av, bv, s1, s2;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        kf[t] = c_ok ? make_float2(k[(8 - t) * C + c0], k[(8 - t) * C + c0 + 1]) : make_float2(0.f, 0.f);
        dkf[t] = make_float2(0.f, 0.f);
    }
    av = (AFFINE && c_ok) ? make_float2(in_a[c0], in_a[c0 + 1]) : make_float2(1.f, 1.f);
    bv = (AFFINE && c_ok) ? make_float2(in_b[c0], in_b[c0 + 1]) : make_float2(0.f, 0.f);
    s1 = s2 = make_float2(0.f, 0.f);
    const int col0 = warp * NC;
    const size_t rowC = (size_t)W * C;
    const int H2 = (H + 1) >> 1, W2 = (W + 1) >> 1;
    float2 G0[NC + 2], G1[NC + 2], G2[NC + 2];

    // Producer duty rotates over the warps (tile i of this CTA is refilled by warp i % ncons): the refill has to
    // wait until EVERY warp has released the stage and then costs a few hundred cycles of coordinate decode + TMA
    // issue; pinned to warp 0 that made warp 0 the last one through every tile and the pace of the whole CTA.
    const uint32_t issuer_lane = elect_one_lane();
    int s = 0, n = 0, duty = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (warp == duty) {  // warp-uniform
            const int nt = tile + (S - 1) * (int)gridDim.x;
            if (nt < n_tiles) {
                const int sp = s == 0 ? S - 1 : s - 1;  // the stage the previous tile used
                if (tile != (int)blockIdx.x) mbar_wait(empty0 + 8 * sp, (uint32_t)(s == 0 ? n - 1 : n) & 1u);
                if (issuer_lane) issue(nt, sp);
            }
        }
        if (++duty == ncons) duty = 0;
        const TileCoord tc = tile_coord(tile, tiles_w, tiles_h, TH, TW);
        const int h0 = tc.h0, w0 = tc.w0;
        mbar_wait(full0 + 8 * s, (uint32_t)n & 1u);
        if (w0 + col0 < W) {
            const int nrow = min(TH, H - h0);
            const int rows = nrow + 2;
            const bool own1 = (w0 + col0 + 1) < W;  // column 0 is owned by the test above
            const uint32_t st = sbase + s * stage_bytes;
            uint32_t s_g = st + (uint32_t)(col0 * 32 + lane) * PB;
            uint32_t s_x = st + g_bytes + (uint32_t)(col0 * 32 + lane) * PB;
            T* o_ptr = gin + ((size_t)tc.b * H + h0) * rowC + (size_t)(w0 + col0) * C + c0;
            // column of this warp that is even in image coordinates (add_strided lands on even (h,w) only)
            const int oc_even = (w0 + col0) & 1;
            const T* sa_ptr = nullptr;
            if (EPI == 2)
                sa_ptr = add_strided + ((size_t)tc.b * H2 * W2 + (size_t)((w0 + col0 + oc_even) >> 1)) * C + c0;
            const bool sa_ok = EPI == 2 && c_ok && (w0 + col0 + oc_even) < W;
            raw_t cur[NC + 2];
#pragma unroll
            for (int j = 0; j < NC + 2; ++j) cur[j] = lds_raw(s_g + j * PIX, (const T*)nullptr);
            int r = 0;
            auto step = [&](float2 (&Ga)[NC + 2], float2 (&Gb)[NC + 2], float2 (&Gc)[NC + 2]) {
                // Gc <- gradient row r of the tile; window (Ga, Gb, Gc) = rows r-2, r-1, r; centre = Gb
#pragma unroll
                for (int j = 0; j < NC + 2; ++j) Gc[j] = widen(cur[j]);
                if (r + 1 < rows) {
                    s_g += grow_bytes;
#pragma unroll
                    for (int j = 0; j < NC + 2; ++j) cur[j] = lds_raw(s_g + j * PIX, (const T*)nullptr);
                }
                if (r >= 2) {
                    const int oh = h0 + r - 2;
                    raw_t xr[NC], ar[NC], sr;
#pragma unroll
                    for (int oc = 0; oc < NC; ++oc) {
                        xr[oc] = lds_raw(s_x + oc * PIX, (const T*)nullptr);
                        if (EPI == 1) ar[oc] = lds_raw(s_x + x_bytes + oc * PIX, (const T*)nullptr);
                    }
                    const bool sa_row = sa_ok && (oh & 1) == 0;
                    if (EPI == 2 && sa_row) sr = ldg_raw(sa_ptr + (size_t)(oh >> 1) * W2 * C);
#pragma unroll
                    for (int oc = 0; oc < NC; ++oc) {
                        if (oc == 1 && !own1) continue;  // warp-uniform
                        const float2 u = widen(xr[oc]);
                        const float2 pre = AFFINE ? ffma2(u, av, bv) : u;
                        const float2 act = act2<RELU>(pre);
                        float2 d = fmul2(Ga[oc], kf[0]);
                        d = ffma2(Ga[oc + 1], kf[1], d);
                        d = ffma2(Ga[oc + 2], kf[2], d);
#pragma unroll
                        for (int b = 0; b < 3; ++b) {
                            d = ffma2(Gb[oc + b], kf[3 + b], d);
                            dkf[b] = ffma2(act, Ga[oc + b], dkf[b]);
                            dkf[3 + b] = ffma2(act, Gb[oc + b], dkf[3 + b]);
                        }
#pragma unroll
                        for (int b = 0; b < 3; ++b) {
                            d = ffma2(Gc[oc + b], kf[6 + b], d);
                            dkf[6 + b] = ffma2(act, Gc[oc + b], dkf[6 + b]);
                        }
                        if (RELU) {
                            if (!act_open<RELU>(pre.x)) d.x = 0.f;
                            if (!act_open<RELU>(pre.y)) d.y = 0.f;
                        }
                        if (stats) {
                            const float2 rr = round_pair(d, (const T*)nullptr);
                            s1 = fadd2(s1, rr);
                            s2 = ffma2(rr, u, s2);
                        }
                        if (EPI == 1) d = fadd2(d, widen(ar[oc]));
                        if (EPI == 2 && sa_row && oc == oc_even) d = fadd2(d, widen(sr));
                        if (c_ok) stg_pair(o_ptr + (size_t)oc * C, d);
                    }
                    o_ptr += rowC;
                    s_x += xrow_bytes;
                }
                ++r;
            };
            while (r + 3 <= rows) { step(G0, G1, G2); step(G1, G2, G0); step(G2, G0, G1); }
            if (r < rows) { step(G0, G1, G2); if (r < rows) step(G1, G2, G0); }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_cta(empty0 + 8 * s);
        if (++s == S) { s = 0; ++n; }
    }

    // ---- CTA reduction over the consumer warps (each holds partials for the same 64 channels)
    const int nthr = ncons * 32;
    consumer_bar_sync(nthr);  // every consumer is done reading the ring before it becomes scratch
    float* red = reinterpret_cast<float*>(dwp_smem + (sbase - smem_u32(dwp_smem)));
    constexpr int NQ = 11;  // 9 taps, sum g, sum g*in
    float2* mine = reinterpret_cast<float2*>(red + (size_t)warp * NQ * CB) + lane;
#pragma unroll
    for (int t = 0; t < 9; ++t) mine[t * 32] = dkf[t];
    mine[9 * 32] = s1;
    mine[10 * 32] = s2;
    consumer_bar_sync(nthr);
    for (int e = threadIdx.x; e < NQ * CB; e += nthr) {
        const int q = e / CB, ch = e % CB;
        const int c = cbase + ch;
        if (c >= C) continue;
        float sum = 0.f;
        for (int w = 0; w < ncons; ++w) sum += red[((size_t)w * NQ + q) * CB + ch];
        if (q < 9) {
            if (dk_acc) stat_add(dk_acc, (long long)(8 - q) * C + c, (double)sum);  // order-independent (run-to-run identical)
            else atomicAdd(dk + (size_t)(8 - q) * C + c, sum);  // un-flip the tap index
        } else if (stats) {
            if (q == 9) {
                stat_add(stats, c, (double)sum);  // sum g
            } else {
                // sum g*xhat = rstd * (sum g*in - mean * sum g)
                float sg = 0.f;
                for (int w = 0; w < ncons; ++w) sg += red[((size_t)w * NQ + 9) * CB + ch];
                stat_add(stats, (long long)C + c, (double)bn_rstd[c] * ((double)sum - (double)bn_mean[c] * (double)sg));
            }
        }
    }
}

// =================================================================================================
// host side
// =================================================================================================
int make_map(CUtensorMap* map, const void* ptr, int dtype, int B, int H, int W, int C, int box_w, int box_h,
             bool nan_fill) {
    PFN_cuTensorMapEncodeTiled enc = spnet_get_tensormap_encoder();
    if (!enc) {
        spnet_set_error("dwconv3x3: cuTensorMapEncodeTiled entry point not available");
        return SPNET_ERR_CUDA;
    }
    const cuuint64_t es = dtype == SPNET_BF16 ? 2 : 4;
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)C * es, (cuuint64_t)W * C * es, (cuuint64_t)H * W * C * es};
    cuuint32_t box[4] = {(cuuint32_t)CB, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, dtype == SPNET_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4,
                     const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     nan_fill ? CU_TENSOR_MAP_FLOAT_OOB_FILL_NAN_REQUEST_ZERO_FMA : CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        spnet_set_error("dwconv3x3: cuTensorMapEncodeTiled failed (%d) for [%d,%d,%d,%d]", (int)r, B, H, W, C);
        return SPNET_ERR_CUDA;
    }
    return SPNET_OK;
}

struct Tiling { int TH, TW, NC, S, tiles_h, tiles_w, threads, chunks, grid_x; size_t smem; };

// kind 0: forward (stage = haloed input tile); 1: backward (haloed gradient + input); 2: backward + add_src tile
Tiling pick_tiling(int kind, int dtype, int B, int H, int W, int C) {
    Tiling t;
    const size_t pix = (size_t)CB * (dtype == SPNET_BF16 ? 2 : 4);
    t.TW = W > 16 ? 32 : (W > 8 ? 16 : 8);
    t.NC = kind == 0 ? 4 : 2;
    t.tiles_w = ceil_div(W, t.TW);
    t.chunks = ceil_div(C, CB);
    const int ncons = t.TW / t.NC;
    t.threads = ncons * 32;
    // resident CTAs per SM this kernel is sized for (registers: <= 64K / threads per thread)
    const int ctas = kind == 0 ? (t.TW == 32 ? 2 : (t.TW == 16 ? 4 : 6)) : (t.TW == 32 ? 1 : (t.TW == 16 ? 2 : 3));
    const size_t budget = (size_t)216 * 1024 / ctas - 1024;
    double best = 1e30;
    t.TH = 0;
    const int cands[] = {2, 3, 4, 6, 8, 12, 16};
    for (int th : cands) {
        if (th > H && th != 2) continue;
        const size_t stage = (size_t)(th + 2) * (t.TW + 2) * pix + (kind ? (size_t)th * t.TW * pix * (kind == 2 ? 2 : 1) : 0);
        int S = (int)(budget / stage);
        if (S > MAX_STAGES) S = MAX_STAGES;
        if (S < 2) continue;
        const long long n = (long long)B * ceil_div(H, th) * t.tiles_w;
        long long gx = ((long long)spnet_num_sms() * ctas) / t.chunks;
        if (gx < 1) gx = 1;
        if (gx > n) gx = n;
        const long long per = (n + gx - 1) / gx;
        if (S > per + 1) S = (int)per + 1;
        // rows a CTA walks (+2 halo rows and ~1 row of per-tile overhead each), scaled by the share of an SM it gets
        const double waves = (double)ceil_div(gx * t.chunks, (long long)spnet_num_sms() * ctas);
        const double cost = (double)per * ((th < H ? th : H) + 3.0) * waves;
        if (cost < best) {
            best = cost;
            t.TH = th; t.S = S; t.tiles_h = ceil_div(H, th); t.grid_x = (int)gx;
            t.smem = stage * S + 128;
        }
    }
    return t;
}

template <typename T, int NC, bool AF, int RL>
int launch_fwd_inst(const CUtensorMap& tm, const float* k, const float* a, const float* b, T* y, int B, int H, int W,
                    int C, const Tiling& t, cudaStream_t stream) {
    auto kern = dw3x3_fwd_packed_kernel<T, NC, AF, RL>;
    static bool configured[64] = {};
    if (spnet_first_use_on_device(configured)) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        if (e != cudaSuccess) {
            spnet_set_error("dwconv3x3_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return SPNET_ERR_CUDA;
        }
    }
    kern<<<dim3(t.grid_x, t.chunks), t.threads, t.smem, stream>>>(tm, k, a, b, y, B, H, W, C, t.TH, t.TW, t.tiles_h,
                                                                  t.tiles_w, t.S);
    return spnet_check_launch("dw3x3_fwd");
}

template <typename T>
int launch_fwd(const void* in, const float* k, const float* a, const float* b, int relu, void* out, int dtype, int B,
               int H, int W, int C, cudaStream_t stream) {
    const Tiling t = pick_tiling(0, dtype, B, H, W, C);
    SPNET_REQUIRE(t.TH > 0, "dwconv3x3_fwd: no tile fits shared memory");
    CUtensorMap tm;
    int rc = make_map(&tm, in, dtype, B, H, W, C, t.TW + 2, t.TH + 2, a && relu);
    if (rc) return rc;
    T* y = reinterpret_cast<T*>(out);
    if (a && relu == 2) return launch_fwd_inst<T, 4, true, 2>(tm, k, a, b, y, B, H, W, C, t, stream);
    if (a && relu) return launch_fwd_inst<T, 4, true, 1>(tm, k, a, b, y, B, H, W, C, t, stream);
    if (a) return launch_fwd_inst<T, 4, true, 0>(tm, k, a, b, y, B, H, W, C, t, stream);
    if (relu == 2) return launch_fwd_inst<T, 4, false, 2>(tm, k, a, b, y, B, H, W, C, t, stream);
    if (relu) return launch_fwd_inst<T, 4, false, 1>(tm, k, a, b, y, B, H, W, C, t, stream);
    return launch_fwd_inst<T, 4, false, 0>(tm, k, a, b, y, B, H, W, C, t, stream);
}

template <typename T, bool AF, int RL, int EPI>
int launch_bwd_inst(const CUtensorMap& tg, const CUtensorMap& tx, const CUtensorMap& ta, const float* k, const float* a,
                    const float* b, const float* mean, const float* rstd, long long* stats, const T* sadd, T* gin,
                    float* dk, long long* dk_acc, int B, int H, int W, int C, const Tiling& t, cudaStream_t stream) {
    auto kern = dw3x3_bwd_packed_kernel<T, AF, RL, EPI>;
    static bool configured[64] = {};
    if (spnet_first_use_on_device(configured)) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        if (e != cudaSuccess) {
            spnet_set_error("dwconv3x3_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return SPNET_ERR_CUDA;
        }
    }
    kern<<<dim3(t.grid_x, t.chunks), t.threads, t.smem, stream>>>(tg, tx, ta, k, a, b, mean, rstd, stats, sadd, gin, dk,
                                                                  dk_acc, B, H, W, C, t.TH, t.TW, t.tiles_h, t.tiles_w, t.S);
    return spnet_check_launch("dw3x3_bwd_fused");
}

template <typename T>
int launch_bwd(const void* gout, const void* in, const float* k, const float* a, const float* b, int relu,
               const float* mean, const float* rstd, long long* stats, const void* add_src, const void* add_strided,
               void* gin, float* dk, long long* dk_acc, int dtype, int B, int H, int W, int C, cudaStream_t stream) {
    const int epi = add_src ? 1 : (add_strided ? 2 : 0);
    Tiling t = pick_tiling(epi == 1 ? 2 : 1, dtype, B, H, W, C);
    SPNET_REQUIRE(t.TH > 0, "dwconv3x3_bwd: no tile fits shared memory");
    const size_t red_bytes = (size_t)(t.TW / 2) * 11 * CB * 4 + 128;
    if (t.smem < red_bytes) t.smem = red_bytes;
    CUtensorMap tg, tx, ta;
    int rc = make_map(&tg, gout, dtype, B, H, W, C, t.TW + 2, t.TH + 2, false);
    if (rc) return rc;
    rc = make_map(&tx, in, dtype, B, H, W, C, t.TW, t.TH, false);
    if (rc) return rc;
    rc = make_map(&ta, add_src ? add_src : in, dtype, B, H, W, C, t.TW, t.TH, false);
    if (rc) return rc;
    const T* sadd = reinterpret_cast<const T*>(add_strided);
    T* y = reinterpret_cast<T*>(gin);
#define DWB(AF, RL)                                                                                                    \
    do {                                                                                                               \
        if (epi == 1) return launch_bwd_inst<T, AF, RL, 1>(tg, tx, ta, k, a, b, mean, rstd, stats, sadd, y, dk, dk_acc, B, H, W, C, t, stream); \
        if (epi == 2) return launch_bwd_inst<T, AF, RL, 2>(tg, tx, ta, k, a, b, mean, rstd, stats, sadd, y, dk, dk_acc, B, H, W, C, t, stream); \
        return launch_bwd_inst<T, AF, RL, 0>(tg, tx, ta, k, a, b, mean, rstd, stats, sadd, y, dk, dk_acc, B, H, W, C, t, stream);   \
    } while (0)
    if (a && relu == 2) DWB(true, 2);
    if (a && relu) DWB(true, 1);
    if (a) DWB(true, 0);
    if (relu == 2) DWB(false, 2);
    if (relu) DWB(false, 1);
    DWB(false, 0);
#undef DWB
}

int check_args(const char* who, const void* in, const void* out, int dtype, int B, int H, int W, int C) {
    SPNET_REQUIRE(in && out, "%s: null pointer", who);
    SPNET_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0, "%s: bad shape", who);
    const int V = dtype == SPNET_BF16 ? 8 : 4;
    SPNET_REQUIRE(C % V == 0, "%s: C=%d must be a multiple of %d", who, C, V);
    return SPNET_OK;
}

}  // namespace

extern "C" {

// out = dw3x3(act(in)),  act(v) = relu?(in_a*v + in_b)   (in_a/in_b nullable, fp32 [C]; relu: 0 none, 1 ReLU, 2 ReLU6)
// k: [3,3,C] fp32 (keras depthwise_kernel (3,3,C,1) flattened)
int spnet_dwconv3x3_fwd(const void* in, const float* k, const float* in_a, const float* in_b, int relu, void* out,
                        int dtype, int B, int H, int W, int C, cudaStream_t stream) {
    int rc = check_args("dwconv3x3_fwd", in, out, dtype, B, H, W, C);
    if (rc) return rc;
    SPNET_REQUIRE(k && ((in_a == nullptr) == (in_b == nullptr)) && relu >= 0 && relu <= 2, "dwconv3x3_fwd: bad weight/affine pointers or relu code");
    SPNET_DISPATCH_DTYPE(dtype, return launch_fwd<T>(in, k, in_a, in_b, relu, out, dtype, B, H, W, C, stream));
}

// Fused backward (see dw3x3_bwd_packed_kernel): gin, dk (+=) and optional BatchNorm-backward sums.
//   in          : the tensor the forward depthwise read (raw), transformed on load by
//                 act(v) = relu?(in_a*v+in_b)
//   stats       : nullable accumulators, 2*C entries; += (sum gin, sum gin*xhat) with xhat = (in-bn_mean)*bn_rstd
//   dk_acc      : nullable accumulators, 9*C entries: the kernel-gradient partial sums of the CTAs go there (order-
//                 independent, spnet_acc_to_f32 adds them into dk) instead of fp32 atomics on dk
//   add_src / add_strided : optional residual-path gradients added to gin (at most one of them)
int spnet_dwconv3x3_bwd_fused(const void* gout, const void* in, const float* k, const float* in_a, const float* in_b,
                              int relu, const float* bn_mean, const float* bn_rstd, long long* stats, const void* add_src,
                              const void* add_strided, void* gin, float* dk, long long* dk_acc, int dtype, int B, int H,
                              int W, int C, cudaStream_t stream) {
    int rc = check_args("dwconv3x3_bwd_fused", gout, gin, dtype, B, H, W, C);
    if (rc) return rc;
    SPNET_REQUIRE(in && k && dk && ((in_a == nullptr) == (in_b == nullptr)) && relu >= 0 && relu <= 2, "dwconv3x3_bwd_fused: bad pointers or relu code");
    SPNET_REQUIRE(!stats || (bn_mean && bn_rstd), "dwconv3x3_bwd_fused: stats need bn_mean / bn_rstd");
    SPNET_REQUIRE(!(add_src && add_strided), "dwconv3x3_bwd_fused: add_src and add_strided are exclusive");
    SPNET_DISPATCH_DTYPE(dtype, return launch_bwd<T>(gout, in, k, in_a, in_b, relu, bn_mean, bn_rstd, stats, add_src,
                                                     add_strided, gin, dk, dk_acc, dtype, B, H, W, C, stream));
}

}  // extern "C"
