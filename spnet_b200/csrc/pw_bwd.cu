// Backward of a pointwise (1x1) convolution whose output feeds a BatchNorm, in one pass over the tensors:
//
//     dz  = a * (g - c1 - xhat * c2)         (BatchNorm backward, per channel; bn.cu bn_bwd_dz_kernel)
//     gA  = dz . W^T                         (data gradient, [M, cin] bf16, stored)
//     gW += t^T . dz                         (weight gradient, [cin, cout] fp32)
//
// The unfused route writes dz to global memory and reads it back twice (weight-gradient GEMM, data-gradient GEMM).
// Here each CTA loads g, z and the layer input t of a 128-pixel tile once, forms dz in shared memory, runs both
// MMAs from that one tile and writes only gA. The weights (<= 32 KB) stay in shared memory for the whole kernel,
// and the weight gradient of all of a CTA's tiles accumulates in one TMEM accumulator that is drained once, at the
// end. Serves Xception's block-2 pointwise layers (cout = 128, cin = 64 or 128: block2_sepconv1, block2_sepconv2
// and the strided residual conv2d_4). A 128 -> 256 layer needs a 160 KB tile next to 64 KB of weights, which
// leaves no room for a second stage; those layers keep the unfused route.
//
// Persistent, warp-specialised, one CTA per SM:
//   warp 0        TMA producer : weights once; per tile t + g (2-stage ring) and z (its own ring, ZST deep)
//   warp 1        MMA issuer   : gW^T += dz^T t (M = cout, N = cin, K = 128 pixels) into the resident accumulator,
//                                then gA = dz W^T (M = 128 pixels, N = cin, K = cout) into one of two accumulators
//   warps 2..9    transform    : dz = fma(g, A, fma(z, Bz, D)) rounded to bf16, in place over g in the swizzled
//                                layout; frees the z stage
//   warps 10..13  epilogue     : gA accumulator -> bf16 -> staging box -> TMA store (rows >= M clipped); at the end
//                                the weight-gradient accumulator -> reduce-add into gW, or a per-CTA slab
//
// Every tile is a 128-row box of 64-channel SWIZZLE_128B blocks (16 KB each): row r, 16-byte chunk j of a block
// holds channels 8 * (j ^ (r & 7)) .. +7. The same bytes are the K-major A operand of the data gradient (rows =
// pixels, K = channels) and the MN-major operands of the weight gradient (K = pixels, 64-channel atoms 16 KB apart).
#include "tcgen05.cuh"

namespace {

constexpr int kRows = 128;                  // pixel rows per tile = UMMA M of the data gradient
constexpr uint32_t kBox = kRows * 128;      // one 64-channel block of a tile
constexpr int kCout = 128;                  // = UMMA M of the weight gradient
constexpr int kUmmaK = 16;
constexpr int kNG = kCout / 64;             // channel blocks of g, z, dz
constexpr int kXWarps = 8;                  // transform warps
constexpr int kEWarps = 4;                  // epilogue warps, one per TMEM lane quadrant
constexpr int kPwThreads = 64 + 32 * (kXWarps + kEWarps);

template <int CIN>
struct PwCfg {
    static constexpr int NT = CIN / 64;                         // channel blocks of t
    static constexpr int ZST = CIN == 64 ? 2 : 1;               // z ring depth (what shared memory leaves)
    static constexpr uint32_t TG_BYTES = (NT + kNG) * kBox;     // one stage: t blocks, then g (-> dz) blocks
    static constexpr uint32_t Z_BYTES = kNG * kBox;
    static constexpr uint32_t W_BYTES = kNG * CIN * 128;        // W as K-major B: kNG blocks of CIN rows x 64
    static constexpr uint32_t OUT_BYTES = kEWarps * 2 * 2048;   // two 32 x 32 bf16 staging boxes per epilogue warp
    static constexpr size_t SMEM = 1024 + 2 * TG_BYTES + ZST * Z_BYTES + W_BYTES + OUT_BYTES;
    static constexpr uint32_t TMEM_COLS = CIN == 64 ? 256 : 512;  // 2 x CIN (gA) + CIN (gW^T), power of two
};

enum { TG_FULL = 0, TG_EMPTY = 2, Z_FULL = 4, Z_EMPTY = 6, DZ_READY = 8, ACC_FULL = 10, ACC_EMPTY = 12, W_FULL = 14,
       WACC_FULL = 15, N_BARS = 16 };

// SWIZZLE_128B shared-memory descriptor (sm_100 version 1), SBO = 1024 B between 8-row groups
__device__ __forceinline__ uint64_t sw128_desc(uint32_t addr, uint32_t lbo) {
    const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    const uint32_t lo = ((lbo >> 4) << 16) | ((addr & 0x3ffffu) >> 4);
    return ((uint64_t)hi << 32) | lo;
}

template <int CIN>
__global__ void __launch_bounds__(kPwThreads, 1) pw_bwd_bn_kernel(
    const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmZ,
    const __grid_constant__ CUtensorMap tmT, const __grid_constant__ CUtensorMap tmW,
    const __grid_constant__ CUtensorMap tmGA, const float* __restrict__ a, const float* __restrict__ mean,
    const float* __restrict__ rstd, const float* __restrict__ c1, const float* __restrict__ c2, float* __restrict__ gW,
    float* __restrict__ slabs, int M, int n_tiles) {
    using Cfg = PwCfg<CIN>;
    constexpr int NT = Cfg::NT, ZST = Cfg::ZST;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t bars[N_BARS];
    __shared__ uint32_t tmem_base_holder;
    const uint32_t tg0 = smem_u32(smem);
    const uint32_t z0 = tg0 + 2 * Cfg::TG_BYTES;
    const uint32_t w0 = z0 + ZST * Cfg::Z_BYTES;
    const uint32_t out0 = w0 + Cfg::W_BYTES;
    const uint32_t bar0 = smem_u32(&bars[0]);
    auto bar = [&](int b) { return bar0 + 8u * (uint32_t)b; };
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar(TG_FULL + s), 1);
            mbar_init(bar(TG_EMPTY + s), 1);
            mbar_init(bar(Z_FULL + s), 1);
            mbar_init(bar(Z_EMPTY + s), kXWarps);
            mbar_init(bar(DZ_READY + s), kXWarps);
            mbar_init(bar(ACC_FULL + s), 1);
            mbar_init(bar(ACC_EMPTY + s), kEWarps);
        }
        mbar_init(bar(W_FULL), 1);
        mbar_init(bar(WACC_FULL), 1);
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc(smem_u32(&tmem_base_holder), Cfg::TMEM_COLS);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_holder;
    const uint32_t tmem_wacc = tmem_base + 2 * CIN;

    if (warp == 0) {
        // ---------------- TMA producer ----------------
        const uint32_t issuer = elect_one();
        if (issuer) {
            mbar_expect_tx(bar(W_FULL), Cfg::W_BYTES);
#pragma unroll
            for (int kb = 0; kb < kNG; ++kb) tma_load_2d(w0 + kb * (CIN * 128), &tmW, bar(W_FULL), kb * 64, 0);
        }
        uint32_t i = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++i) {
            const int m0 = tile * kRows;
            const uint32_t s = i & 1u, ph = (i >> 1) & 1u;
            mbar_wait(bar(TG_EMPTY + s), ph ^ 1u);
            if (issuer) {
                const uint32_t b = bar(TG_FULL + s), dst = tg0 + s * Cfg::TG_BYTES;
                mbar_expect_tx(b, Cfg::TG_BYTES);
                // rows >= M of t, g and z are zero-filled by the TMA unit
#pragma unroll
                for (int j = 0; j < NT; ++j) tma_load_2d(dst + j * kBox, &tmT, b, j * 64, m0);
#pragma unroll
                for (int j = 0; j < kNG; ++j) tma_load_2d(dst + (NT + j) * kBox, &tmG, b, j * 64, m0);
            }
            __syncwarp();
            const uint32_t zs = i % ZST, zph = (i / ZST) & 1u;
            mbar_wait(bar(Z_EMPTY + zs), zph ^ 1u);
            if (issuer) {
                const uint32_t b = bar(Z_FULL + zs), dst = z0 + zs * Cfg::Z_BYTES;
                mbar_expect_tx(b, Cfg::Z_BYTES);
#pragma unroll
                for (int j = 0; j < kNG; ++j) tma_load_2d(dst + j * kBox, &tmZ, b, j * 64, m0);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer ----------------
        // instruction descriptors: fp32 accumulate, bf16 x bf16, N = CIN, M = 128; the weight gradient reads both
        // operands MN-major
        constexpr uint32_t idesc_dg = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(CIN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        constexpr uint32_t idesc_wg = idesc_dg | (1u << 15) | (1u << 16);
        const uint32_t leader = elect_one();
        mbar_wait(bar(W_FULL), 0u);
        uint32_t i = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++i) {
            const uint32_t s = i & 1u, ph = (i >> 1) & 1u, as = i & 1u;
            const uint32_t tb = tg0 + s * Cfg::TG_BYTES, gb = tb + NT * kBox;
            mbar_wait(bar(DZ_READY + s), ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (leader) {
                // gW^T[co, ci] += sum over the tile's pixels p of dz[p, co] * t[p, ci]: 16 pixels (2 KB) per MMA
#pragma unroll
                for (int k = 0; k < kRows / kUmmaK; ++k)
                    umma_bf16(tmem_wacc, sw128_desc(gb + k * 2048, kBox), sw128_desc(tb + k * 2048, kBox), idesc_wg,
                              (i > 0 || k > 0) ? 1u : 0u, 1u);
            }
            __syncwarp();
            mbar_wait(bar(ACC_EMPTY + as), ((i >> 1) & 1u) ^ 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (leader) {
                // gA = dz W^T, K = cout in the order of the unfused GEMM: channel blocks, 16 channels (32 B) per MMA
#pragma unroll
                for (int kb = 0; kb < kNG; ++kb)
#pragma unroll
                    for (int k = 0; k < 64 / kUmmaK; ++k)
                        umma_bf16(tmem_base + as * CIN, sw128_desc(gb + kb * kBox + k * 32, 0),
                                  sw128_desc(w0 + kb * (CIN * 128) + k * 32, 0), idesc_dg, (kb > 0 || k > 0) ? 1u : 0u, 1u);
                umma_commit(bar(ACC_FULL + as), 1u);
                umma_commit(bar(TG_EMPTY + s), 1u);  // t and dz of this stage are consumed when these MMAs retire
            }
            __syncwarp();
        }
        if (leader && i > 0) umma_commit(bar(WACC_FULL), 1u);
        __syncwarp();
    } else if (warp < 2 + kXWarps) {
        // ---------------- transform: dz over g ----------------
        // thread xt always handles 16-byte chunk (xt & 7) of rows (xt >> 3) + 32 u, so its channels are fixed:
        // block b, 8 * ((xt & 7) ^ ((xt >> 3) & 7)) + 0..7. Coefficients as bn_bwd_dz_kernel computes them.
        const int xt = threadIdx.x - 64;
        const int cq = 8 * ((xt & 7) ^ ((xt >> 3) & 7));
        float cA[kNG][8], cB[kNG][8], cD[kNG][8];
#pragma unroll
        for (int b = 0; b < kNG; ++b)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = b * 64 + cq + j;
                const float A = a[c], mu = mean[c], rs = rstd[c], k1 = c1[c], k2 = c2[c];
                const float kx = rs * k2;
                cA[b][j] = A;
                cB[b][j] = -A * kx;
                cD[b][j] = A * (kx * mu - k1);
            }
        const uint32_t row_off = (uint32_t)(xt >> 3) * 128u + (uint32_t)(xt & 7) * 16u;
        uint32_t i = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++i) {
            const uint32_t s = i & 1u, ph = (i >> 1) & 1u;
            const uint32_t zs = i % ZST, zph = (i / ZST) & 1u;
            const uint32_t gb = tg0 + s * Cfg::TG_BYTES + NT * kBox, zb = z0 + zs * Cfg::Z_BYTES;
            mbar_wait(bar(TG_FULL + s), ph);
            mbar_wait(bar(Z_FULL + zs), zph);
            // Rows >= M arrive as zeros, so their dz is D, not 0. They add nothing to gW only because t's rows >= M
            // are zero-filled the same way, and their gA rows are clipped by the store: keep all three maps alike.
#pragma unroll
            for (int b = 0; b < kNG; ++b)
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t off = (uint32_t)b * kBox + (uint32_t)u * 4096u + row_off;
                    uint32_t gv[4], zv[4];
                    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(gv[0]), "=r"(gv[1]), "=r"(gv[2]), "=r"(gv[3]) : "r"(gb + off) : "memory");
                    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(zv[0]), "=r"(zv[1]), "=r"(zv[2]), "=r"(zv[3]) : "r"(zb + off) : "memory");
                    uint32_t dv[4];
#pragma unroll
                    for (int w = 0; w < 4; ++w) {
                        const float g0 = __uint_as_float(gv[w] << 16), g1 = __uint_as_float(gv[w] & 0xffff0000u);
                        const float z0f = __uint_as_float(zv[w] << 16), z1f = __uint_as_float(zv[w] & 0xffff0000u);
                        dv[w] = pack_bf16x2(fmaf(g0, cA[b][2 * w], fmaf(z0f, cB[b][2 * w], cD[b][2 * w])),
                                            fmaf(g1, cA[b][2 * w + 1], fmaf(z1f, cB[b][2 * w + 1], cD[b][2 * w + 1])));
                    }
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(gb + off), "r"(dv[0]), "r"(dv[1]),
                                 "r"(dv[2]), "r"(dv[3])
                                 : "memory");
                }
            // dz written by the generic proxy is read by tcgen05.mma (async proxy)
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(bar(Z_EMPTY + zs));
                mbar_arrive(bar(DZ_READY + s));
            }
            __syncwarp();
        }
    } else {
        // ---------------- epilogue ----------------
        const uint32_t e_leader = elect_one();
        const int q = warp & 3;                    // TMEM lane quadrant this warp may access
        const int ew = warp - 2 - kXWarps;         // 0..3
        uint32_t sbox = 0, i = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++i) {
            const uint32_t as = i & 1u;
            const int row0 = tile * kRows + q * 32;
            mbar_wait(bar(ACC_FULL + as), (i >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
            for (int c = 0; c < CIN / 32; ++c) {
                uint32_t v[32];
                tmem_ld32(tmem_base + as * CIN + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
                uint32_t packed[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) packed[j] = pack_bf16x2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
                if (row0 < M) {  // warp-uniform; rows >= M inside the box are clipped by the TMA unit
                    const uint32_t stg = out0 + ((uint32_t)ew * 2u + sbox) * 2048u;
                    if (e_leader) tma_store_wait_read<1>();  // this box was read out
                    __syncwarp();
                    stage_box_row_sw64(stg, (uint32_t)lane, packed);
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (e_leader) {
                        tma_store_2d(&tmGA, stg, c * 32, row0);
                        tma_store_commit();
                    }
                    sbox ^= 1u;
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (e_leader) mbar_arrive(bar(ACC_EMPTY + as));
        }
        if (i > 0) {
            // weight gradient of all of this CTA's tiles: lane = output channel co, columns = input channels ci
            mbar_wait(bar(WACC_FULL), 0u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int co = q * 32 + lane;
            float* dst = slabs ? slabs + (size_t)blockIdx.x * CIN * kCout : gW;
#pragma unroll 1
            for (int c = 0; c < CIN / 32; ++c) {
                uint32_t v[32];
                tmem_ld32(tmem_wacc + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float* p = dst + (size_t)(c * 32 + j) * kCout + co;  // a warp writes 32 consecutive floats
                    if (slabs) *p = __uint_as_float(v[j]);
                    else atomicAdd(p, __uint_as_float(v[j]));
                }
            }
        }
        if (e_leader) tma_store_wait_read<0>();  // staging may not die under a store
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

int pw_map(CUtensorMap* map, const void* ptr, long long rows, int cols, int box_cols, int box_rows, bool bf16_out) {
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows}, strides[1] = {(cuuint64_t)cols * 2};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    return spnet_encode_tiled(map, "pw_bwd_bn", CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ptr, dims, strides, box,
                              bf16_out ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                              bf16_out ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

template <int CIN>
int launch_pw_bwd(const CUtensorMap& tg, const CUtensorMap& tz, const CUtensorMap& tt, const CUtensorMap& tw,
                  const CUtensorMap& tga, const float* a, const float* mean, const float* rstd, const float* c1,
                  const float* c2, float* gW, float* slabs, int M, int n_tiles, int grid, cudaStream_t stream) {
    auto kern = pw_bwd_bn_kernel<CIN>;
    static bool configured[64] = {};
    const int rc = spnet_smem_optin(configured, kern, PwCfg<CIN>::SMEM, "pw_bwd_bn");
    if (rc) return rc;
    kern<<<grid, kPwThreads, PwCfg<CIN>::SMEM, stream>>>(tg, tz, tt, tw, tga, a, mean, rstd, c1, c2, gW, slabs, M, n_tiles);
    return spnet_check_launch("pw_bwd_bn");
}

}  // namespace

extern "C" {

int spnet_pw_bwd_bn(const void* g, const void* z, const void* t, const void* W, const float* a, const float* save_mean,
                    const float* save_rstd, const float* c1, const float* c2, void* gA, float* gW, float* slabs, int nslabs,
                    int M, int cin, int cout, cudaStream_t stream) {
    SPNET_REQUIRE(g && z && t && W && a && save_mean && save_rstd && c1 && c2 && gA && gW, "pw_bwd_bn: null pointer");
    SPNET_REQUIRE(M > 0 && cout == kCout && (cin == 64 || cin == 128), "pw_bwd_bn: unsupported shape M=%d %d -> %d", M,
                  cin, cout);
    SPNET_REQUIRE(((uintptr_t)g | (uintptr_t)z | (uintptr_t)t | (uintptr_t)W | (uintptr_t)gA) % 16 == 0,
                  "pw_bwd_bn: pointers must be 16-byte aligned");
    CUtensorMap tg, tz, tt, tw, tga;
    int rc = pw_map(&tg, g, M, cout, 64, kRows, false);
    if (!rc) rc = pw_map(&tz, z, M, cout, 64, kRows, false);
    if (!rc) rc = pw_map(&tt, t, M, cin, 64, kRows, false);
    if (!rc) rc = pw_map(&tw, W, cin, cout, 64, cin, false);  // W^T as the K-major B operand: rows = ci, K = co
    if (!rc) rc = pw_map(&tga, gA, M, cin, 32, 32, true);
    if (rc) return rc;
    const int n_tiles = (M + kRows - 1) / kRows;
    // slabs: one CTA per slab, a fixed set of tiles each (tile = CTA, CTA + grid, ...), so the sum is bit-reproducible
    SPNET_REQUIRE(!slabs || (nslabs >= 1 && nslabs <= n_tiles), "pw_bwd_bn: nslabs must be in [1, %d]", n_tiles);
    const int grid = slabs ? nslabs : (n_tiles < spnet_num_sms() ? n_tiles : spnet_num_sms());
    if (cin == 64) return launch_pw_bwd<64>(tg, tz, tt, tw, tga, a, save_mean, save_rstd, c1, c2, gW, slabs, M, n_tiles, grid, stream);
    return launch_pw_bwd<128>(tg, tz, tt, tw, tga, a, save_mean, save_rstd, c1, c2, gW, slabs, M, n_tiles, grid, stream);
}

}  // extern "C"
