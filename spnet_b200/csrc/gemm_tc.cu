// bf16 GEMM on the 5th-generation tensor cores: TMA (cp.async.bulk.tensor) feeds a
// shared-memory ring, one elected thread issues tcgen05.mma with the fp32 accumulator
// in TMEM, eight warps drain it with tcgen05.ld. Serves the pointwise 1x1 convolutions
// of SeparableConv2D, the strided 1x1 residual convolutions, block1_conv2 (as an
// im2col GEMM) and the Dense head of the reference model (spnet/models.py:359,388),
// forward, data-gradient and weight-gradient, and - as implicit GEMM, template parameter
// CONV - the k x k stride-1 convolutions of the InceptionResNetV2 backbone
// (spnet/models.py:18,357-359) and block1_conv2's data gradient:
//
//     D[M,N] (op)= A[M,K] * B[K,N]
//
// Each operand is described by its memory order relative to the reduction dim K:
//   K-major  : element (r, k) at  ptr[r*ld + k]   (activations in forward/dgrad)
//   MN-major : element (r, k) at  ptr[k*ld + r]   (keras (Cin,Cout) weights in forward,
//                                                  both operands in weight-gradient)
// so no transposed weight copies are needed. Out-of-range rows/cols/k are zero-filled
// by TMA, which makes ragged M, N (728 = 5*128+88) and K (728 = 11*64+24) exact.
//
// Epilogue modes: store bf16, store fp32, atomic-add fp32 (split-K); optional fused
// per-column sum / sum-of-squares (BatchNorm batch statistics) accumulated in fp64.
#include "tma.cuh"

#ifdef SPNET_GEMM_TRACE
// diagnostic build only (tests/micro/gemm_trace.py): per-CTA cycle stamps of the kernel's phases
__device__ unsigned long long g_gemm_trace[256 * 16];
#define TRACE(slot) do { g_gemm_trace[blockIdx.x * 16 + (slot)] = (unsigned long long)clock64(); } while (0)
#define TRACE_G(slot) do { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); g_gemm_trace[blockIdx.x * 16 + (slot)] = t_; } while (0)
#else
#define TRACE(slot) do { } while (0)
#define TRACE_G(slot) do { } while (0)
#endif

namespace {

constexpr int BM = 128;          // UMMA M (cta_group::1)
constexpr int BK = 64;           // 64 bf16 = 128 B = one SWIZZLE_128B row
constexpr int UMMA_K = 16;
constexpr int kEpiWarps = 8;    // two per TMEM lane quadrant, each draining half of the columns
// ONE producer warp. (Several were tried for the convolution modes: striping k-blocks over four warps is unsafe -
// an mbarrier parity wait tells adjacent phases apart, not a producer that ran two ring rounds ahead; it passed the
// unit tests and trapped at full InceptionResNetV2 size - and striping the boxes of a k-block was not faster once
// the issue path ran on the uniform datapath.)
constexpr int kThreads = 64 + 32 * kEpiWarps;  // TMA warp, MMA warp, epilogue warps

enum { OUT_BF16 = 0, OUT_F32 = 1, OUT_ATOMIC_F32 = 2, OUT_SLAB_F32 = 3 };

struct GemmEpi {
    void* out;
    long long ldc;
    int mode;
    int slab_rows;     // unused (kept for layout); OUT_SLAB_F32 stores through a 3-D output map {N, M, split}
    long long* colstats;  // order-independent accumulators (common.cuh stat_add), 2*N entries (sum, sumsq), or nullptr
};

// Implicit-GEMM convolution on the same kernel (template parameter CONV). The activation operand is a 4-D
// NHWC tensor map; a "row" of the GEMM is an output pixel and the rows of one tile are a
// (2^lw x 2^lh x images) box of pixels, so the A tile of filter tap (ky, kx) is ONE TMA box at the tile's
// origin shifted by the tap (out-of-image pixels and channels past Cin are zero-filled by the TMA unit:
// 'same' padding and ragged channel counts cost nothing, and there is no im2col buffer).
//   CONV 1 (forward / data gradient): k-block = (tap, 64-channel block); 128-pixel tiles.
//   CONV 2 (weight gradient)        : one unit = one tap; k-blocks = 64-pixel boxes of the batch, both
//                                     operands MN-major; output rows are offset by tap * Cin.
struct ConvGeom {
    int lw, lh;            // log2 of the pixel box's width / height (images per box = rows >> (lw + lh))
    int tiles_w, tiles_h;  // pixel boxes per image along W / H
    int OW, OH, NB;        // extent of the output pixels (CONV 1: masks the fused statistics)
    int KW, cin_blocks, ntaps;
    int pt, pl, sign;      // A-box origin = pixel + sign * (tap - pad)
    int b_tap_stride;      // rows between taps in the 2-D weight map
    int b_tap_on_k;        // 1: taps advance B's K coordinate (forward), 0: its N coordinate (data gradient)
};

// The MMA warp runs its loop CONVERGED: every lane computes the (warp-uniform) descriptors and the instruction
// itself is guarded by a predicate that is true in lane 0 only. Inside an `if (lane == 0)` block ptxas cannot
// keep the descriptors in uniform registers and wraps every tcgen05.mma in an ELECT / 5 x R2UR.BROADCAST /
// BRA.U.ANY loop: ~110 dependent instructions (~600 cycles) per k-block, more than the MMAs of a narrow tile.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
// one lane of a converged warp (always the same one), in a form the compiler recognises as "one thread"
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t leader;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));
    return leader;
}
__device__ __forceinline__ void umma_commit(uint32_t bar, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptors (sm_100 version 1, SWIZZLE_128B) are assembled in the MMA warp:
//  K-major : rows of 128 B, 8-row groups 1024 B apart (SBO); LBO unused.
//  MN-major: atoms of 64 elements (128 B) x 8 k-rows; SBO = distance between 8-k-row
//            groups (1024 B), LBO = distance between 64-element atoms along M/N.

__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                               uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster "
        "[%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t cta_mask, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %2, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}" ::"r"(bar),
        "h"(cta_mask), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_cta_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void epi_bar_sync() {  // named barrier 1: the four epilogue warps only
    asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
}

// Persistent, warp-specialised kernel. One CTA per SM walks work units (split, m-tile, n-tile):
//   warp 0      TMA producer   : fills the STAGES-deep smem ring
//   warp 1      MMA issuer     : one elected lane issues tcgen05.mma into one of TWO TMEM accumulators
//   warps 2..9  epilogue       : drain the other accumulator (tcgen05.ld -> convert -> staging box -> TMA store,
//                                fused BatchNorm column statistics) while the next unit's MMAs run
// CL = 2: CTA pairs (thread-block cluster of 2 along M). Both CTAs of a pair work on the same
// n-tile and k-range with adjacent m-tiles; each loads its own A tile and HALF of the shared B tile,
// multicast by TMA into both CTAs' shared memory, so the pair reads B from L2 once.
// BRES (CONV 1, one n-tile, few k-blocks): the whole B operand (the convolution's weights, <= 72 KB) is loaded into
// shared memory ONCE per CTA and stays there for all of its pixel tiles; the ring then carries A boxes only. Narrow
// convolutions are bound by L2 -> SM delivery (a 128x64x64 k-block is 0.09 us of MMA), and re-fetching the weights for
// every tile was a third of that traffic.
template <int BN, bool A_MN, bool B_MN, int STAGES, int CL, int CONV, bool BRES = false>
__global__ void __launch_bounds__(kThreads, 1) gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                              const __grid_constant__ CUtensorMap tmB,
                                                              const __grid_constant__ CUtensorMap tmD, GemmEpi epi,
                                                              int M, int N, int K, int kb_per_split, int tiles_m,
                                                              int tiles_n, int n_units, ConvGeom cg) {
    static_assert(CONV == 0 || CL == 1, "convolution modes run without CTA pairs");
    constexpr uint32_t A_BYTES = BM * BK * 2;
    constexpr uint32_t B_BYTES = BN * BK * 2;
    static_assert(!BRES || (CONV == 1 && CL == 1), "resident B is a mode of the forward-type implicit convolution");
    constexpr uint32_t STAGE_BYTES = A_BYTES + (BRES ? 0u : B_BYTES);
    // TMA boxes per k-block issued by THIS CTA: A is one 128-row box (K-major) or BM/64 atoms (MN-major);
    // B one box (K-major) or BN/64 atoms (MN-major), of which a CTA of a pair issues 1/CL (multicast)
    constexpr int NA_BOX = (A_MN || CONV == 2) ? BM / 64 : 1;
    constexpr int NB_BOX = (B_MN || CONV == 2) ? BN / 64 / CL : 1;
    constexpr int N_BOX = NA_BOX + NB_BOX;
    constexpr uint32_t A_BOX_BYTES = A_BYTES / NA_BOX;
    constexpr uint32_t B_BOX_BYTES = B_BYTES / (NB_BOX * CL);  // what one of this CTA's B boxes lands
    extern __shared__ uint8_t smem_raw[];
    // SWIZZLE_128B tiles need 1024-byte alignment
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t bars[2 * STAGES + 5];
    __shared__ uint32_t tmem_base_holder;
    __shared__ float sstat[2][2][4][BN];  // [accumulator parity][sum | sumsq][lane quadrant][column]

    // warp index through a shuffle: the compiler then KNOWS it is warp-uniform, keeps the role branches and everything
    // derived from uniform values in the uniform datapath (no ELECT / R2UR.BROADCAST loops around TMA and MMA issue)
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    // output staging for the TMA-store epilogue: SD boxes of 32 rows x 64 bytes (SWIZZLE_64B) per epilogue warp;
    // two where shared memory allows (BN = 128: the HBM-bound shapes), so a box is filled while the previous
    // one is still being read out
    constexpr int SD = BN <= 128 ? 2 : 1;
    const int total_kb = (K + BK - 1) / BK;
    const uint32_t resb0 = smem_u32(smem) + STAGES * STAGE_BYTES;  // BRES: total_kb B tiles, k-block after k-block
    const uint32_t stage_out0 = resb0 + (BRES ? (uint32_t)total_kb * B_BYTES : 0u);
    uint32_t sbox = 0, last_box = 0;  // staging box this warp fills next; address of the one it filled last
    const uint32_t crank = CL > 1 ? cluster_cta_rank() : 0u;
    const int cluster_id = blockIdx.x / CL, n_clusters = gridDim.x / CL;
    constexpr uint16_t kMask = (uint16_t)((1u << CL) - 1u);
    const uint32_t full0 = smem_u32(&bars[0]);
    const uint32_t empty0 = smem_u32(&bars[STAGES]);
    const uint32_t tfull0 = smem_u32(&bars[2 * STAGES]);
    const uint32_t tempty0 = smem_u32(&bars[2 * STAGES + 2]);
    const uint32_t bres_bar = smem_u32(&bars[2 * STAGES + 4]);

    if (threadIdx.x == 0) { TRACE(0); TRACE_G(8); }
    if (threadIdx.x == 32) {  // descriptor fetch overlaps the barrier / TMEM set-up
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmD) : "memory");
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full0 + 8 * s, 1);  // one arrive.expect_tx per k-block
            mbar_init(empty0 + 8 * s, CL);  // every CTA's MMAs must have consumed the stage
        }
        mbar_init(bres_bar, 1);
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull0 + 8 * a, 1);
            mbar_init(tempty0 + 8 * a, kEpiWarps);  // one arrive per epilogue warp
        }
        mbar_fence_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_holder)),
                     "r"((uint32_t)(2 * BN))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    if (CL > 1) cluster_sync_all(); else __syncthreads();  // barrier inits visible cluster-wide
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_holder;
    if (threadIdx.x == 0) TRACE(1);
    // with CL = 2, tiles_m counts m-tile PAIRS; this CTA owns m-tile 2*pair + rank

    if (warp == 0) {
        // ---------------- TMA producer ----------------
        // every box of a k-block is issued by one elected thread, which announces the stage's bytes on its full
        // barrier (B boxes of a CTA pair land in both CTAs: each CTA expects CL x its own)
        constexpr uint32_t my_bytes = NA_BOX * A_BOX_BYTES + (BRES ? 0u : NB_BOX * B_BOX_BYTES * CL);
        uint32_t g0 = 0;  // k-blocks of the units before this one
        const uint32_t issuer = elect_one();
        if (BRES && issuer && cluster_id < n_units) {  // the weights, once: k-block kb = (tap, channel block)
            mbar_expect_tx(bres_bar, (uint32_t)total_kb * B_BYTES);
            int tp = 0, cb = 0;
            for (int kb = 0; kb < total_kb; ++kb) {
                const int kA = cb * BK;
                const int kB = kA + (cg.b_tap_on_k ? tp * cg.b_tap_stride : 0);
                const int nB = cg.b_tap_on_k ? 0 : tp * cg.b_tap_stride;
                const uint32_t dst = resb0 + (uint32_t)kb * B_BYTES;
#pragma unroll
                for (int jb = 0; jb < NB_BOX; ++jb) {
                    if (B_MN) tma_load_2d(dst + jb * (BK * 128), &tmB, bres_bar, nB + 64 * jb, kB);
                    else tma_load_2d(dst, &tmB, bres_bar, kB, nB);
                }
                if (++cb == cg.cin_blocks) { cb = 0; ++tp; }
            }
        }
        for (int unit = cluster_id; unit < n_units; unit += n_clusters) {
            const int n0 = (unit % tiles_n) * BN;
            const int mt = (unit / tiles_n) % tiles_m;
            const int m0 = (mt * CL + (int)crank) * BM;
            int rest = unit / (tiles_n * tiles_m), tap = 0;
            if (CONV == 2) { tap = rest % cg.ntaps; rest /= cg.ntaps; }
            const int kb_begin = rest * kb_per_split;
            const int nkb = min(total_kb, kb_begin + kb_per_split) - kb_begin;
            // convolution modes: the k-block -> (tap, channel block) / pixel-box decode runs on counters; a
            // division per k-block made this single-warp instruction stream (~800 cycles per k-block) the
            // bottleneck of the whole kernel
            int px0 = 0, py0 = 0, pimg = 0;  // CONV 1: origin of this tile's pixel box
            int c_cb = 0, c_kx = 0, c_ky = 0, c_tp = 0;  // CONV 1: channel block, tap of this warp's next k-block
            int c_tx = 0, c_ty = 0, c_g = 0, w_kx = 0, w_ky = 0;  // CONV 2: pixel box of the next k-block; this unit's tap
            const int kb_first = kb_begin;
            if (CONV == 1) {
                const int t2 = mt / cg.tiles_w;
                px0 = (mt - t2 * cg.tiles_w) << cg.lw;
                py0 = (t2 % cg.tiles_h) << cg.lh;
                pimg = (t2 / cg.tiles_h) << (7 - cg.lw - cg.lh);
                c_tp = kb_first / cg.cin_blocks; c_cb = kb_first - c_tp * cg.cin_blocks;
                c_ky = c_tp / cg.KW; c_kx = c_tp - c_ky * cg.KW;
            }
            if (CONV == 2) {
                const int t2 = kb_first / cg.tiles_w;
                c_tx = kb_first - t2 * cg.tiles_w; c_ty = t2 % cg.tiles_h; c_g = t2 / cg.tiles_h;
                w_ky = tap / cg.KW; w_kx = tap - w_ky * cg.KW;
            }
            for (int i = 0; i < nkb; ++i) {
                const uint32_t g = g0 + (uint32_t)i;  // running k-block index of this CTA -> ring stage and phase
                const uint32_t s = g % STAGES, ph = (g / STAGES) & 1u;
                // coordinates that depend on the mode (warp-uniform, computed before the wait)
                const int k0 = (kb_begin + i) * BK;
                int ax = 0, ay = 0, aimg = 0, bx = 0, by = 0, kA = k0, kB = k0, nB = n0;
                if (CONV == 1) {
                    kA = c_cb * BK;
                    ax = px0 + cg.sign * (c_kx - cg.pl); ay = py0 + cg.sign * (c_ky - cg.pt); aimg = pimg;
                    kB = kA + (cg.b_tap_on_k ? c_tp * cg.b_tap_stride : 0);
                    nB = n0 + (cg.b_tap_on_k ? 0 : c_tp * cg.b_tap_stride);
                    if (++c_cb == cg.cin_blocks) {  // advance to the next k-block
                        c_cb = 0; ++c_tp;
                        if (++c_kx == cg.KW) { c_kx = 0; ++c_ky; }
                    }
                } else if (CONV == 2) {
                    bx = c_tx << cg.lw; by = c_ty << cg.lh;
                    aimg = c_g << (6 - cg.lw - cg.lh);
                    ax = bx + w_kx - cg.pl; ay = by + w_ky - cg.pt;
                    if (++c_tx == cg.tiles_w) {
                        c_tx = 0;
                        if (++c_ty == cg.tiles_h) { c_ty = 0; ++c_g; }
                    }
                }
                mbar_wait(empty0 + 8 * s, ph ^ 1u);
                if (issuer) {
                    const uint32_t sa = smem_u32(smem + (size_t)s * STAGE_BYTES);
                    const uint32_t sb = sa + A_BYTES;
                    const uint32_t bar = full0 + 8 * s;
                    mbar_expect_tx(bar, my_bytes);
#pragma unroll
                    for (int j = 0; j < (BRES ? NA_BOX : N_BOX); ++j) {
                        if (j < NA_BOX) {
                            if (CONV == 1) tma_load_4d(sa, &tmA, bar, kA, ax, ay, aimg);
                            else if (CONV == 2) tma_load_4d(sa + j * (BK * 128), &tmA, bar, m0 + 64 * j, ax, ay, aimg);
                            else if (A_MN) tma_load_2d(sa + j * (BK * 128), &tmA, bar, m0 + 64 * j, k0);
                            else tma_load_2d(sa, &tmA, bar, k0, m0);
                        } else {
                            const int jb = j - NA_BOX;
                            if (CONV == 2) {
                                tma_load_4d(sb + jb * (BK * 128), &tmB, bar, n0 + 64 * jb, bx, by, aimg);
                            } else if (CL == 1) {
                                if (B_MN) tma_load_2d(sb + jb * (BK * 128), &tmB, bar, nB + 64 * jb, kB);
                                else tma_load_2d(sb, &tmB, bar, kB, nB);
                            } else {
                                // this CTA's half of the B tile, written into BOTH CTAs' stage (same smem offset,
                                // completing on the same barrier offset in each destination CTA)
                                if (B_MN) {
                                    const int jj = (int)crank * NB_BOX + jb;
                                    tma_load_2d_mc(sb + jj * (BK * 128), &tmB, bar, n0 + 64 * jj, k0, kMask);
                                } else {
                                    const int r0 = (int)crank * (BN / CL);
                                    tma_load_2d_mc(sb + r0 * 128, &tmB, bar, k0, n0 + r0, kMask);
                                }
                            }
                        }
                    }
                }
                __syncwarp();
            }
            g0 += (uint32_t)nkb;
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer ----------------
        // instruction descriptor: fp32 accumulate, bf16 x bf16, majors, N>>3, M>>4
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((A_MN ? 1u : 0u) << 15) |
                               ((B_MN ? 1u : 0u) << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
        // Shared-memory descriptors differ between stages / k-steps only in the 14-bit address field of
        // the low word: build the constant parts once so the per-MMA issue cost is a couple of adds.
        const uint32_t a_lbo = A_MN ? (uint32_t)(BK * 128) : 0u, b_lbo = B_MN ? (uint32_t)(BK * 128) : 0u;
        const uint32_t desc_hi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO 1024 B, version 1, SWIZZLE_128B
        const uint32_t a_lo_base = ((a_lbo >> 4) << 16) + ((smem_u32(smem) & 0x3ffffu) >> 4);
        const uint32_t b_lo_base = ((b_lbo >> 4) << 16) + (((BRES ? resb0 : smem_u32(smem) + A_BYTES) & 0x3ffffu) >> 4);
        constexpr uint32_t A_KSTEP = (A_MN ? UMMA_K * 128 : UMMA_K * 2) >> 4;
        constexpr uint32_t B_KSTEP = (B_MN ? UMMA_K * 128 : UMMA_K * 2) >> 4;
        constexpr uint32_t STAGE_STEP = STAGE_BYTES >> 4;
        const uint32_t leader = elect_one();  // the one thread that issues (and commits) every MMA
        uint32_t s = 0, ph = 0, u = 0;
        if (BRES && cluster_id < n_units) mbar_wait(bres_bar, 0u);  // the resident weights have landed
        for (int unit = cluster_id; unit < n_units; unit += n_clusters, ++u) {
            int rest = unit / (tiles_n * tiles_m);
            if (CONV == 2) rest /= cg.ntaps;
            const int kb_begin = rest * kb_per_split;
            const int nkb = min(total_kb, kb_begin + kb_per_split) - kb_begin;
            const uint32_t as = u & 1u;
            mbar_wait(tempty0 + 8 * as, ((u >> 1) & 1u) ^ 1u);  // epilogue has drained this accumulator
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t tacc = tmem_base + as * BN;
            for (int i = 0; i < nkb; ++i) {
                mbar_wait(full0 + 8 * s, ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (leader && u == 0 && i == 0) TRACE(2);
                if (leader) {
                    const uint32_t a_lo = a_lo_base + s * STAGE_STEP;
                    const uint32_t b_lo = b_lo_base + (BRES ? (uint32_t)(kb_begin + i) * (B_BYTES >> 4) : s * STAGE_STEP);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t ad = ((uint64_t)desc_hi << 32) | (uint64_t)(a_lo + k * A_KSTEP);
                        const uint64_t bd = ((uint64_t)desc_hi << 32) | (uint64_t)(b_lo + k * B_KSTEP);
                        umma_bf16(tacc, ad, bd, idesc, (i > 0 || k > 0) ? 1u : 0u, 1u);
                    }
                    // frees the smem stage (in every CTA of the cluster) when these MMAs retire
                    if (CL > 1) umma_commit_mc(empty0 + 8 * s, kMask, 1u);
                    else umma_commit(empty0 + 8 * s, 1u);
                    if (i == nkb - 1) umma_commit(tfull0 + 8 * as, 1u);  // accumulator complete
                    if (i == nkb - 1) { if (u == 0) TRACE(3); TRACE(4); }
                }
                __syncwarp();
                if (++s == STAGES) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp >= 2) {
        // ---------------- epilogue warps ----------------
        const uint32_t e_leader = elect_one();  // this warp's TMA-store / barrier thread (always the same lane)
        const int q = warp & 3;                 // TMEM lane quadrant this warp may access
        const int chalf = (warp - 2) >> 2;      // which half of the column chunks this warp drains
        const int et = (warp - 2) * 32 + lane;  // 0..255 within the epilogue group
        // BatchNorm column statistics: thread `et` owns column `et` of the tile and keeps fp64 running
        // sums across the units this CTA walks; they go to global memory (fixed-point integer atomics) only when the
        // n-tile changes or the CTA is done. Per-unit atomics to the same few addresses from every CTA
        // were 36 % of a skinny GEMM (744000 x 128 x 128: 125 us -> 80 us without them).
        double acc_s = 0.0, acc_q = 0.0;
        int acc_n0 = -1;
        auto flush_stats = [&]() {
            if (acc_n0 >= 0 && et < BN && acc_n0 + et < N) {
                stat_add(epi.colstats, acc_n0 + et, acc_s);
                stat_add(epi.colstats, N + (acc_n0 + et), acc_q);
            }
            acc_s = 0.0;
            acc_q = 0.0;
        };
        uint32_t u = 0;
        for (int unit = cluster_id; unit < n_units; unit += n_clusters, ++u) {
            const int n0 = (unit % tiles_n) * BN;
            const int mt = (unit / tiles_n) % tiles_m;
            const int m0 = (mt * CL + (int)crank) * BM;
            // where this warp's 32 rows go: GEMM rows, pixels of the tile's box (CONV 1), rows of the tap's
            // [Cin, Cout] gradient slab (CONV 2)
            int drow = m0 + q * 32, dx = 0, dy = 0, dimg = 0;
            uint32_t rowmask = 0xffffffffu;  // CONV 1: rows of this warp's box that are real output pixels
            if (CONV == 2) drow += ((unit / (tiles_n * tiles_m)) % cg.ntaps) * M;
            const int dslab = unit / (tiles_n * tiles_m);  // OUT_SLAB_F32: this unit's split = its output slab
            if (CONV == 1) {
                const int t2 = mt / cg.tiles_w, lwh = cg.lw + cg.lh;
                const int x0 = (mt - t2 * cg.tiles_w) << cg.lw, y0 = (t2 % cg.tiles_h) << cg.lh;
                const int i0 = (t2 / cg.tiles_h) << (7 - lwh);
                const int r0 = q * 32, r = r0 + lane;
                dx = x0 + (r0 & ((1 << cg.lw) - 1));
                dy = y0 + ((r0 >> cg.lw) & ((1 << cg.lh) - 1));
                dimg = i0 + (r0 >> lwh);
                const bool ok = (x0 + (r & ((1 << cg.lw) - 1))) < cg.OW &&
                                (y0 + ((r >> cg.lw) & ((1 << cg.lh) - 1))) < cg.OH && (i0 + (r >> lwh)) < cg.NB;
                rowmask = __ballot_sync(0xffffffffu, ok);
            }
            const bool rows_live = CONV == 1 ? rowmask != 0u : (m0 + q * 32 < M);  // warp-uniform
            const uint32_t as = u & 1u;
            mbar_wait(tfull0 + 8 * as, (u >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (threadIdx.x == 64) { if (u == 0) TRACE(5); TRACE(6); }
#pragma unroll 1
            for (int c = chalf; c < BN / 32; c += kEpiWarps / 4) {
                uint32_t v[32];
                tmem_ld32(tmem_base + as * BN + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
                const int col0 = n0 + c * 32;
                float f[32];
                if (epi.mode == OUT_BF16) {
                    uint32_t packed[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        packed[j] = pack_bf16x2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
                        f[2 * j] = __uint_as_float(packed[j] << 16);  // statistics of the values as stored
                        f[2 * j + 1] = __uint_as_float(packed[j] & 0xffff0000u);
                    }
                    // registers -> swizzled staging box -> one TMA store per 32 x 32 chunk: the row-per-lane
                    // global stores this replaces cost 32 LSU cycles each (32 different lines per instruction);
                    // rows >= M and columns >= N are clipped by the TMA unit
                    if (col0 < N && rows_live) {  // warp-uniform
                        const uint32_t stg = stage_out0 + ((uint32_t)(warp - 2) * SD + sbox) * 2048u;
                        if (e_leader) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(SD - 1) : "memory");  // this box was read out
                        __syncwarp();
                        const uint32_t rowaddr = stg + (uint32_t)lane * 64u, sw = ((uint32_t)lane >> 1) & 3u;
#pragma unroll
                        for (int g = 0; g < 4; ++g)
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowaddr + (((uint32_t)g ^ sw) << 4)),
                                         "r"(packed[4 * g]), "r"(packed[4 * g + 1]), "r"(packed[4 * g + 2]),
                                         "r"(packed[4 * g + 3])
                                         : "memory");
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (e_leader) {
                            if (CONV == 1)
                                asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(&tmD),
                                             "r"(stg), "r"(col0), "r"(dx), "r"(dy), "r"(dimg)
                                             : "memory");
                            else
                                asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tmD),
                                             "r"(stg), "r"(col0), "r"(drow)
                                             : "memory");
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                        last_box = stg;
                        if (SD > 1) sbox ^= 1u;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                    // fp32 store / split-K accumulation through the same 2 KB staging box, 16 columns (64-byte
                    // rows) at a time: TMA store, or TMA reduce-add into the fp32 gradient for OUT_ATOMIC_F32
                    if (CONV != 1 && rows_live) {  // warp-uniform (the convolution forward / data gradient store bf16 only)
                        const uint32_t sw = ((uint32_t)lane >> 1) & 3u;
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            if (col0 + 16 * h >= N) break;  // warp-uniform
                            const uint32_t stg = stage_out0 + ((uint32_t)(warp - 2) * SD + sbox) * 2048u;
                            const uint32_t rowaddr = stg + (uint32_t)lane * 64u;
                            if (SD > 1) sbox ^= 1u;
                            if (e_leader) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(SD - 1) : "memory");
                            __syncwarp();
#pragma unroll
                            for (int g = 0; g < 4; ++g)
                                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowaddr + (((uint32_t)g ^ sw) << 4)),
                                             "r"(v[16 * h + 4 * g]), "r"(v[16 * h + 4 * g + 1]), "r"(v[16 * h + 4 * g + 2]),
                                             "r"(v[16 * h + 4 * g + 3])
                                             : "memory");
                            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                            __syncwarp();
                            if (e_leader) {
                                if (epi.mode == OUT_SLAB_F32)  // rows >= M of the slab are clipped: slabs may sit inside other data
                                    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(&tmD),
                                                 "r"(stg), "r"(col0 + 16 * h), "r"(drow), "r"(dslab)
                                                 : "memory");
                                else if (epi.mode != OUT_ATOMIC_F32)
                                    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tmD),
                                                 "r"(stg), "r"(col0 + 16 * h), "r"(drow)
                                                 : "memory");
                                else
                                    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tmD),
                                                 "r"(stg), "r"(col0 + 16 * h), "r"(drow)
                                                 : "memory");
                                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                            }
                        }
                    }
                }
                if (epi.colstats) {  // rows past M hold exact zeros (TMA zero fill)
                    if (epi.mode == OUT_BF16) {
                        // column sums straight from the staged bf16 box (the values as stored): lane = one
                        // column pair x one half of the rows, 16 32-bit reads instead of two 31-shuffle
                        // butterflies per chunk. (Shared-memory fp32 atomics into CTA-wide accumulators were
                        // tried instead of the per-unit barrier below and were slower: 94 vs 81 us on
                        // 744000 x 128 x 128.)
                        float sx = 0.f, sy = 0.f, qx = 0.f, qy = 0.f;
                        if (col0 < N && rows_live) {
                            const uint32_t half = (uint32_t)lane >> 4, p = (uint32_t)lane & 15u;
                            const uint32_t base = last_box + half * 1024u + (p & 3u) * 4u;
                            const uint32_t jb = (p >> 2) << 4;
                            const uint32_t mybits = rowmask >> (half * 16u);
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                uint32_t w;
                                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(base + i * 64 + (jb ^ (((i >> 1) & 3) << 4))));
                                if (CONV == 1 && !((mybits >> i) & 1u)) w = 0u;  // pixel outside the output: not a sample
                                const float lo = __uint_as_float(w << 16), hi = __uint_as_float(w & 0xffff0000u);
                                sx += lo; sy += hi;
                                qx = fmaf(lo, lo, qx); qy = fmaf(hi, hi, qy);
                            }
                            sx += __shfl_xor_sync(0xffffffffu, sx, 16); sy += __shfl_xor_sync(0xffffffffu, sy, 16);
                            qx += __shfl_xor_sync(0xffffffffu, qx, 16); qy += __shfl_xor_sync(0xffffffffu, qy, 16);
                        }
                        if (lane < 16) {
                            sstat[as][0][q][c * 32 + 2 * lane] = sx; sstat[as][0][q][c * 32 + 2 * lane + 1] = sy;
                            sstat[as][1][q][c * 32 + 2 * lane] = qx; sstat[as][1][q][c * 32 + 2 * lane + 1] = qy;
                        }
                    } else {
                        float sq[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) sq[j] = f[j] * f[j];
                        const float cs = warp_colsum32(f, lane);
                        const float cq = warp_colsum32(sq, lane);
                        sstat[as][0][q][c * 32 + lane] = cs;
                        sstat[as][1][q][c * 32 + lane] = cq;
                    }
                }
            }
            // accumulator fully read: hand it back to the MMA warp
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (e_leader) mbar_arrive(tempty0 + 8 * as);
            if (threadIdx.x == 64) { if (u == 0) TRACE(7); TRACE(9); }
            if (epi.colstats) {
                // partial sums of this unit are visible after the barrier; the buffer alternates with the
                // accumulator parity, so the next unit's writers never race with these reads
                epi_bar_sync();
                if (n0 != acc_n0) {
                    flush_stats();
                    acc_n0 = n0;
                }
                if (et < BN) {
                    acc_s += (double)(sstat[as][0][0][et] + sstat[as][0][1][et] + sstat[as][0][2][et] + sstat[as][0][3][et]);
                    acc_q += (double)(sstat[as][1][0][et] + sstat[as][1][1][et] + sstat[as][1][2][et] + sstat[as][1][3][et]);
                }
            }
        }
        if (epi.colstats) flush_stats();
        if (e_leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // staging may not die under a store
        if (threadIdx.x == 64) TRACE(10);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    if (CL > 1) cluster_sync_all(); else __syncthreads();  // no CTA may exit while its peer still multicasts into it
    if (threadIdx.x == 0) { TRACE(11); TRACE_G(12); }
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BN)) : "memory");
}

// ---------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------
constexpr int kMaxResidentKb = 9;  // resident-B convolutions: at most 9 k-blocks of 64-wide weights (72 KB)
// operand with `rows` along M/N and `kdim` along K; ld in elements
int make_operand_map(CUtensorMap* map, const void* ptr, long long rows, long long kdim, long long ld, bool mn_major,
                     int tile_rows) {
    PFN_cuTensorMapEncodeTiled enc = spnet_get_tensormap_encoder();
    if (!enc) {
        spnet_set_error("gemm_bf16: cuTensorMapEncodeTiled entry point not available");
        return SPNET_ERR_CUDA;
    }
    cuuint64_t dims[2], strides[1];
    cuuint32_t box[2], estr[2] = {1, 1};
    if (mn_major) {
        dims[0] = (cuuint64_t)rows; dims[1] = (cuuint64_t)kdim;
        box[0] = 64; box[1] = BK;
    } else {
        dims[0] = (cuuint64_t)kdim; dims[1] = (cuuint64_t)rows;
        box[0] = BK; box[1] = (cuuint32_t)tile_rows;
    }
    strides[0] = (cuuint64_t)ld * 2;
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        spnet_set_error("gemm_bf16: cuTensorMapEncodeTiled failed (%d) rows=%lld k=%lld ld=%lld mn=%d", (int)r, rows,
                        kdim, ld, (int)mn_major);
        return SPNET_ERR_CUDA;
    }
    return SPNET_OK;
}

// CONV 0: tiles_m_conv / ntaps unused. CONV 1: tiles_m_conv = number of pixel tiles. CONV 2: ntaps = cg.ntaps.
template <int BN, bool A_MN, bool B_MN, int CL, int CONV = 0, bool BRES = false>
int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& td, GemmEpi epi, int M, int N, int K,
                int splits, cudaStream_t stream, ConvGeom cg = ConvGeom(), int tiles_m_conv = 0) {
    // BN = 128: one ring stage traded for the second staging box; BN = 64 (narrow convolutions): deep ring
    constexpr int STAGES = BN <= 64 ? 7 : (BN <= 128) ? 5 : 4;
    // (resident B: the ring carries A only; the weights take ceil(K/64) tiles of BN x 64 next to it)
    const size_t smem = (size_t)STAGES * (BM * BK * 2 + (BRES ? 0 : BN * BK * 2)) +
                        (BRES ? (size_t)((K + BK - 1) / BK) * BN * BK * 2 : 0) + 1024 + kEpiWarps * 2048 * (BN <= 128 ? 2 : 1);
    auto kern = gemm_tc_kernel<BN, A_MN, B_MN, STAGES, CL, CONV, BRES>;
    // per (instantiation, device): the dynamic shared-memory opt-in is a per-device function attribute
    static bool configured[64] = {};
    if (spnet_first_use_on_device(configured)) {
        // (resident B: the size depends on K; opt in to the largest this mode is dispatched with)
        const size_t smem_max = BRES ? (size_t)STAGES * BM * BK * 2 + (size_t)kMaxResidentKb * BN * BK * 2 + 1024 + kEpiWarps * 2048 * 2 : smem;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max);
        if (e != cudaSuccess) {
            spnet_set_error("gemm_bf16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return SPNET_ERR_CUDA;
        }
    }
    const int total_kb = (K + BK - 1) / BK;
    if (splits < 1) splits = 1;
    if (splits > total_kb) splits = total_kb;
    const int kbps = (total_kb + splits - 1) / splits;
    splits = (total_kb + kbps - 1) / kbps;  // no empty splits
    const int tiles_m = CONV == 1 ? tiles_m_conv : ((M + BM - 1) / BM + CL - 1) / CL;  // m-tile groups of CL
    const int tiles_n = (N + BN - 1) / BN;
    const long long units = (long long)tiles_m * tiles_n * splits * (CONV == 2 ? cg.ntaps : 1);
    if (units > 0x7fffffffLL) {
        spnet_set_error("gemm_bf16: too many tiles");
        return SPNET_ERR_ARG;
    }
    // persistent grid: one CTA per SM; CL > 1 launches the grid as clusters of CL CTAs (the CTA pairs)
    const int max_clusters = spnet_num_sms() / CL;
    const int grid = (int)(units < max_clusters ? units : max_clusters) * CL;
    cudaLaunchAttribute cluster = {};
    cluster.id = cudaLaunchAttributeClusterDimension;
    cluster.val.clusterDim.x = CL;
    cluster.val.clusterDim.y = 1;
    cluster.val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cfg.attrs = &cluster;
    cfg.numAttrs = CL > 1 ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, ta, tb, td, epi, M, N, K, kbps, tiles_m, tiles_n, (int)units, cg);
    if (e != cudaSuccess) {
        spnet_set_error("gemm_bf16: launch: %s", cudaGetErrorString(e));
        return SPNET_ERR_CUDA;
    }
    return spnet_check_launch("gemm_bf16");
}

}  // namespace

extern "C" {

#ifdef SPNET_GEMM_TRACE
int spnet_gemm_trace_read(unsigned long long* host) {
    return cudaMemcpyFromSymbol(host, g_gemm_trace, sizeof(g_gemm_trace)) == cudaSuccess ? 0 : 1;
}
#endif

// D[M,N] (op)= A[M,K] * B[K,N], bf16 operands, fp32 accumulation in TMEM.
//   a_mn / b_mn : 0 = K-major (ptr[r*ld + k]), 1 = MN-major (ptr[k*ld + r])
//   out_mode    : 0 store bf16, 1 store fp32, 2 reduce-add fp32 (split-K, order of the adds not fixed), 3 fp32
//                 SLABS: split s (k-blocks [s*kbps, (s+1)*kbps), kbps = ceil(ceil(K/64) / splits)) stores its partial
//                 product as an [M, N] matrix (row stride ldd) at D + s * slab_stride elements. Two uses: split-K with
//                 a FIXED summation order (spnet_slab_reduce adds the slabs in order), and BATCHED GEMMs whose
//                 operands are stacked along K - e.g. the weight gradients of the 24 identical middle-flow layers in
//                 one launch: K = 24 x rows, splits = 24, slab s = dW of layer s, written straight into the flat
//                 gradient buffer (rows >= M are clipped by the TMA unit, so slabs may be embedded in other data)
//   colstats    : nullable fp64 [2*N]; per-column sum and sum of squares of the values as
//                 stored (after bf16 rounding in mode 0) are atomically added
//   Requirements: pointers 16-byte aligned, lda/ldb multiples of 8, N % 8 == 0 (bf16 out)
//                 or N % 4 == 0 (fp32 store).
int spnet_gemm_bf16(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, void* D,
                    long long ldd, long long slab_stride, int out_mode, int M, int N, int K, int splits, long long* colstats,
                    cudaStream_t stream) {
    SPNET_REQUIRE(A && B && D, "gemm_bf16: null pointer");
    SPNET_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_bf16: bad shape %d %d %d", M, N, K);
    SPNET_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, "gemm_bf16: lda/ldb must be multiples of 8 elements");
    SPNET_REQUIRE(((uintptr_t)A % 16 == 0) && ((uintptr_t)B % 16 == 0) && ((uintptr_t)D % 16 == 0),
                  "gemm_bf16: pointers must be 16-byte aligned");
    SPNET_REQUIRE(out_mode >= 0 && out_mode <= 3, "gemm_bf16: bad out_mode %d", out_mode);
    SPNET_REQUIRE(out_mode != OUT_BF16 || (N % 8 == 0 && ldd % 8 == 0), "gemm_bf16: bf16 output needs N, ldd %% 8 == 0");
    SPNET_REQUIRE(out_mode == OUT_BF16 || ldd % 4 == 0, "gemm_bf16: fp32 output needs ldd %% 4 == 0");
    // 128x256 tiles when N is wide: one A tile then feeds 256 output columns, which cuts the
    // L2->SM operand traffic per FLOP by a third (the 128x128 kernel is L2-bandwidth bound).
    const bool wide = N >= 512;
    // CTA pairs (B tile multicast) when there are at least two m-tiles to pair up
    const bool pair = wide && M > BM;
    if (splits <= 0) {
        // auto split-K (atomic output only): fill the SMs (or SM pairs) once without spilling into a
        // second, nearly empty round; keep at least 4 k-blocks per split
        splits = 1;
        if (out_mode == OUT_ATOMIC_F32) {
            const int bn = wide ? 256 : 128, cl = pair ? 2 : 1;
            const long long tiles = (long long)(((M + BM - 1) / BM + cl - 1) / cl) * ((N + bn - 1) / bn);
            const long long slots = spnet_num_sms() / cl;
            long long sp = tiles >= slots ? 1 : slots / tiles;
            const long long kb = (K + BK - 1) / BK;
            if (sp > kb / 4) sp = kb / 4;
            splits = (int)(sp < 1 ? 1 : sp);
        }
    }
    SPNET_REQUIRE(splits <= 1 || out_mode == OUT_ATOMIC_F32 || out_mode == OUT_SLAB_F32, "gemm_bf16: split-K needs out_mode 2 or 3");
    int n_slabs = 1;
    if (out_mode == OUT_SLAB_F32) {
        SPNET_REQUIRE(slab_stride > 0 && slab_stride % 4 == 0, "gemm_bf16: slab_stride must be a positive multiple of 4 elements");
        const int kb = (K + BK - 1) / BK;
        int sp = splits < 1 ? 1 : (splits > kb ? kb : splits);
        const int kbps = (kb + sp - 1) / sp;
        n_slabs = (kb + kbps - 1) / kbps;
    }
    SPNET_REQUIRE(!(colstats && splits > 1), "gemm_bf16: column statistics are not defined for split-K partials");
    CUtensorMap ta, tb;
    int rc = make_operand_map(&ta, A, M, K, lda, a_mn != 0, BM);
    if (rc) return rc;
    rc = make_operand_map(&tb, B, N, K, ldb, b_mn != 0, wide ? (pair ? 128 : 256) : (N <= 64 ? 64 : 128));
    if (rc) return rc;
    CUtensorMap td;  // output boxes of the TMA-store epilogue: 32 x 32 bf16 or 32 x 16 fp32 (64-byte rows, SWIZZLE_64B)
    {
        PFN_cuTensorMapEncodeTiled enc = spnet_get_tensormap_encoder();
        const bool ob = out_mode == OUT_BF16;
        const bool slabs = out_mode == OUT_SLAB_F32;
        cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)M, (cuuint64_t)n_slabs};
        cuuint64_t strides[2] = {(cuuint64_t)ldd * (ob ? 2 : 4), (cuuint64_t)slab_stride * 4};
        cuuint32_t box[3] = {ob ? 32u : 16u, 32u, 1u}, estr[3] = {1, 1, 1};
        CUresult r = enc(&td, ob ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, slabs ? 3 : 2, D, dims,
                         strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                         CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        SPNET_REQUIRE(r == CUDA_SUCCESS, "gemm_bf16: cuTensorMapEncodeTiled (output) failed (%d) M=%d N=%d ldd=%lld", (int)r, M, N, ldd);
    }
    GemmEpi epi = {D, ldd, out_mode, 0, colstats};
#define SPNET_GEMM_DISPATCH(BN_, CL_)                                                                                       \
    do {                                                                                                                    \
        if (a_mn) {                                                                                                         \
            if (b_mn) return launch_gemm<BN_, true, true, CL_>(ta, tb, td, epi, M, N, K, splits, stream);                   \
            return launch_gemm<BN_, true, false, CL_>(ta, tb, td, epi, M, N, K, splits, stream);                            \
        }                                                                                                                   \
        if (b_mn) return launch_gemm<BN_, false, true, CL_>(ta, tb, td, epi, M, N, K, splits, stream);                      \
        return launch_gemm<BN_, false, false, CL_>(ta, tb, td, epi, M, N, K, splits, stream);                               \
    } while (0)
    // CTA pairs run one cta_group::1 MMA per CTA over a multicast copy of B; a cta_group::2 pair MMA (one 256-row MMA
    // over both CTAs' shared memory) measured slower on every shape of this network on B200 (step 7.32 against 7.16 ms).
    if (pair) SPNET_GEMM_DISPATCH(256, 2);
    if (wide) SPNET_GEMM_DISPATCH(256, 1);
    // N <= 64 (the data gradients into Xception's 64-channel block 1 output): 64-wide tiles - a 128-wide tile would
    // spend half of its B traffic, MMA columns and epilogue on columns that do not exist
    if (N <= 64) SPNET_GEMM_DISPATCH(64, 1);
    SPNET_GEMM_DISPATCH(128, 1);
#undef SPNET_GEMM_DISPATCH
}

// ---------------------------------------------------------------------------------
// implicit-GEMM convolutions (stride 1, any kernel size / padding, NHWC bf16)
// ---------------------------------------------------------------------------------
}  // extern "C"

namespace {

// pixel box (2^lw x 2^lh x 2^(log_rows-lw-lh) images) that wastes the fewest rows on overhang
void pick_pixel_box(int log_rows, int OW, int OH, int NB, int* lw_out, int* lh_out) {
    double best = -1.0;
    for (int lw = 0; lw <= log_rows; ++lw)
        for (int lh = 0; lw + lh <= log_rows; ++lh) {
            const long long TW = 1 << lw, TH = 1 << lh, TN = 1 << (log_rows - lw - lh);
            const long long cover = ((OW + TW - 1) / TW * TW) * ((OH + TH - 1) / TH * TH) * ((NB + TN - 1) / TN * TN);
            const double util = (double)OW * OH * NB / (double)cover + 1e-6 * lw;  // ties: wider boxes
            if (util > best) { best = util; *lw_out = lw; *lh_out = lh; }
        }
}

// NHWC activation [NB, H, W, C] with pixel stride ld (elements): 4-D map, box = 64 channels x pixel box
// row_ld: elements between image rows (W * ld for a dense image; larger when W is a clipped extent, see the kw-fold
// entry points below)
int make_pixel_map(CUtensorMap* map, const void* ptr, int NB, int H, int W, int C, long long ld, int lw, int lh, int ln,
                   int box_c, CUtensorMapSwizzle swz, CUtensorMapL2promotion prom, long long row_ld = 0) {
    if (row_ld <= 0) row_ld = (long long)W * ld;
    PFN_cuTensorMapEncodeTiled enc = spnet_get_tensormap_encoder();
    if (!enc) {
        spnet_set_error("conv_tc: cuTensorMapEncodeTiled entry point not available");
        return SPNET_ERR_CUDA;
    }
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)NB};
    cuuint64_t strides[3] = {(cuuint64_t)ld * 2, (cuuint64_t)row_ld * 2, (cuuint64_t)H * row_ld * 2};
    cuuint32_t box[4] = {(cuuint32_t)box_c, 1u << lw, 1u << lh, 1u << ln}, estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swz, prom, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        spnet_set_error("conv_tc: cuTensorMapEncodeTiled failed (%d) NB=%d H=%d W=%d C=%d ld=%lld box=%d,%d,%d,%d", (int)r, NB,
                        H, W, C, ld, box_c, 1 << lw, 1 << lh, 1 << ln);
        return SPNET_ERR_CUDA;
    }
    return SPNET_OK;
}

// forward (dgrad = 0): out[n, y, x, :] = sum_taps in[n, y + ky - pt, x + kx - pl, :] . Wt[ky, kx, :, :]
// data gradient (dgrad = 1): out = dX [NB, OH, OW, Cin] from in = dY [NB, IH, IW, Cout]:
//                            out[n, y, x, ci] = sum_taps in[n, y - ky + pt, x - kx + pl, :] . Wt[ky, kx, ci, :]
// Wt is the Keras kernel [KH, KW, Cin, Cout]; c_in / c_out are the channel counts of `in` / `out`.
int conv_tc_fwd_like(bool dgrad, const void* in, long long ld_in, int NB, int IH, int IW, int c_in, const void* Wt,
                     int Cin, int Cout, void* out, long long ld_out, int OH, int OW, int c_out, int KH, int KW, int pt,
                     int pl, long long* colstats, cudaStream_t stream, long long row_ld_in = 0) {
    ConvGeom cg = {};
    pick_pixel_box(7, OW, OH, NB, &cg.lw, &cg.lh);
    const int ln = 7 - cg.lw - cg.lh;
    cg.tiles_w = (OW + (1 << cg.lw) - 1) >> cg.lw;
    cg.tiles_h = (OH + (1 << cg.lh) - 1) >> cg.lh;
    const int groups = (NB + (1 << ln) - 1) >> ln;
    cg.OW = OW; cg.OH = OH; cg.NB = NB;
    cg.KW = KW; cg.ntaps = KH * KW;
    cg.cin_blocks = (c_in + BK - 1) / BK;
    cg.pt = pt; cg.pl = pl; cg.sign = dgrad ? -1 : 1;
    cg.b_tap_stride = Cin;
    cg.b_tap_on_k = dgrad ? 0 : 1;
    const long long tiles_m = (long long)cg.tiles_w * cg.tiles_h * groups;
    SPNET_REQUIRE(tiles_m < (1 << 24), "conv_tc: too many pixel tiles");
    const int N = c_out, K = cg.ntaps * cg.cin_blocks * BK;
    const int bn = N <= 64 ? 64 : 128;
    CUtensorMap ta, tb, td;
    int rc = make_pixel_map(&ta, in, NB, IH, IW, c_in, ld_in, cg.lw, cg.lh, ln, BK, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, row_ld_in);
    if (rc) return rc;
    // weights as one 2-D matrix: forward [taps*Cin (k), Cout (n)] MN-major; data gradient: rows (n) = tap*Cin + ci,
    // k = Cout contiguous, K-major
    if (!dgrad) rc = make_operand_map(&tb, Wt, Cout, (long long)cg.ntaps * Cin, Cout, true, bn);
    else rc = make_operand_map(&tb, Wt, (long long)cg.ntaps * Cin, Cout, Cout, false, bn);
    if (rc) return rc;
    {   // output boxes: this epilogue warp's 32 rows of the tile = a (bw x bh x bn) sub-box of pixels
        const int lbw = cg.lw < 5 ? cg.lw : 5, lbh = cg.lh < 5 - lbw ? cg.lh : 5 - lbw, lbn = 5 - lbw - lbh;
        rc = make_pixel_map(&td, out, NB, OH, OW, c_out, ld_out, lbw, lbh, lbn, 32, CU_TENSOR_MAP_SWIZZLE_64B,
                            CU_TENSOR_MAP_L2_PROMOTION_NONE);
        if (rc) return rc;
    }
    GemmEpi epi = {out, ld_out, OUT_BF16, 0, colstats};
    const int M = (int)(tiles_m * BM);
    // one 64-wide n-tile and at most kMaxResidentKb k-blocks: the weights stay in shared memory (BRES)
    const bool bres = bn == 64 && K / BK <= kMaxResidentKb;
    if (!dgrad) {
        if (bres) return launch_gemm<64, false, true, 1, 1, true>(ta, tb, td, epi, M, N, K, 1, stream, cg, (int)tiles_m);
        if (bn == 64) return launch_gemm<64, false, true, 1, 1>(ta, tb, td, epi, M, N, K, 1, stream, cg, (int)tiles_m);
        return launch_gemm<128, false, true, 1, 1>(ta, tb, td, epi, M, N, K, 1, stream, cg, (int)tiles_m);
    }
    if (bres) return launch_gemm<64, false, false, 1, 1, true>(ta, tb, td, epi, M, N, K, 1, stream, cg, (int)tiles_m);
    if (bn == 64) return launch_gemm<64, false, false, 1, 1>(ta, tb, td, epi, M, N, K, 1, stream, cg, (int)tiles_m);
    return launch_gemm<128, false, false, 1, 1>(ta, tb, td, epi, M, N, K, 1, stream, cg, (int)tiles_m);
}

int conv_tc_wgrad_impl(const void* X, long long ldx, int NB, int H, int W, int Cin, const void* dY, long long ldy, int OH,
                       int OW, int Cout, float* dW, int KH, int KW, int pt, int pl, cudaStream_t stream, long long row_ld_x) {
    ConvGeom cg = {};
    pick_pixel_box(6, OW, OH, NB, &cg.lw, &cg.lh);
    const int ln = 6 - cg.lw - cg.lh;
    cg.tiles_w = (OW + (1 << cg.lw) - 1) >> cg.lw;
    cg.tiles_h = (OH + (1 << cg.lh) - 1) >> cg.lh;
    const int groups = (NB + (1 << ln) - 1) >> ln;
    cg.OW = OW; cg.OH = OH; cg.NB = NB;
    cg.KW = KW; cg.ntaps = KH * KW;
    cg.cin_blocks = 1;
    cg.pt = pt; cg.pl = pl; cg.sign = 1;
    const long long pixel_blocks = (long long)cg.tiles_w * cg.tiles_h * groups;
    SPNET_REQUIRE(pixel_blocks < (1 << 24), "conv_tc_wgrad: too many pixel blocks");
    const int M = Cin, N = Cout, K = (int)pixel_blocks * BK;
    const int bn = N <= 64 ? 64 : 128;
    CUtensorMap ta, tb, td;
    int rc = make_pixel_map(&ta, X, NB, H, W, Cin, ldx, cg.lw, cg.lh, ln, 64, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, row_ld_x);
    if (rc) return rc;
    rc = make_pixel_map(&tb, dY, NB, OH, OW, Cout, ldy, cg.lw, cg.lh, ln, 64, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
    if (rc) return rc;
    {
        PFN_cuTensorMapEncodeTiled enc = spnet_get_tensormap_encoder();
        cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)cg.ntaps * M}, strides[1] = {(cuuint64_t)N * 4};
        cuuint32_t box[2] = {16u, 32u}, estr[2] = {1, 1};
        CUresult r = enc(&td, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dW, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        SPNET_REQUIRE(r == CUDA_SUCCESS, "conv_tc_wgrad: cuTensorMapEncodeTiled (output) failed (%d)", (int)r);
    }
    // split the pixel reduction so that taps x tiles x splits fills the SMs about once; >= 4 pixel blocks per split
    const long long tiles = (long long)((M + BM - 1) / BM) * ((N + bn - 1) / bn) * cg.ntaps;
    const long long nsm_ = spnet_num_sms();
    long long sp = tiles >= nsm_ ? 1 : nsm_ / tiles;
    if (sp > pixel_blocks / 4) sp = pixel_blocks / 4;
    const int splits = (int)(sp < 1 ? 1 : sp);
    GemmEpi epi = {dW, N, OUT_ATOMIC_F32, 0, nullptr};
    if (bn == 64) return launch_gemm<64, true, true, 1, 2>(ta, tb, td, epi, M, N, K, splits, stream, cg, 0);
    return launch_gemm<128, true, true, 1, 2>(ta, tb, td, epi, M, N, K, splits, stream, cg, 0);
}

}  // namespace

extern "C" {

#define SPNET_CONV_TC_CHECKS(X, ldx, Wt, Y, ldy, Cin, Cout)                                                          \
    SPNET_REQUIRE(X && Wt && Y, "conv_tc: null pointer");                                                            \
    SPNET_REQUIRE(Cin % 8 == 0 && Cout % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && ldx >= Cin && ldy >= Cout,        \
                  "conv_tc: channel counts and pixel strides must be multiples of 8 (Cin %d Cout %d)", Cin, Cout);   \
    SPNET_REQUIRE(((uintptr_t)X % 16 == 0) && ((uintptr_t)Wt % 16 == 0) && ((uintptr_t)Y % 16 == 0),                 \
                  "conv_tc: pointers must be 16-byte aligned")

// Y[NB, OH, OW, Cout] = conv(X[NB, H, W, Cin], Wt[KH, KW, Cin, Cout]), stride 1, top / left padding pt / pl
// (bottom / right padding is whatever OH / OW imply), bf16 in / out, fp32 accumulation; optional fused
// per-channel sum / sum of squares of Y as stored (fp64 [2*Cout], atomically added).
int spnet_conv_tc_fwd(const void* X, long long ldx, int NB, int H, int W, int Cin, const void* Wt, void* Y, long long ldy,
                      int OH, int OW, int Cout, int KH, int KW, int pt, int pl, long long* colstats, cudaStream_t stream) {
    SPNET_CONV_TC_CHECKS(X, ldx, Wt, Y, ldy, Cin, Cout);
    SPNET_REQUIRE(NB > 0 && OH > 0 && OW > 0 && KH > 0 && KW > 0, "conv_tc_fwd: bad shape");
    return conv_tc_fwd_like(false, X, ldx, NB, H, W, Cin, Wt, Cin, Cout, Y, ldy, OH, OW, Cout, KH, KW, pt, pl, colstats,
                            stream);
}

// dX[NB, H, W, Cin] = data gradient of the convolution above from dY[NB, OH, OW, Cout] (overwrites dX)
int spnet_conv_tc_dgrad(const void* dY, long long ldy, int NB, int OH, int OW, int Cout, const void* Wt, void* dX,
                        long long ldx, int H, int W, int Cin, int KH, int KW, int pt, int pl, cudaStream_t stream) {
    SPNET_CONV_TC_CHECKS(dX, ldx, Wt, dY, ldy, Cin, Cout);
    SPNET_REQUIRE(NB > 0 && OH > 0 && OW > 0 && KH > 0 && KW > 0, "conv_tc_dgrad: bad shape");
    return conv_tc_fwd_like(true, dY, ldy, NB, OH, OW, Cout, Wt, Cin, Cout, dX, ldx, H, W, Cin, KH, KW, pt, pl, nullptr,
                            stream);
}

// dW[KH, KW, Cin, Cout] (fp32) += sum over pixels X[n, y + ky - pt, x + kx - pl, ci] * dY[n, y, x, co]
// (TMA reduce-add: the caller zeroes dW or accumulates into it on purpose).
int spnet_conv_tc_wgrad(const void* X, long long ldx, int NB, int H, int W, int Cin, const void* dY, long long ldy, int OH,
                        int OW, int Cout, float* dW, int KH, int KW, int pt, int pl, cudaStream_t stream) {
    SPNET_CONV_TC_CHECKS(X, ldx, dW, dY, ldy, Cin, Cout);
    SPNET_REQUIRE(NB > 0 && OH > 0 && OW > 0 && KH > 0 && KW > 0, "conv_tc_wgrad: bad shape");
    return conv_tc_wgrad_impl(X, ldx, NB, H, W, Cin, dY, ldy, OH, OW, Cout, dW, KH, KW, pt, pl, stream, 0);
}

// ---- 'valid' convolutions of a DENSE NHWC tensor with the KW taps folded into the channel axis ----------------
// The KW taps of one filter row read KW * Cin CONTIGUOUS elements of X (pixels x .. x+KW-1 of one image row), so
// X is described to the TMA unit as [NB, H, W-KW+1, KW*Cin] with a pixel stride of Cin elements (rows of the map
// overlap) and the convolution runs as a KH x 1 one over KW*Cin channels: KH * ceil(KW*Cin/64) k-blocks per tile
// instead of KH*KW half-empty ones when Cin = 32 (block1_conv2 of the reference's Xception: 3x3, 32 -> 64,
// spnet/models.py:359 via keras.applications.xception), and no im2col buffer. The Keras kernel [KH, KW, Cin, Cout]
// is already the [KH, 1, KW*Cin, Cout] kernel of the folded problem.
int spnet_conv_tc_fwd_kwfold(const void* X, int NB, int H, int W, int Cin, const void* Wt, void* Y, long long ldy, int Cout,
                             int KH, int KW, long long* colstats, cudaStream_t stream) {
    SPNET_CONV_TC_CHECKS(X, (long long)Cin, Wt, Y, ldy, Cin, Cout);
    const int OH = H - KH + 1, OW = W - KW + 1;
    SPNET_REQUIRE(NB > 0 && OH > 0 && OW > 0 && KH > 0 && KW > 0, "conv_tc_fwd_kwfold: bad shape");
    return conv_tc_fwd_like(false, X, Cin, NB, H, OW, KW * Cin, Wt, KW * Cin, Cout, Y, ldy, OH, OW, Cout, KH, 1, 0, 0,
                            colstats, stream, (long long)W * Cin);
}

// dW[KH, KW, Cin, Cout] (fp32) += weight gradient of the convolution above (TMA reduce-add)
int spnet_conv_tc_wgrad_kwfold(const void* X, int NB, int H, int W, int Cin, const void* dY, long long ldy, int Cout,
                               float* dW, int KH, int KW, cudaStream_t stream) {
    SPNET_CONV_TC_CHECKS(X, (long long)Cin, dW, dY, ldy, Cin, Cout);
    const int OH = H - KH + 1, OW = W - KW + 1;
    SPNET_REQUIRE(NB > 0 && OH > 0 && OW > 0 && KH > 0 && KW > 0, "conv_tc_wgrad_kwfold: bad shape");
    return conv_tc_wgrad_impl(X, Cin, NB, H, OW, KW * Cin, dY, ldy, OH, OW, Cout, dW, KH, 1, 0, 0, stream,
                              (long long)W * Cin);
}

}  // extern "C"
