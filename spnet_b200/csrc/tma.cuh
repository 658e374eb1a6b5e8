// TMA (cp.async.bulk.tensor) + mbarrier helpers shared by the GEMM and depthwise kernels.
#pragma once
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// one lane of a converged warp (always the same one), in a form the compiler recognises as "one thread"
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t leader;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));
    return leader;
}

// generic-proxy writes to shared memory (st.shared) made visible to the async proxy (TMA, tcgen05.mma)
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fence_proxy_async_smem();
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a lost arrive turns into a trap (reported as a launch failure) instead of a hang.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    long long t0 = 0;
    for (uint32_t spins = 0; !ok; ++spins) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!ok && (spins & 1023u) == 1023u) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000LL) __trap();  // ~2 s at 2 GHz
        }
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// ---- TMA-store epilogue: registers -> 32-row x 64-byte staging box (SWIZZLE_64B) -> one bulk tensor store -------
// Row `lane` of the box, its 16-byte chunk g at lane * 64 + ((g ^ ((lane >> 1) & 3)) << 4): the layout a SWIZZLE_64B
// map reads, and conflict-free for the warp's four v4 stores.
__device__ __forceinline__ void stage_box_row_sw64(uint32_t box, uint32_t lane, const uint32_t* v) {
    const uint32_t rowaddr = box + lane * 64u, sw = (lane >> 1) & 3u;
#pragma unroll
    for (int g = 0; g < 4; ++g)
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rowaddr + (((uint32_t)g ^ sw) << 4)),
                     "r"(v[4 * g]), "r"(v[4 * g + 1]), "r"(v[4 * g + 2]), "r"(v[4 * g + 3])
                     : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src),
                 "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map), "r"(src),
                 "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map),
                 "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
// fp32 add of the box into global memory, element-wise (not ordered between boxes)
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
                 "r"(src), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N committed store groups still read their shared-memory source (N an immediate)
template <int N> __device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

static inline PFN_cuTensorMapEncodeTiled spnet_get_tensormap_encoder() {
    static PFN_cuTensorMapEncodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
    }
    return fn;
}

// A tiled tensor map with unit element strides and no interleave. dims and box give the `rank` dimensions innermost
// first; strides are the byte strides of dimensions 1 .. rank-1. `who` names the caller in the error message.
static inline int spnet_encode_tiled(CUtensorMap* map, const char* who, CUtensorMapDataType dtype, int rank,
                                     const void* ptr, const cuuint64_t* dims, const cuuint64_t* strides,
                                     const cuuint32_t* box, CUtensorMapSwizzle swizzle,
                                     CUtensorMapL2promotion promotion, CUtensorMapFloatOOBfill oob_fill) {
    PFN_cuTensorMapEncodeTiled enc = spnet_get_tensormap_encoder();
    if (!enc) {
        spnet_set_error("%s: cuTensorMapEncodeTiled entry point not available", who);
        return SPNET_ERR_CUDA;
    }
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const CUresult r = enc(map, dtype, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, promotion, oob_fill);
    if (r != CUDA_SUCCESS) {
        char s[320];  // at most 5 dims: 5 x (dim/box) + 4 strides fit
        int n = 0;
        const int nd = rank < 5 ? rank : 5;
        for (int i = 0; i < nd; ++i) n += snprintf(s + n, sizeof(s) - n, " %llu/%u", (unsigned long long)dims[i], box[i]);
        n += snprintf(s + n, sizeof(s) - n, ", byte strides");
        for (int i = 1; i < nd; ++i) n += snprintf(s + n, sizeof(s) - n, " %llu", (unsigned long long)strides[i - 1]);
        spnet_set_error("%s: cuTensorMapEncodeTiled failed (%d) for %p, dim/box%s", who, (int)r, ptr, s);
        return SPNET_ERR_CUDA;
    }
    return SPNET_OK;
}
