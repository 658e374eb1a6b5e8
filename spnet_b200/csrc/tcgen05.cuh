// tcgen05 (5th-generation tensor core) issue and TMEM helpers shared by the GEMM and the fused pointwise backward.
#pragma once
#include "tma.cuh"

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

// One warp allocates `ncols` TMEM columns (a power of two >= 32) for the CTA and writes their base address to the
// shared-memory word at `holder`, then gives up the CTA's right to allocate more.
__device__ __forceinline__ void tmem_alloc(uint32_t holder, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(holder), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
// by the warp that allocated, once every tcgen05 access of the CTA is complete
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}
