// mctq_tcgen05.cuh -- the tensor-core pieces shared by the packed-weight GEMMs (mctq_packed_gemm.cu, mctq_packed_igemm.cu):
// thread-block-cluster helpers for the split-K reduction over distributed shared memory, tcgen05 fences, and the
// K-major 128-byte-swizzle shared-memory operand layout with its matrix descriptor.
#pragma once
#include "mctq_common.cuh"

namespace mctq {

__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_size() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t peer_addr(uint32_t local_addr, uint32_t rank) {
    uint32_t a;
    asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(local_addr), "r"(rank));
    return a;
}
// ordered after the cluster barrier by its acquire (asm volatile keeps it below); no memory clobber, so loads overlap
__device__ __forceinline__ float ld_peer(uint32_t cluster_addr) {
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(cluster_addr));
    return v;
}
__device__ __forceinline__ int32_t ld_peer_s32(uint32_t cluster_addr) {
    int32_t v;
    asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(cluster_addr));
    return v;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor: K-major, 128-byte swizzle, 8-row groups 1024 bytes apart (sm_100 descriptor version 1)
__device__ __forceinline__ uint64_t sw128_desc(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}
// byte offset of the 16-byte group j of row r inside a stage operand: Swizzle<3,4,3> on 1024-byte atoms (the layout a TMA
// copy with CU_TENSOR_MAP_SWIZZLE_128B writes)
__device__ __forceinline__ uint32_t sw128_off(uint32_t r, uint32_t j) { return r * 128u + ((j ^ (r & 7u)) << 4); }

__device__ __forceinline__ void st_shared_v4(uint32_t addr, const uint32_t* w) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
}

// TMEM lanes 32 * (warp % 4) .. + 31, 16 consecutive 32-bit columns from `taddr` (one value per thread and column)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* u) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
                   "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// TMEM columns of an accumulator of nt columns: a power of two >= 32
inline uint32_t tmem_columns(int nt) {
    uint32_t cols = 32;
    while (cols < (uint32_t)nt) cols *= 2;
    return cols;
}
// dynamic shared memory that keeps co-resident CTAs within the SM's 512 TMEM columns: enough that no more of them fit
inline size_t tmem_smem_floor(uint32_t cols) {
    const size_t sm_bytes = 228 * 1024, max_ctas = 512 / cols;
    return sm_bytes / (max_ctas + 1) + 1 - 1024 + 256;
}

}  // namespace mctq
