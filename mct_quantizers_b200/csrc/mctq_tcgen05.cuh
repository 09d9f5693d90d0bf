// mctq_tcgen05.cuh -- the tensor-core frame of the packed-weight GEMMs (mctq_packed_gemm.cu, mctq_packed_igemm.cu): 128
// output features on the MMA's M, nt batch rows on its N, the accumulator in tensor memory, the row length split over the
// CTAs of a cluster.  Here: TMEM lifetime, MMA issue and commit, the 128-byte-swizzle operand layout, the split-K tile and
// the reduction of its partial sums over distributed shared memory, and the host's row tile, ring size and launch loop.
// Each GEMM keeps its own main loop, split policy and per-value epilogue arithmetic.
#pragma once
#include <algorithm>

#include "mctq_common.cuh"

namespace mctq {

constexpr int kTcRows = 128;          // output features per CTA: the MMA's M, one TMEM lane each

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
template <typename Acc>
__device__ __forceinline__ Acc ld_peer(uint32_t cluster_addr) {
    Acc v;
    if constexpr (std::is_same<Acc, float>::value) asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(cluster_addr));
    else asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(cluster_addr));
    return v;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// warp 0 allocates `cols` TMEM columns (the address lands in *slot) and gives up the permit, so co-resident CTAs can allocate
__device__ __forceinline__ void tmem_alloc(int warp, uint32_t* slot, uint32_t cols) {
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(slot)), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
}
// every thread, after tmem_alloc (and the mbarrier inits): the CTA-wide barrier publishes both
__device__ __forceinline__ uint32_t tmem_address(const uint32_t* slot) {
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *slot;
}
// every thread, last: once all tensor-memory reads are done, warp 0 frees the columns
__device__ __forceinline__ void tmem_dealloc(int warp, uint32_t tmem, uint32_t cols) {
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(cols) : "memory");
    }
}

// instruction descriptor, A and B K-major, M = kTcRows, N = nt: accumulator `d` (1 f32, 2 s32), operands `a` / `b`
// (kind::f16: 0 f16, 1 bf16; kind::i8: 0 unsigned, 1 signed)
__host__ __device__ __forceinline__ uint32_t tc_idesc(uint32_t d, uint32_t a, uint32_t b, int nt) {
    return (d << 4) | (a << 7) | (b << 10) | ((uint32_t)(nt >> 3) << 17) | ((uint32_t)(kTcRows >> 4) << 24);
}
// D (tmem) = A B, + D when acc != 0; ad / bd are shared-memory matrix descriptors.  kind::i8 when I8, else kind::f16
template <bool I8>
__device__ __forceinline__ void tc_mma(uint32_t tmem, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
    if constexpr (I8)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                     :: "r"(tmem), "l"(ad), "l"(bd), "r"(idesc), "r"(acc) : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                     :: "r"(tmem), "l"(ad), "l"(bd), "r"(idesc), "r"(acc) : "memory");
}
// one arrival on *bar once every MMA this thread has issued is complete
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}

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

// Split-K: the S CTAs of a cluster share the tile of output features o0 .. o0 + 127 and batch rows n0 .. n0 + rows - 1
// (rows >= 1) and take consecutive, possibly empty, chunk ranges [c_begin, c_end) of the row length.
struct TcTile {
    uint32_t S, rank;
    int64_t o0, n0, rows;
    int c_begin, c_end;
};
// from the launch arguments (a.M rows in this launch, a.nchunks chunks of the row length) and the row tile nt
template <typename Args>
__device__ __forceinline__ TcTile tc_tile(const Args& a, int nt) {
    TcTile t;
    t.S = cluster_size();
    t.rank = cluster_rank();
    t.o0 = (int64_t)(blockIdx.x / t.S) * kTcRows;
    t.n0 = (int64_t)blockIdx.y * nt;
    t.rows = a.M - t.n0 < nt ? a.M - t.n0 : nt;
    t.c_begin = (int)((int64_t)a.nchunks * t.rank / t.S);
    t.c_end = (int)((int64_t)a.nchunks * (t.rank + 1) / t.S);
    return t;
}

// The epilogue: warp w reads TMEM lanes 32 (w % 4) .. + 31, one output feature (tile row r) per thread, and column blocks
// of 16 batch rows alternate between warps w and w + 4.  Ranks >= 1 park their partial sums in their idle stage memory
// `part` as [batch row][feature]; after the cluster barrier rank 0 adds them to its own in rank order.  Acc is float
// (added with __fadd_rn: the order fixes the bits) or int32_t (added with wrap-around: the sum is exact).
struct TcEpilogue {
    uint32_t taddr, part;       // TMEM address of this thread's lane, the parked partial sums
    int r, cb0, nblocks;        // tile row; column blocks cb0, cb0 + 2, .. < nblocks
    bool have;                  // the CTA had a chunk (else its accumulator was never written and reads as zeros)
};
// every thread, once the last MMA has completed
__device__ __forceinline__ TcEpilogue tc_epilogue(const TcTile& t, int nt, uint32_t tmem, uint32_t part, int tid) {
    const int warp = tid >> 5, lane = tid & 31;
    TcEpilogue e;
    e.r = 32 * (warp & 3) + lane;
    e.part = part;
    e.taddr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
    e.cb0 = warp >> 2;
    e.nblocks = nt / 16;
    e.have = t.c_begin < t.c_end;
    return e;
}
__device__ __forceinline__ float acc_add(float x, float y) { return __fadd_rn(x, y); }
__device__ __forceinline__ int32_t acc_add(int32_t x, int32_t y) { return (int32_t)((uint32_t)x + (uint32_t)y); }

// column block cb of this thread's lane of the accumulator
template <typename Acc>
__device__ __forceinline__ void tmem_block(const TcEpilogue& e, int cb, Acc* v) {
    if (e.have) {
        uint32_t u[16];
        tmem_ld16(e.taddr + 16 * cb, u);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if constexpr (std::is_same<Acc, float>::value) v[j] = __uint_as_float(u[j]);
            else v[j] = (int32_t)u[j];
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0;
    }
}
// every thread: ranks >= 1 park their partial sums, then the cluster barrier after which rank 0 may read them
template <typename Acc>
__device__ __forceinline__ void splitk_park(const TcEpilogue& e, const TcTile& t) {
    if (t.rank != 0) {
        for (int cb = e.cb0; cb < e.nblocks; cb += 2) {
            Acc v[16];
            tmem_block(e, cb, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const uint32_t addr = e.part + (uint32_t)(((cb * 16 + j) * kTcRows + e.r) * 4);
                if constexpr (std::is_same<Acc, float>::value) asm volatile("st.shared.f32 [%0], %1;" :: "r"(addr), "f"(v[j]) : "memory");
                else asm volatile("st.shared.s32 [%0], %1;" :: "r"(addr), "r"(v[j]) : "memory");
            }
        }
    }
    __syncwarp();
    cluster_sync();
}
// rank 0: column block cb of the whole sum, its own partial sum first and then those of ranks 1 .. S-1
template <typename Acc>
__device__ __forceinline__ void splitk_sum(const TcEpilogue& e, const TcTile& t, int cb, Acc* v) {
    tmem_block(e, cb, v);
    for (uint32_t p = 1; p < t.S; ++p) {
        const uint32_t base = peer_addr(e.part + (uint32_t)((cb * 16 * kTcRows + e.r) * 4), p);
        Acc pv[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) pv[j] = ld_peer<Acc>(base + j * kTcRows * 4);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = acc_add(v[j], pv[j]);
    }
}
// every thread, after rank 0's sums: the peers' partial sums stay in place until rank 0 has read them
__device__ __forceinline__ void splitk_release() { __syncwarp(); cluster_sync(); }

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
// batch rows per CTA: M split evenly into tiles of at most max_nt rows, rounded up to a multiple of 16
inline int32_t tc_row_tile(int64_t M, int64_t max_nt) {
    const int64_t ntiles = (M + max_nt - 1) / max_nt, per = (M + ntiles - 1) / ntiles;
    return (int32_t)((per + 15) / 16 * 16);
}
// a ring of `stages` stages, + 1024 bytes to align them, and at least the TMEM floor
inline size_t tc_ring_smem(size_t stages, size_t stage_bytes, uint32_t tmem_cols) {
    return std::max(stages * stage_bytes + 1024, tmem_smem_floor(tmem_cols));
}
inline int sm_count(int* sms) {
    int dev = 0, rc = cuda_rc(cudaGetDevice(&dev));
    return rc ? rc : cuda_rc(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
}
// M rows in launches of at most 65535 row tiles (grid.y's limit); grid.x is S CTAs (one cluster) per feature tile.
// set_rows(b, m0, m) points b, a copy of a, at rows m0 .. m0 + m - 1.
template <typename Args, typename SetRows>
int tc_launch_rows(void (*kernel)(Args), const Args& a, int64_t M, int nt, int64_t tiles, int64_t S, size_t smem,
                   cudaStream_t st, SetRows set_rows) {
    const int64_t rows_per_launch = (int64_t)65535 * nt;
    for (int64_t m0 = 0; m0 < M; m0 += rows_per_launch) {
        Args b = a;
        const int64_t m = M - m0 < rows_per_launch ? M - m0 : rows_per_launch;
        set_rows(b, m0, m);
        const dim3 grid((unsigned)(tiles * S), (unsigned)((m + nt - 1) / nt));
        pdl_plan_launch(st, nullptr, 0, nullptr, 0);                        // ranges "unknown": late order for the successor
        if (const int rc = launch_planned_cluster(kernel, grid, (unsigned)S, smem, st, b)) return rc;
    }
    return 0;
}

}  // namespace mctq
