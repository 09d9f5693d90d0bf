// mctq_packed_gemm.cu -- y = x @ W^T + b straight from packed codes on the tensor cores (tcgen05 MMA, kind::f16), for the
// batched row counts (9 to a few hundred) of batched decode, speculative decoding and short prefills.  The batched mode of
// packed nn.Linear wrappers (pytorch/packed_weights.py) calls it above the row limit of mctq_packed_linear.cu.
//
// W is the rebuilt weight of mctq_unpack.cu, [out][in] row-major.  Every operand the tensor cores see is exact, so the only
// rounding is that of the f32 accumulation (and of the epilogue):
//   affine, bf16 / f16: A = T((q - zp_c) * s_c), the rebuilt weight itself;  B = x;                  y = acc (+ b)
//   affine, f32:        A = q - zp_c in bf16 (exact for |q - zp| <= 256);     B = x0, x1, x2;         y = acc * s_c (+ b)
//   LUT, f32:           A = q_idx in bf16 (checked exact on the host);        B = x0, x1, x2;         y = acc * thr_c (+ b)
// where x = x0 + x1 + x2 splits an f32 x into three bf16 terms by truncation (exact for finite x down to bf16's subnormal
// grain; non-finite x gives x0 = x, x1 = x2 = 0).  The three terms run as three MMAs into the same accumulator.
//
// Shape (A and B swapped against the usual GEMM): output features are the MMA's M (128 per CTA), batch rows its N (nt, a
// multiple of 16 up to 256 (16-bit x) / 128 (f32 x); more rows run as further CTAs along grid.y).  A CTA walks its share of
// the row length in chunks of 64: all 256 threads load the codes (and x) of the next chunk while they decode the current
// one into a ring of kStages shared-memory stages (K-major, 128-byte swizzle), thread 0 issues the chunk's MMAs and commits
// them onto the stage's mbarrier, which releases the stage.  The accumulator [128 x nt] f32 lives in tensor memory.
// Split-K: the S CTAs of a thread-block cluster share one 128-row tile and take consecutive chunk ranges; ranks 1..S-1
// leave their partial sums in their shared memory and rank 0 adds them to its own in rank order (distributed shared
// memory), so the result is deterministic with no workspace.  The epilogue (tcgen05.ld) gives each thread one output feature,
// so stores of consecutive lanes coalesce.  TMEM, MMA issue, split-K tile and reduction and the launches over row ranges are
// the frame of mctq_tcgen05.cuh, shared with mctq_packed_igemm.cu; this file owns the decode loop, the split policy and the
// epilogue arithmetic.
#include <type_traits>

#include "mctq_tcgen05.cuh"

namespace mctq {

constexpr int kChunk = 64;              // elements of the row length per stage (one 128-byte swizzle row of bf16 / f16)
constexpr int kStages = 3;
constexpr int kMaxSplit = 8;            // portable cluster size

struct GemmArgs {
    const uint8_t* codes;
    const void* x;
    const void* bias;            // or null
    void* y;
    const float* scale;          // affine: scale[C]; LUT: thr[C]
    const int32_t* zp;           // affine: zp[C]
    int64_t M;                   // rows of x / y in this launch
    int32_t N, K;                // out_features, in_features
    int32_t per_channel, is_signed;
    int32_t nt;                  // batch rows per CTA: multiple of 16, <= 256
    int32_t nchunks;             // ceil(K / kChunk)
    uint32_t tmem_cols;          // power of two >= max(32, nt)
    int32_t fast_codes, fast_x;  // vector loads (K % 8 == 0 and aligned bases)
    float quot[256];             // LUT quotients (bf16-exact; entries past the table's K are 0)
};

// x0 + x1 + x2 == x (bf16 terms by truncation; exact for finite x above bf16's subnormal grain), x1 = x2 = 0 for inf / NaN
__device__ __forceinline__ void split3(float x, float& x0, float& x1, float& x2) {
    if (!isfinite(x)) { x0 = x; x1 = 0.0f; x2 = 0.0f; return; }
    x0 = __uint_as_float(__float_as_uint(x) & 0xFFFF0000u);
    const float r = __fsub_rn(x, x0);
    x1 = __uint_as_float(__float_as_uint(r) & 0xFFFF0000u);
    x2 = __fsub_rn(r, x1);
}

template <int KIND, typename T>
__global__ void __launch_bounds__(kThreads, 2) packed_gemm_kernel(const __grid_constant__ GemmArgs a) {
    constexpr bool LUT = pack_is_lut(KIND);
    constexpr int CODE = pack_code_mode(KIND);
    constexpr int RAW = CodeVec<CODE, 8>::kWords;                        // 32-bit code words per 8 elements
    constexpr bool F32X = std::is_same<T, float>::value;
    constexpr bool FACTOR = LUT || F32X;
    constexpr int TERMS = F32X ? 3 : 1;
    using OT = typename std::conditional<std::is_same<T, __half>::value, __half, __nv_bfloat16>::type;   // operand type
    constexpr int XW = F32X ? 8 : 4;                                     // 32-bit words of x per 8 elements
    constexpr int XU = (F32X ? 128 : 256) * 8 / kThreads;                // max x units (row, 8-element group) per thread
    constexpr int WU = kTcRows * 8 / kThreads;                           // weight units per thread (4)
    static_assert(kThreads == 256 && WU == 4, "thread mapping");

    extern __shared__ __align__(1024) uint8_t dsm[];
    __shared__ uint64_t bar_empty[kStages];
    __shared__ uint64_t bar_done;
    __shared__ uint32_t tmem_slot;
    __shared__ float sm_q[LUT ? 256 : 1];

    const int tid = threadIdx.x, warp = tid >> 5;
    const int nt = a.nt;
    const uint32_t a_bytes = kTcRows * 128, b_bytes = (uint32_t)nt * 128, stage_bytes = a_bytes + TERMS * b_bytes;
    const uint32_t sbase = (smem_u32(dsm) + 1023u) & ~1023u;             // swizzle atoms need 1024-byte alignment

    pdl_wait();                 // x may be the output of the previous launch; TMEM is taken only after the wait
    pdl_launch_dependents();
    tmem_alloc(warp, &tmem_slot, a.tmem_cols);
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) mbar_init(&bar_empty[s], 1);
        mbar_init(&bar_done, 1);
    }
    if constexpr (LUT) {
        for (int i = tid; i < 256; i += kThreads) sm_q[i] = a.quot[i];
    }
    const uint32_t tmem = tmem_address(&tmem_slot);
    const LutCodeOp lut{a.scale, sm_q};

    const int64_t N = a.N, K = a.K;
    const TcTile tile = tc_tile(a, nt);
    const int64_t o0 = tile.o0, rows = tile.rows;
    const int c_begin = tile.c_begin, c_end = tile.c_end;

    // weight units of this thread: rows wr[u] = tid / 8 + 32 u, 8-element group wj = tid % 8 of every chunk
    const int wj = tid & 7;
    AffineCodeOp::Param prm[WU];
#pragma unroll
    for (int u = 0; u < WU; ++u) {
        const int64_t o = o0 + (tid >> 3) + 32 * u;
        const uint32_t c = a.per_channel ? (uint32_t)(o < N ? o : N - 1) : 0u;
        prm[u].s = LUT ? 0.0f : __ldg(a.scale + c);
        prm[u].zp = LUT ? 0 : __ldg(a.zp + c);
    }
    const T* __restrict__ xg = reinterpret_cast<const T*>(a.x) + tile.n0 * K;
    const int xunits = nt * 8;

    using WRaw = uint32_t[WU][RAW];
    using XRaw = uint32_t[XU][XW];
    auto load_w = [&](int c, WRaw& wraw) {
#pragma unroll
        for (int u = 0; u < WU; ++u) {
            const int64_t o = o0 + (tid >> 3) + 32 * u, k = (int64_t)c * kChunk + 8 * wj;
#pragma unroll
            for (int w = 0; w < RAW; ++w) wraw[u][w] = 0;
            if (o >= N || k >= K) continue;
            const int64_t g = o * K + k;
            if (a.fast_codes) {                                          // a whole, aligned 8-element vector
                load_code_vec<CODE, 8>(a.codes, g, g + 8, wraw[u]);
            } else {
                uint32_t t[RAW] = {};                                    // (dynamically indexed: kept apart from wraw)
                load_code_elems<CODE, 8>(a.codes, g, K - k < 8 ? (int)(K - k) : 8, t);
#pragma unroll
                for (int w = 0; w < RAW; ++w) wraw[u][w] = t[w];
            }
        }
    };
    auto load_x = [&](int c, XRaw& xraw) {
#pragma unroll
        for (int i = 0; i < XU; ++i) {
            const int unit = tid + i * kThreads;
            const int64_t n = unit >> 3, k = (int64_t)c * kChunk + 8 * (unit & 7);
#pragma unroll
            for (int w = 0; w < XW; ++w) xraw[i][w] = 0;
            if (unit >= xunits || n >= rows || k >= K) continue;
            const T* p = xg + n * K + k;
            if (a.fast_x) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
                xraw[i][0] = v.x; xraw[i][1] = v.y; xraw[i][2] = v.z; xraw[i][3] = v.w;
                if constexpr (F32X) {
                    const uint4 v2 = __ldg(reinterpret_cast<const uint4*>(p) + 1);
                    xraw[i][4] = v2.x; xraw[i][5] = v2.y; xraw[i][6] = v2.z; xraw[i][7] = v2.w;
                }
            } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    if (k + e >= K) break;
                    if constexpr (F32X) xraw[i][e] = __float_as_uint(p[e]);
                    else xraw[i][e >> 1] |= (uint32_t)(*reinterpret_cast<const uint16_t*>(p + e)) << (16 * (e & 1));
                }
            }
        }
    };
    auto store_chunk = [&](int c, uint32_t st, const WRaw& wraw, const XRaw& xraw) {
#pragma unroll
        for (int u = 0; u < WU; ++u) {
            const int r = (tid >> 3) + 32 * u;
            const int64_t o = o0 + r, k = (int64_t)c * kChunk + 8 * wj;
            float v[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int q = code_at<CODE, 8>(wraw[u], e, LUT ? 0 : a.is_signed);
                float w;
                if constexpr (LUT) w = lut.level(q);
                else if constexpr (FACTOR) w = AffineCodeOp::level(q, prm[u]);
                else w = AffineCodeOp::value(q, prm[u]);
                v[e] = (o < N && k + e < K) ? w : 0.0f;               // the tail of the row and rows past N are zero
            }
            uint32_t p[4];
            Pack<OT, 8>::pack(v, p);
            st_shared_v4(st + sw128_off(r, wj), p);
        }
#pragma unroll
        for (int i = 0; i < XU; ++i) {
            const int unit = tid + i * kThreads;
            if (unit >= xunits) continue;
            const uint32_t off = a_bytes + sw128_off(unit >> 3, unit & 7);
            if constexpr (F32X) {
                float t[3][8];
#pragma unroll
                for (int e = 0; e < 8; ++e) split3(__uint_as_float(xraw[i][e]), t[0][e], t[1][e], t[2][e]);
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    uint32_t p[4];
                    Pack<__nv_bfloat16, 8>::pack(t[s], p);
                    st_shared_v4(st + off + s * b_bytes, p);
                }
            } else {
                st_shared_v4(st + off, xraw[i]);
            }
        }
    };

    // f32 accumulator, A and B bf16 (1) or f16 (0)
    constexpr uint32_t ab = std::is_same<OT, __half>::value ? 0u : 1u;
    const uint32_t idesc = tc_idesc(1u, ab, ab, nt);

    // chunk c: wait for its stage, decode it from registers into the stage, issue its MMAs
    auto run_chunk = [&](int c, const WRaw& wraw, const XRaw& xraw) {
        const int i = c - c_begin, s = i % kStages;
        const uint32_t st = sbase + (uint32_t)s * stage_bytes;
        if (i >= kStages) mbar_wait(&bar_empty[s], (uint32_t)((i / kStages - 1) & 1));
        store_chunk(c, st, wraw, xraw);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> tensor-core reads
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
#pragma unroll
            for (int ks = 0; ks < kChunk / 16; ++ks) {
                const uint64_t ad = sw128_desc(st + 32 * ks);
#pragma unroll
                for (int t = 0; t < TERMS; ++t) {
                    const uint64_t bd = sw128_desc(st + a_bytes + t * b_bytes + 32 * ks);
                    tc_mma<false>(tmem, ad, bd, idesc, (i > 0 || ks > 0 || t > 0) ? 1u : 0u);
                }
            }
            tc_commit(&bar_empty[s]);
            if (c + 1 == c_end) tc_commit(&bar_done);
        }
    };
    // two register sets: the loads of chunk c + 1 are in flight while chunk c is decoded
    WRaw w0, w1;
    XRaw x0, x1;
    if (c_begin < c_end) { load_w(c_begin, w0); load_x(c_begin, x0); }
    for (int c = c_begin; c < c_end; c += 2) {
        if (c + 1 < c_end) { load_w(c + 1, w1); load_x(c + 1, x1); }
        run_chunk(c, w0, x0);
        if (c + 1 < c_end) {
            if (c + 2 < c_end) { load_w(c + 2, w0); load_x(c + 2, x0); }
            run_chunk(c + 1, w1, x1);
        }
    }
    if (c_begin < c_end) mbar_wait(&bar_done, 0);
    tc_fence_after();

    // epilogue (one output feature o per thread): the split-K sum in f32, added in rank order, then the factor and the bias
    const TcEpilogue e = tc_epilogue(tile, nt, tmem, sbase, tid);
    const int64_t o = o0 + e.r;
    splitk_park<float>(e, tile);
    if (tile.rank == 0) {
        const float f = FACTOR && o < N ? __ldg(a.scale + (a.per_channel ? o : 0)) : 1.0f;
        const float b = a.bias && o < N ? to_f32<T>(reinterpret_cast<const T*>(a.bias)[o]) : 0.0f;
        T* y = reinterpret_cast<T*>(a.y) + tile.n0 * N;
        for (int cb = e.cb0; cb < e.nblocks; cb += 2) {
            float v[16];
            splitk_sum(e, tile, cb, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int64_t n = cb * 16 + j;
                if (o >= N || n >= rows) continue;
                float s = v[j];
                if (FACTOR) s = __fmul_rn(s, f);
                if (a.bias) s = __fadd_rn(s, b);
                y[n * N + o] = from_f32<T>(s);
            }
        }
    }
    splitk_release();
    tmem_dealloc(warp, tmem, a.tmem_cols);
}

}  // namespace mctq

using namespace mctq;

namespace {

template <int KIND, typename T>
int launch_gemm(GemmArgs a, cudaStream_t st) {
    constexpr int TERMS = std::is_same<T, float>::value ? 3 : 1;
    const int64_t M = a.M;
    const int max_nt = TERMS == 3 ? 128 : 256;
    const int64_t ntiles = (M + max_nt - 1) / max_nt;
    a.nt = tc_row_tile(M, max_nt);
    a.nchunks = (int32_t)((a.K + kChunk - 1) / kChunk);
    a.tmem_cols = tmem_columns(a.nt);
    const int64_t tiles = (a.N + kTcRows - 1) / kTcRows;
    const size_t smem = tc_ring_smem(kStages, (size_t)kTcRows * 128 + (size_t)TERMS * a.nt * 128, a.tmem_cols);
    auto kernel = packed_gemm_kernel<KIND, T>;
    int rc = ensure_smem(kernel, smem);                                     // per device: set on every launch
    if (rc) return rc;
    // split-K: about two CTAs per SM (measured faster than one wave of longer CTAs), at least one chunk per CTA
    int sms = 0;
    if ((rc = sm_count(&sms))) return rc;
    int64_t S = (2 * (int64_t)sms + tiles * ntiles - 1) / (tiles * ntiles);
    S = S < 1 ? 1 : S > kMaxSplit ? kMaxSplit : S;
    if (S > a.nchunks) S = a.nchunks;
    return tc_launch_rows(kernel, a, M, a.nt, tiles, S, smem, st, [&](GemmArgs& b, int64_t m0, int64_t m) {
        b.M = m;
        b.x = reinterpret_cast<const T*>(a.x) + m0 * a.K;
        b.y = reinterpret_cast<T*>(a.y) + m0 * a.N;
    });
}

}  // namespace

extern "C" {

int mctq_packed_linear_batched(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x, int x_dtype,
                               int64_t M, const void* bias, void* y, const float* lut_quotients_host, void* stream) {
    MCTQ_NVTX("mctq_packed_linear_batched");
    if (const int rc = packed_linear_check(w, out_features, in_features, x, x_dtype, M, y)) return rc;
    const bool lut = pack_is_lut(w->kind);
    GemmArgs a;
    memset(&a, 0, sizeof(a));
    if (lut) {
        if (!lut_quotients_host) return MCTQ_E_LUT;
        for (int k = 0; k < w->K; ++k) {
            uint32_t bits;
            memcpy(&bits, lut_quotients_host + k, 4);
            if (bits & 0xFFFFu) return MCTQ_E_LUT;                            // not exact in bf16
            a.quot[k] = lut_quotients_host[k];
        }
    }
    if (M == 0) return 0;
    a.codes = reinterpret_cast<const uint8_t*>(w->codes);
    a.x = x;
    a.bias = bias;
    a.y = y;
    a.scale = w->scale;
    a.zp = lut ? nullptr : w->zp;
    a.M = M;
    a.N = (int32_t)out_features;
    a.K = (int32_t)in_features;
    a.per_channel = w->C != 1;
    a.is_signed = lut ? 0 : (w->is_signed ? 1 : 0);
    const uintptr_t cp = reinterpret_cast<uintptr_t>(w->codes);
    a.fast_codes = in_features % 8 == 0 && (cp & (pack_is_int4(w->kind) ? 3u : 7u)) == 0;
    a.fast_x = in_features % 8 == 0 && aligned16(x);
    cudaStream_t st = (cudaStream_t)stream;
    return dispatch_packed(w->kind, x_dtype, [&](auto kind, auto type) {
        return launch_gemm<decltype(kind)::value, typename decltype(type)::type>(a, st);
    });
}

}  // extern "C"
