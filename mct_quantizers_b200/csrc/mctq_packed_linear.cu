// mctq_packed_linear.cu -- y = x @ W^T + b computed straight from packed codes (affine int8 / int4 codes, LUT indices), for the
// small row counts of decode-style inference: W is never built in memory.  The fused mode of packed nn.Linear wrappers
// (pytorch/packed_weights.py) calls it instead of mctq_unpack_multi followed by F.linear.
//
// W is the rebuilt weight of mctq_unpack.cu, [out][in] row-major, parameters per tensor or per output row.  Accumulation is in
// f32 with __fmaf_rn; the per-row factor is applied once per row where that keeps the error within one f32 rounding per term:
//   LUT (f32 out):      acc = sum_k x_k * q_idx(k);                 y = acc * thr_c (+ b)
//   affine, f32 out:    acc = sum_k x_k * (q_k - zp_c);             y = acc * s_c (+ b)
//   affine, bf16 / f16: acc = sum_k x_k * T((q_k - zp_c) * s_c);    y = acc (+ b)       (T-rounded weight: no factoring)
// and y is rounded once to x's dtype.  The reduction order is fixed (per-thread sequential, xor butterfly over the warp, warps
// 0..7 in order), so two runs give the same bits.
//
// Loop shape: a warp owns R output rows and walks their length in 8-byte code vectors (16 int4 / 8 int8 elements) per lane,
// so every x value a lane loads serves R rows; the CTA's 8 warps are 8 / S row groups x S segments of the row length.  That
// split-K (S = 2) doubles the CTAs of a layer, so that 4096-row layers fill the 148 SMs; the S partial sums of a row meet in
// shared memory in segment order.
// FAST: rows start on 8-byte code boundaries and x rows on 16 bytes (in % 16 for int4, % 8 for int8, aligned bases); every
// other shape (odd `in`, an int4 row that starts in a high nibble) loads codes and x element by element with the row tail
// masked.
#include <type_traits>

#include "mctq_common.cuh"

namespace mctq {

struct LinearArgs {
    const uint8_t* codes;
    const void* x;
    const void* bias;            // or null
    void* y;
    const float* scale;          // affine: scale[C]; LUT: thr[C]
    const int32_t* zp;           // affine: zp[C]
    const float* quot;           // LUT: q_k, nq entries
    int64_t M;
    int32_t N, K;                // out_features, in_features
    int32_t per_channel, is_signed, nq;
};

constexpr int kLinWarps = kThreads / 32;

template <int MT> struct LinRows { static constexpr int value = MT <= 4 ? 4 : 2; };
constexpr int kLinSplit = 2;                                     // S: warps that share one row group
constexpr int kLinGroups = kLinWarps / kLinSplit;

template <int KIND, typename T, int MT, bool FAST>
__global__ void __launch_bounds__(kThreads, MT >= 8 ? 1 : 2) packed_linear_kernel(const __grid_constant__ LinearArgs a) {
    constexpr bool LUT = pack_is_lut(KIND);
    constexpr int CODE = pack_code_mode(KIND);
    constexpr int EPW = CODE == MCTQ_CODES_INT4 ? 8 : 4;        // elements per 32-bit word of codes
    constexpr int EPV = 2 * EPW;                                 // elements per 8-byte vector
    constexpr int NQ = pack_max_k(KIND);
    constexpr bool FACTOR = LUT || std::is_same<T, float>::value;
    constexpr int R = LinRows<MT>::value;
    __shared__ float sm_q[LUT ? NQ : 1];
    __shared__ float sm_red[kLinWarps][R * MT];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = warp / kLinSplit, seg = warp % kLinSplit;

    pdl_wait();
    pdl_launch_dependents();
    if constexpr (LUT) {
        for (int i = threadIdx.x; i < NQ; i += kThreads) sm_q[i] = i < a.nq ? __ldg(a.quot + i) : 0.0f;
        __syncthreads();
    }
    const LutCodeOp lut{a.scale, sm_q};
    const int64_t N = a.N, K = a.K;
    const int64_t n0 = ((int64_t)blockIdx.x * kLinGroups + grp) * R;
    AffineCodeOp::Param prm[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int64_t n = n0 + r < N ? n0 + r : N - 1;
        const uint32_t c = a.per_channel ? (uint32_t)n : 0u;
        prm[r].s = __ldg(a.scale + c);
        prm[r].zp = LUT ? 0 : __ldg(a.zp + c);
    }
    const T* __restrict__ x = reinterpret_cast<const T*>(a.x);
    const int64_t nvec = (K + EPV - 1) / EPV;

    for (int64_t m0 = (int64_t)blockIdx.y * MT; m0 < a.M; m0 += (int64_t)gridDim.y * MT) {
        float acc[R][MT];
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int m = 0; m < MT; ++m) acc[r][m] = 0.0f;

        for (int64_t v = seg * 32 + lane; v < nvec; v += 32 * kLinSplit) {
            const int64_t e = v * EPV;
            // codes of the R rows: every load is issued before the first use
            uint32_t raw[R][2];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                raw[r][0] = raw[r][1] = 0;
                if (n0 + r >= N) continue;
                const int64_t g = (n0 + r) * K + e;                       // element index of the vector's first code
                if (FAST) {
                    const uint2 w = ld_stream(reinterpret_cast<const uint2*>(a.codes + (CODE == MCTQ_CODES_INT4 ? g >> 1 : g)));
                    raw[r][0] = w.x;
                    raw[r][1] = w.y;
                } else {
                    const int cnt = K - e < EPV ? (int)(K - e) : EPV;
                    load_code_elems<CODE, EPW>(a.codes, g, cnt < EPW ? cnt : EPW, &raw[r][0]);
                    if (cnt > EPW) load_code_elems<CODE, EPW>(a.codes, g + EPW, cnt - EPW, &raw[r][1]);
                }
            }
#pragma unroll
            for (int kk = 0; kk < EPV / 4; ++kk) {                      // 4 elements at a time
                const int64_t eb = e + 4 * kk;
                float xv[MT][4];
#pragma unroll
                for (int m = 0; m < MT; ++m) {
                    const int64_t row = m0 + m;
                    if (row >= a.M) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) xv[m][j] = 0.0f;
                    } else if (FAST) {
                        const T* p = x + row * K + eb;
                        if constexpr (sizeof(T) == 4) {
                            const float4 f = __ldg(reinterpret_cast<const float4*>(p));
                            xv[m][0] = f.x; xv[m][1] = f.y; xv[m][2] = f.z; xv[m][3] = f.w;
                        } else {
                            const uint2 w = __ldg(reinterpret_cast<const uint2*>(p));
                            const uint32_t ww[2] = {w.x, w.y};
                            Pack<T, 4>::unpack(ww, xv[m]);
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) xv[m][j] = eb + j < K ? to_f32<T>(x[row * K + eb + j]) : 0.0f;
                    }
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int k = 4 * kk + j;
                        const int q = code_at<CODE, EPW>(&raw[r][k / EPW], k % EPW, LUT ? 0 : a.is_signed);
                        float w;
                        if constexpr (LUT) w = lut.level(q);
                        else if constexpr (FACTOR) w = AffineCodeOp::level(q, prm[r]);
                        else w = to_f32<T>(from_f32<T>(AffineCodeOp::value(q, prm[r])));
#pragma unroll
                        for (int m = 0; m < MT; ++m) acc[r][m] = __fmaf_rn(xv[m][j], w, acc[r][m]);
                    }
                }
            }
        }

        // fixed-order reduction: xor butterfly inside the warp, then the segments of a row group in order
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int m = 0; m < MT; ++m) {
                float s = acc[r][m];
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, off));
                if (lane == 0) sm_red[warp][r * MT + m] = s;
            }
        __syncthreads();
        if (threadIdx.x < kLinGroups * R * MT) {
            const int g = threadIdx.x / (R * MT), i = threadIdx.x % (R * MT);
            const int r = i / MT, m = i % MT;
            const int64_t n = ((int64_t)blockIdx.x * kLinGroups + g) * R + r, row = m0 + m;
            if (n < N && row < a.M) {
                float s = sm_red[g * kLinSplit][i];
#pragma unroll
                for (int w = 1; w < kLinSplit; ++w) s = __fadd_rn(s, sm_red[g * kLinSplit + w][i]);
                if (FACTOR) s = __fmul_rn(s, __ldg(a.scale + (a.per_channel ? n : 0)));
                if (a.bias) s = __fadd_rn(s, to_f32<T>(reinterpret_cast<const T*>(a.bias)[n]));
                reinterpret_cast<T*>(a.y)[row * N + n] = from_f32<T>(s);
            }
        }
        __syncthreads();
    }
}

}  // namespace mctq

using namespace mctq;

namespace {

template <int KIND, typename T, int MT>
int launch_linear_mt(const LinearArgs& a, bool fast, cudaStream_t st) {
    constexpr int R = LinRows<MT>::value;
    const int64_t tiles = (a.M + MT - 1) / MT;
    const int64_t rows_per_cta = (int64_t)kLinGroups * R;
    const dim3 grid((unsigned)((a.N + rows_per_cta - 1) / rows_per_cta), (unsigned)(tiles < 65535 ? tiles : 65535));
    // ranges "unknown": the successor of this launch takes the late dependent-launch order
    return fast ? launch_streaming(packed_linear_kernel<KIND, T, MT, true>, grid, 0, st, a)
                : launch_streaming(packed_linear_kernel<KIND, T, MT, false>, grid, 0, st, a);
}

template <int KIND, typename T>
int launch_linear_typed(const LinearArgs& a, bool fast, cudaStream_t st) {
    if (a.M == 1) return launch_linear_mt<KIND, T, 1>(a, fast, st);
    if (a.M == 2) return launch_linear_mt<KIND, T, 2>(a, fast, st);
    if (a.M <= 4) return launch_linear_mt<KIND, T, 4>(a, fast, st);
    return launch_linear_mt<KIND, T, 8>(a, fast, st);
}

}  // namespace

extern "C" {

int mctq_packed_linear(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x, int x_dtype,
                       int64_t M, const void* bias, void* y, void* stream) {
    MCTQ_NVTX("mctq_packed_linear");
    if (const int rc = packed_linear_check(w, out_features, in_features, x, x_dtype, M, y)) return rc;
    if (M == 0) return 0;
    const bool lut = pack_is_lut(w->kind);
    LinearArgs a;
    memset(&a, 0, sizeof(a));
    a.codes = reinterpret_cast<const uint8_t*>(w->codes);
    a.x = x;
    a.bias = bias;
    a.y = y;
    a.scale = w->scale;
    a.zp = lut ? nullptr : w->zp;
    a.quot = lut ? w->lut_quotients : nullptr;
    a.M = M;
    a.N = (int32_t)out_features;
    a.K = (int32_t)in_features;
    a.per_channel = w->C != 1;
    a.is_signed = lut ? 0 : (w->is_signed ? 1 : 0);
    a.nq = lut ? w->K : 0;
    const int64_t epv = pack_is_int4(w->kind) ? 16 : 8;
    const bool fast = in_features % epv == 0 && aligned16(w->codes) && aligned16(x);
    cudaStream_t st = (cudaStream_t)stream;
    return dispatch_packed(w->kind, x_dtype, [&](auto kind, auto type) {
        return launch_linear_typed<decltype(kind)::value, typename decltype(type)::type>(a, fast, st);
    });
}

}  // extern "C"
