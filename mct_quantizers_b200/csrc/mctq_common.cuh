// mctq_common.cuh -- shared device utilities of libmctq_sm100 (see mctq_affine.cu / mctq_lut.cu / mctq_host.cu).
// Build: mct_quantizers_b200/build.py
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo --fmad=false ... (one object per .cu, linked into one .so)
// (--fmad=false: the reference never contracts a multiply-add; the fused operations these kernels need are
//  written explicitly with __fmaf_rn, which the flag does not touch.)
//
// All kernels are HBM-bound streaming kernels (no tensor cores): one CTA = one tile of kThreads * UNROLL vectors,
// every load of the tile is issued before the first use, per-channel parameters of the rows the tile touches are
// staged in shared memory while the loads are in flight.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <atomic>
#include <type_traits>
#include <utility>

#include "mctq.h"

namespace mctq {

constexpr int kThreads = 256;

// process-wide state (defined in mctq_host.cu)
extern std::atomic<int64_t> g_launches;
extern int g_pdl;           // programmatic dependent launch for the streaming kernels (mctq_set_tuning key 3)
extern int g_nvtx;          // NVTX ranges around the C-ABI compute entry points (mctq_set_tuning key 9 / MCTQ_TUNE=9=1; off by default)

enum ChMode { CH_PT = 0, CH_VEC = 1, CH_ELEM = 2, CH_LAST = 3 };

// ------------------------------------------------------------------------------------------ small utils
struct FastDiv {   // floor(u / d) for 0 <= u < 2^31, 1 <= d < 2^31  (round-up multiplier, Granlund-Montgomery)
    uint32_t mul, shift, d;
};
inline FastDiv make_fastdiv(uint32_t d) {
    FastDiv f;
    f.d = d;
    uint32_t s = 0;
    while (s < 32 && (1ull << s) < d) ++s;
    f.shift = s;
    f.mul = (uint32_t)((((1ull << 32) * ((1ull << s) - d)) / d) + 1);
    return f;
}
__device__ __forceinline__ uint32_t fdiv_u32(uint32_t u, const FastDiv& f) {
    return (__umulhi(u, f.mul) + u) >> f.shift;
}

template <int BYTES> struct Vec;
template <> struct Vec<16> { using type = uint4; };
template <> struct Vec<8> { using type = uint2; };
template <> struct Vec<4> { using type = uint32_t; };
template <> struct Vec<2> { using type = uint16_t; };
template <> struct Vec<1> { using type = uint8_t; };

// streaming loads: read-only path, do not allocate in L1 (every byte is touched exactly once)
__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ld_stream(const uint2* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(uint4* p, const uint4& v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_stream(uint2* p, const uint2& v) {
    asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" :: "l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream(uint32_t* p, const uint32_t& v) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_stream(uint16_t* p, const uint16_t& v) {
    asm volatile("st.global.L1::no_allocate.u16 [%0], %1;" :: "l"(p), "h"(v) : "memory");
}

// 256-bit streaming store (sm_100: STG.256): one instruction covers 32 contiguous bytes per lane, so a warp writes 1 KB of
// contiguous memory -- two 128-bit stores per lane at a 32-byte lane stride would half-fill every sector twice
__device__ __forceinline__ void st_stream256(void* p, const uint32_t* w) {
    asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
}
__device__ __forceinline__ void ld_stream256(const void* p, uint32_t* w) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "l"(p));
}

// element <-> f32
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

// unpack a register-resident vector of V elements of T (V * sizeof(T) bytes, as 32-bit words) to floats
template <typename T, int V> struct Pack;
template <int V> struct Pack<float, V> {
    static constexpr int kWords = V;
    __device__ static __forceinline__ void unpack(const uint32_t* w, float* f) {
#pragma unroll
        for (int i = 0; i < V; ++i) f[i] = __uint_as_float(w[i]);
    }
    __device__ static __forceinline__ void pack(const float* f, uint32_t* w) {
#pragma unroll
        for (int i = 0; i < V; ++i) w[i] = __float_as_uint(f[i]);
    }
};
template <int V> struct Pack<__nv_bfloat16, V> {
    static constexpr int kWords = V / 2;
    __device__ static __forceinline__ void unpack(const uint32_t* w, float* f) {
#pragma unroll
        for (int i = 0; i < V / 2; ++i) {
            f[2 * i] = __uint_as_float(w[i] << 16);
            f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
    __device__ static __forceinline__ void pack(const float* f, uint32_t* w) {
#pragma unroll
        for (int i = 0; i < V / 2; ++i) {
            __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t*>(&h);
        }
    }
};
template <int V> struct Pack<__half, V> {
    static constexpr int kWords = V / 2;
    __device__ static __forceinline__ void unpack(const uint32_t* w, float* f) {
#pragma unroll
        for (int i = 0; i < V / 2; ++i) {
            __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
            float2 v = __half22float2(h);
            f[2 * i] = v.x;
            f[2 * i + 1] = v.y;
        }
    }
    __device__ static __forceinline__ void pack(const float* f, uint32_t* w) {
#pragma unroll
        for (int i = 0; i < V / 2; ++i) {
            __half2 h = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t*>(&h);
        }
    }
};

template <int WORDS> __device__ __forceinline__ void ld_words(const void* p, uint32_t* w);
template <> __device__ __forceinline__ void ld_words<4>(const void* p, uint32_t* w) {
    uint4 v = ld_stream(reinterpret_cast<const uint4*>(p));
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
}
template <> __device__ __forceinline__ void ld_words<2>(const void* p, uint32_t* w) {
    uint2 v = ld_stream(reinterpret_cast<const uint2*>(p));
    w[0] = v.x; w[1] = v.y;
}
template <int WORDS> __device__ __forceinline__ void st_words(void* p, const uint32_t* w);
template <> __device__ __forceinline__ void st_words<4>(void* p, const uint32_t* w) {
    st_stream(reinterpret_cast<uint4*>(p), make_uint4(w[0], w[1], w[2], w[3]));
}
template <> __device__ __forceinline__ void st_words<2>(void* p, const uint32_t* w) {
    st_stream(reinterpret_cast<uint2*>(p), make_uint2(w[0], w[1]));
}

// integer codes of one vector -> global.  INT8: V bytes; INT4: V/2 bytes (element 2j in the low nibble)
template <int V, int CODE> __device__ __forceinline__ void st_codes(void* codes, int64_t elem, const int* c) {
    if (CODE == MCTQ_CODES_INT8) {
        uint32_t w[V / 4];
#pragma unroll
        for (int i = 0; i < V / 4; ++i)
            w[i] = (uint32_t)(c[4 * i] & 0xff) | ((uint32_t)(c[4 * i + 1] & 0xff) << 8) |
                   ((uint32_t)(c[4 * i + 2] & 0xff) << 16) | ((uint32_t)(c[4 * i + 3] & 0xff) << 24);
        uint8_t* p = reinterpret_cast<uint8_t*>(codes) + elem;
        if (V == 4) st_stream(reinterpret_cast<uint32_t*>(p), w[0]);
        else st_stream(reinterpret_cast<uint2*>(p), make_uint2(w[0], w[V / 4 - 1]));
    } else if (CODE == MCTQ_CODES_INT4) {
        uint32_t w = 0;
#pragma unroll
        for (int i = 0; i < V; ++i) w |= (uint32_t)(c[i] & 0xf) << (4 * i);
        uint8_t* p = reinterpret_cast<uint8_t*>(codes) + (elem >> 1);
        if (V == 4) st_stream(reinterpret_cast<uint16_t*>(p), (uint16_t)w);
        else st_stream(reinterpret_cast<uint32_t*>(p), w);
    }
}
constexpr float kMagic = 12582912.0f;      // 1.5 * 2^23: (t + kMagic) - kMagic == rint(t) for |t| < 2^22

// (float)k for |k| < 2^22 without I2F (a quarter-rate conversion): the mantissa of 1.5 * 2^23 + k holds k
__device__ __forceinline__ float small_int_to_float(int k) { return __fsub_rn(__int_as_float(0x4B400000 + k), kMagic); }

// ------------------------------------------------------------------------------------------ consumers of codes
// The read side of the code wire format (MCTQ_CODES_INT8: one byte per element; MCTQ_CODES_INT4: two per byte, element 2j
// in the low nibble), shared by mctq_dequant_affine and the multi-tensor unpack kernels (mctq_unpack.cu).  A tile is
// kThreads x UNROLL vectors of V codes; a vector is one 32-bit / 16-bit load (V = 4) or 64-bit / 32-bit load (V = 8).
//   MODE 0  per-tensor: parameters loaded once per thread
//   MODE 1  per-channel, rows a multiple of V: one channel (one division, one parameter load) per vector
//   MODE 2  per-channel, any row length below 2^32: the vector's first channel from one 32-bit division, the following
//           elements walk (rem, c) forward
// Op turns (code, channel parameters) into the f32 value: `Param load(uint32_t c)` and `float value(int q, const Param&)`.
template <int CODE, int V> struct CodeVec {
    static constexpr int kWords = (CODE == MCTQ_CODES_INT8 && V == 8) ? 2 : 1;   // 32-bit words of codes per vector
};

// the first cnt (<= V) codes of elements [e, e + V), one byte load each: any e, including an int4 element in a high nibble;
// raw must be zeroed by the caller
template <int CODE, int V>
__device__ __forceinline__ void load_code_elems(const uint8_t* cb, int64_t e, int cnt, uint32_t* raw) {
    constexpr int RAW = CodeVec<CODE, V>::kWords;
    for (int k = 0; k < cnt; ++k) {
        const int64_t i = e + k;
        if (CODE == MCTQ_CODES_INT8) raw[(k >> 2) % RAW] |= (uint32_t)cb[i] << (8 * (k & 3));
        else raw[0] |= (uint32_t)((cb[i >> 1] >> ((i & 1) * 4)) & 0xf) << (4 * k);
    }
}

// codes of elements [e, e + V) into raw (a vector that crosses n reads only the elements below n)
template <int CODE, int V>
__device__ __forceinline__ void load_code_vec(const uint8_t* cb, int64_t e, int64_t n, uint32_t* raw) {
    constexpr int RAW = CodeVec<CODE, V>::kWords;
#pragma unroll
    for (int r = 0; r < RAW; ++r) raw[r] = 0;
    if (e + V <= n) {
        if (CODE == MCTQ_CODES_INT8) {
            if (V == 8) { const uint2 v = __ldg(reinterpret_cast<const uint2*>(cb + e)); raw[0] = v.x; raw[RAW - 1] = v.y; }
            else raw[0] = __ldg(reinterpret_cast<const uint32_t*>(cb + e));
        } else {
            if (V == 8) raw[0] = __ldg(reinterpret_cast<const uint32_t*>(cb + (e >> 1)));
            else raw[0] = __ldg(reinterpret_cast<const uint16_t*>(cb + (e >> 1)));
        }
    } else {
        load_code_elems<CODE, V>(cb, e, n - e < V ? (int)(n - e) : V, raw);
    }
}

// code k of a loaded vector, sign-extended when is_signed
template <int CODE, int V>
__device__ __forceinline__ int code_at(const uint32_t* raw, int k, int is_signed) {
    if (CODE == MCTQ_CODES_INT8) {
        const uint32_t word = raw[(k >> 2) % CodeVec<CODE, V>::kWords];
        return is_signed ? (int)(int8_t)(word >> (8 * (k & 3))) : (int)((word >> (8 * (k & 3))) & 0xffu);
    }
    const int nib = (int)((raw[0] >> (4 * k)) & 0xfu);
    return is_signed ? ((nib ^ 8) - 8) : nib;
}

// V values to y[e, e + V) as T: one 32-byte (f32, V = 8), 16-byte or 8-byte store; element stores for a vector crossing n
template <typename T, int V>
__device__ __forceinline__ void store_vec(T* y, int64_t e, int64_t n, const float* v) {
    if (e + V <= n) {
        if constexpr (sizeof(T) == 4) {
            uint32_t w[V];
#pragma unroll
            for (int k = 0; k < V; ++k) w[k] = __float_as_uint(v[k]);
            if (V == 8) st_stream256(y + e, w);
            else st_stream(reinterpret_cast<uint4*>(y + e), make_uint4(w[0], w[1], w[2], w[3]));
        } else {
            uint32_t w[V / 2];
            Pack<T, V>::pack(v, w);
            st_words<V / 2>(y + e, w);
        }
    } else {
        for (int k = 0; k < V && e + k < n; ++k) y[e + k] = from_f32<T>(v[k]);
    }
}

// one tile of a code consumer: every load of the tile is issued before the first use
template <int CODE, int MODE, int V, int UNROLL, typename T, class Op>
__device__ __forceinline__ void codes_tile(const uint8_t* cb, T* y, int64_t t0, int64_t n, int is_signed, uint32_t C,
                                           uint32_t inner, int64_t elem_offset, const FastDiv& div_inner,
                                           const FastDiv& div_C, const Op& op) {
    constexpr int RAW = CodeVec<CODE, V>::kWords;
    static_assert(V == 4 || (V == 8 && MODE != 2), "vector width");
    using Param = typename Op::Param;
    uint32_t raw[UNROLL][RAW];
#pragma unroll
    for (int j = 0; j < UNROLL; ++j)
        load_code_vec<CODE, V>(cb, t0 + (int64_t)(j * kThreads + threadIdx.x) * V, n, raw[j]);
    Param p0 = {};
    if (MODE == 0) p0 = op.load(0);
    const bool small = (uint64_t)(elem_offset + n) < (1ull << 31);
#pragma unroll
    for (int j = 0; j < UNROLL; ++j) {
        const int64_t e = t0 + (int64_t)(j * kThreads + threadIdx.x) * V;
        if (e >= n) continue;
        uint32_t c = 0, rem = 0;
        Param p = p0;
        if (MODE != 0) {
            const uint64_t g = (uint64_t)(elem_offset + e);
            if (small) {                                        // the usual case (< 2^31 elements): multiply-shift division
                const uint32_t g32 = (uint32_t)g, r = fdiv_u32(g32, div_inner);
                rem = g32 - r * inner;
                c = r - fdiv_u32(r, div_C) * C;
            } else {
                const uint64_t r = g / inner;
                rem = (uint32_t)(g - r * inner);
                c = (uint32_t)(r % C);
            }
            p = op.load(c);
        }
        // MODE 2, rows of at least one vector: the vector crosses at most one row boundary, so the parameters of the next
        // channel are fetched up front and selected per element (no divergent reloads inside the element loop)
        const bool two_rows = MODE == 2 && inner >= (uint32_t)V;
        uint32_t first_cnt = V;
        Param p1 = p;
        if (two_rows) {
            first_cnt = inner - rem;
            p1 = op.load((c + 1 == C) ? 0 : c + 1);
        }
        float out[V];
#pragma unroll
        for (int k = 0; k < V; ++k) {
            const int q = code_at<CODE, V>(raw[j], k, is_signed);
            out[k] = op.value(q, (two_rows && (uint32_t)k >= first_cnt) ? p1 : p);
            if (MODE == 2 && !two_rows) {
                if (++rem == inner) {
                    rem = 0;
                    c = (c + 1 == C) ? 0 : c + 1;
                    p = op.load(c);
                }
            }
        }
        store_vec<T, V>(y, e, n, out);
    }
}

// affine codes: y = (q - zp_c) * s_c, one f32 rounding; exact (q - zp) for |q - zp| < 2^22.  level() is the value before the
// per-channel factor, which a consumer that sums over a row (mctq_packed_linear.cu) may apply once per row instead
struct AffineCodeOp {
    struct Param { float s; int zp; };
    const float* __restrict__ scale;
    const int32_t* __restrict__ zp;
    __device__ __forceinline__ Param load(uint32_t c) const { return {__ldg(scale + c), __ldg(zp + c)}; }
    __device__ static __forceinline__ float level(int q, const Param& p) { return small_int_to_float(q - p.zp); }
    __device__ static __forceinline__ float value(int q, const Param& p) { return __fmul_rn(level(q, p), p.s); }
};

// LUT indices: y = q_idx * thr_c with the quotients q_k of the tensor's centroid list in shared memory (staged once per CTA;
// entries past K are 0, so no index of the code width can read outside the table)
struct LutCodeOp {
    using Param = float;
    const float* __restrict__ thr;
    const float* sm_q;
    __device__ __forceinline__ float load(uint32_t c) const { return __ldg(thr + c); }
    __device__ __forceinline__ float level(int q) const { return sm_q[q]; }
    __device__ __forceinline__ float value(int q, float t) const { return __fmul_rn(level(q), t); }
};

// facts of a packed-weight kind (MCTQ_PACK_*, include/mctq.h): which op decodes it, its code width, and for the LUT kinds
// the table size its indices can address (the largest K)
__host__ __device__ constexpr bool pack_is_lut(int kind) { return kind == MCTQ_PACK_LUT_U8 || kind == MCTQ_PACK_LUT_I4; }
__host__ __device__ constexpr bool pack_is_int4(int kind) { return kind == MCTQ_PACK_AFFINE_I4 || kind == MCTQ_PACK_LUT_I4; }
__host__ __device__ constexpr int pack_code_mode(int kind) { return pack_is_int4(kind) ? MCTQ_CODES_INT4 : MCTQ_CODES_INT8; }
__host__ __device__ constexpr int pack_max_k(int kind) { return pack_is_int4(kind) ? 16 : 256; }

// ------------------------------------------------------------------------------------------ channel window
// A tile covers logical elements [g0, g0 + tile) of the [outer][C][inner] view.  It touches rows
// r0 .. r0 + nr - 1 (row = g / inner, channel = row % C).  Slot jj of the window holds channel (r0 + jj) % C,
// for jj < W = min(max rows per tile, C); row j of the tile maps to slot j % W.
struct Window {
    uint32_t off0;     // offset of g0 inside its row (bigrow: unused)
    uint32_t split;    // bigrow: first local element of the second row (or > tile if none)
};

template <class Op>
__device__ __forceinline__ void stage_window(float* sm_par, Window* sm_win, int64_t g0, uint32_t tile_elems,
                                             const typename Op::Args& a) {
    const uint32_t tid = threadIdx.x;
    if (tid < a.W || tid == 0) {
        int64_t r0 = g0 / a.inner;
        int64_t off = g0 - r0 * a.inner;
        if (tid == 0) {
            Window w;
            w.off0 = a.bigrow ? 0u : (uint32_t)off;
            int64_t sp = a.inner - off;
            w.split = (uint32_t)(sp > (int64_t)tile_elems ? (int64_t)tile_elems + 1 : sp);
            *sm_win = w;
        }
        int64_t c0 = r0 % a.C;
        for (uint32_t jj = tid; jj < a.W; jj += kThreads) {
            int64_t c = c0 + jj;
            c = c % a.C;
            Op::stage(sm_par, a.W, jj, c, a);
        }
    }
}

// row (slot) of local element l
template <class Args>
__device__ __forceinline__ void locate(uint32_t l, const Window& w, const Args& a, uint32_t& slot, uint32_t& rem) {
    uint32_t j;
    if (a.bigrow) {
        j = l >= w.split ? 1u : 0u;
        rem = 0;   // unused in bigrow mode
    } else {
        uint32_t u = w.off0 + l;
        j = fdiv_u32(u, a.div_inner);
        rem = u - j * a.div_inner.d;
    }
    slot = j - fdiv_u32(j, a.div_W) * a.div_W.d;
}


// ------------------------------------------------------------------------------------------ dependent launch
// Every streaming kernel is launched with the programmatic-stream-serialization attribute and brackets its work with
// griddepcontrol.wait (returns once the preceding kernel in the stream has completed and its writes are visible; a no-op
// when the launch carries no programmatic dependency) and griddepcontrol.launch_dependents, which lets the NEXT kernel of
// the stream be scheduled while this one is still running: its CTAs take the SM slots that free up during our tail.
//
// Three orders exist, selected per launch by the host (`early` in the kernel arguments, see pdl_plan_launch):
//   0 late  : wait -> trigger -> loads -> math -> stores         the default; legal whatever else runs on the stream
//   1 early : loads -> wait -> trigger -> math -> stores         the dependent CTAs already have their tile in flight while
//             the predecessor's last wave drains.  Needs: the input is not an output of any launch still in flight.
//   2 free  : trigger -> loads -> math -> stores -> wait         the launch does not wait for anything until its CTAs are
//             done: consecutive launches overlap completely, there is no drain / ramp between them.  The wait at the end
//             keeps the stream's completion order (a kernel finishes only after its predecessor has).  Needs: inputs AND
//             outputs are disjoint from the inputs and outputs of every launch still in flight; at most two
//             such launches in a row, then a late one.
// Orders 1 and 2 are OPT-IN (mctq_set_tuning key 3 = 2 / 3; Python: `with mct_quantizers_b200.private_stream():`): the library
// cannot see kernels other libraries enqueue between two of its launches -- such a kernel may itself release its dependents
// before its stores are visible (cuDNN / CUTLASS kernels do), and the caching allocator may hand one of its input buffers
// to a later launch of ours as output -- so they are only legal while the stream carries this library's launches alone.
// Measured on the MobileNetV2 step (54 back-to-back launches): late 6656, early 6761 GB/s; an L2-prefetch-before-the-wait
// variant that would be legal unconditionally gained nothing (6647) and was dropped.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter(uint32_t order) {          // first statement of a streaming kernel
    if (order == 0) pdl_wait();
    if (order != 1) pdl_launch_dependents();
}
__device__ __forceinline__ void pdl_loaded(uint32_t order) {         // the tile's loads are issued; nothing has been written yet
    if (order == 1) { pdl_wait(); pdl_launch_dependents(); }
}
__device__ __forceinline__ void pdl_exit(uint32_t order) {           // last statement, every thread
    if (order == 2) pdl_wait();
}

// Host side (mctq_host.cu; consulted when the caller opted in): the library remembers, per (device, stream), the memory
// ranges of its launches that may still be in flight -- back to the last launch that waited before touching memory -- and
// picks the most permissive order the new launch's ranges allow.  Launches whose ranges are not described (multi-tensor
// plans) record "unknown", which forces the late order on their successor.
struct IoSpan { const void* p; size_t bytes; };
// `tables` (optional): the prepared blob the kernel stages into shared memory; *tab_early = 1 when it may do so before its wait
int pdl_plan_launch(cudaStream_t st, const IoSpan* in, int n_in, const IoSpan* out, int n_out,    // 0 late, 1 early, 2 free
                    const IoSpan* tables = nullptr, uint32_t* tab_early = nullptr);
// a prepare kernel (plain launch: waits for everything before it) that writes `blob`
void pdl_note_prepare(cudaStream_t st, const void* blob, size_t bytes);
void pdl_forget_streams();                                           // every stream starts over with a late launch

// ------------------------------------------------------------------------------------------ TMA bulk staging
// Parameter tables that are already laid out in global memory the way a CTA wants them in shared memory (prepared LUT
// records, prepared per-channel affine parameters) are staged with the bulk-copy engine instead of per-thread loops:
// one elected thread arms an mbarrier with the byte count and issues cp.async.bulk (1-D TMA, no tensor map) copies;
// the copies run while all threads of the CTA issue their streaming loads of the data tile, and everybody waits on
// the barrier's phase 0 just before the first use.  Addresses and sizes must be multiples of 16 bytes.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");     // make the init visible to the async proxy
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}

// ------------------------------------------------------------------------------------------ host helpers
// NVTX (header-only v3: no link dependency; a no-op unless a profiler injected itself) -- one range per C-ABI call, named
// after the entry point, so that an `ncu --nvtx` / Nsight Systems timeline shows which call of the reference's API a kernel
// belongs to.  Costs one predictable branch when off.
struct NvtxRange {
    bool on;
    explicit NvtxRange(const char* name);
    ~NvtxRange();
};
#define MCTQ_NVTX(name) mctq::NvtxRange mctq_nvtx_range_(name)
inline int cuda_rc(cudaError_t e) { return e == cudaSuccess ? 0 : (int)e; }

// launch with the programmatic-serialization attribute, in thread-block clusters of cluster_x CTAs along x when
// cluster_x > 1; the caller has already declared the launch to pdl_plan_launch
template <typename... KArgs, typename... Args>
inline int launch_planned_cluster(void (*kernel)(KArgs...), dim3 grid, unsigned cluster_x, size_t smem, cudaStream_t st,
                                  Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cluster_x > 1) {
        attr[1].id = cudaLaunchAttributeClusterDimension;
        attr[1].val.clusterDim.x = cluster_x;
        attr[1].val.clusterDim.y = 1;
        attr[1].val.clusterDim.z = 1;
        cfg.numAttrs = 2;
    }
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cuda_rc(e);
}

template <typename... KArgs, typename... Args>
inline int launch_planned(void (*kernel)(KArgs...), dim3 grid, size_t smem, cudaStream_t st, Args&&... args) {
    return launch_planned_cluster(kernel, grid, 1u, smem, st, std::forward<Args>(args)...);
}

// same, for kernels that always use the late order: their outputs are recorded as "unknown"
template <typename... KArgs, typename... Args>
inline int launch_streaming(void (*kernel)(KArgs...), dim3 grid, size_t smem, cudaStream_t st, Args&&... args) {
    pdl_plan_launch(st, nullptr, 0, nullptr, 0);
    return launch_planned(kernel, grid, smem, st, std::forward<Args>(args)...);
}

template <typename K>
int ensure_smem(K kernel, size_t bytes) {
    if (bytes <= 48 * 1024) return 0;
    if (bytes > 200 * 1024) return MCTQ_E_BADARG;
    return cuda_rc(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }

// ------------------------------------------------------------------------------------------ packed-weight descriptors
// The checks of every entry point that reads an MctqPackedDesc.  Their order fixes the error code of a descriptor with
// several faults: kind and dtype (pack_check_kind), then the entry point's shape and pointer checks, then the parameters.
// kind in range (MCTQ_E_BADARG); dtype a valid tag, f32 for the LUT kinds (MCTQ_E_DTYPE)
inline int pack_check_kind(int kind, int dtype) {
    if (kind < MCTQ_PACK_AFFINE_I8 || kind > MCTQ_PACK_LUT_I4) return MCTQ_E_BADARG;
    if (dtype != MCTQ_F32 && dtype != MCTQ_BF16 && dtype != MCTQ_F16) return MCTQ_E_DTYPE;
    if (pack_is_lut(kind) && dtype != MCTQ_F32) return MCTQ_E_DTYPE;          // LUT weights rebuild as f32, like the reference
    return 0;
}
// LUT kinds: quotients and 1 <= K <= pack_max_k (MCTQ_E_LUT); affine kinds: zero points (MCTQ_E_BADARG)
inline int pack_check_params(const MctqPackedDesc& d) {
    if (pack_is_lut(d.kind)) {
        if (!d.lut_quotients || d.K < 1 || d.K > pack_max_k(d.kind)) return MCTQ_E_LUT;
    } else if (!d.zp) {
        return MCTQ_E_BADARG;
    }
    return 0;
}
// the checks shared by mctq_packed_linear and mctq_packed_linear_batched: w is a row-major [out][in] weight with parameters
// per tensor or per output row, x and y have its dtype
inline int packed_linear_check(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x, int x_dtype,
                               int64_t M, const void* y) {
    if (!w) return MCTQ_E_BADARG;
    if (const int rc = pack_check_kind(w->kind, x_dtype)) return rc;
    if (w->y_dtype != x_dtype) return MCTQ_E_DTYPE;
    if (out_features < 1 || in_features < 1 || out_features >= (1LL << 31) || in_features >= (1LL << 31) || M < 0)
        return MCTQ_E_BADARG;
    if (w->n != out_features * in_features) return MCTQ_E_BADARG;
    if (w->C != 1 && !(w->C == out_features && w->inner == in_features)) return MCTQ_E_BADARG;
    if (!w->codes || !w->scale || !x || !y) return MCTQ_E_BADARG;
    return pack_check_params(*w);
}

// f(kind, type) with kind a std::integral_constant<int, MCTQ_PACK_*> and type a PackType<T>, for the (kind, dtype) of a
// checked descriptor: only the pairs the packed-weight kernels are built for, affine x {f32, bf16, f16} and LUT x f32
template <typename T> struct PackType { using type = T; };
template <class F>
int dispatch_packed(int kind, int dtype, F&& f) {
    auto typed = [&](auto k) {
        if constexpr (pack_is_lut(decltype(k)::value)) {
            return f(k, PackType<float>{});
        } else {
            if (dtype == MCTQ_F32) return f(k, PackType<float>{});
            if (dtype == MCTQ_BF16) return f(k, PackType<__nv_bfloat16>{});
            return f(k, PackType<__half>{});
        }
    };
    switch (kind) {
        case MCTQ_PACK_AFFINE_I8: return typed(std::integral_constant<int, MCTQ_PACK_AFFINE_I8>{});
        case MCTQ_PACK_AFFINE_I4: return typed(std::integral_constant<int, MCTQ_PACK_AFFINE_I4>{});
        case MCTQ_PACK_LUT_U8: return typed(std::integral_constant<int, MCTQ_PACK_LUT_U8>{});
        default: return typed(std::integral_constant<int, MCTQ_PACK_LUT_I4>{});
    }
}

// geometry of the channel window for a tile of `tile` elements
template <class Args>
void set_window(Args& a, uint32_t tile) {
    a.bigrow = a.inner >= (int64_t)tile ? 1u : 0u;
    int64_t rows = a.bigrow ? 2 : (int64_t)tile / a.inner + 2;
    a.W = (uint32_t)(rows < a.C ? rows : a.C);
    a.div_inner = make_fastdiv(a.bigrow ? 1u : (uint32_t)a.inner);
    a.div_W = make_fastdiv(a.W);
}

}  // namespace mctq
