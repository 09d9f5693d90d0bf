// mctq_affine.cu -- affine (round-clip-dequant) fake-quant kernels and their C ABI entry points.
#include <algorithm>

#include "mctq_common.cuh"

namespace mctq {

constexpr int32_t kFastRangeLimit = 1 << 21;

struct AffineArgs {
    const void* x;
    void* y;
    void* codes;
    int64_t n;
    const float* scale;     // device [C] or NULL (then scale_val / zp_val)
    const int32_t* zp;
    float scale_val;
    int32_t zp_val;
    int64_t C, inner, elem_offset;
    int32_t qmin, qmax;
    // channel-window geometry (host-derived)
    FastDiv div_inner, div_W;
    uint32_t W;             // staged channel slots
    uint32_t bigrow;        // inner >= tile elems: a tile touches at most two rows
    // CH_LAST (channel is the innermost dimension): parameters are staged for one period = lcm(C, V) of the channel
    // pattern, so that every aligned vector of V elements reads V consecutive entries
    uint32_t period;
    FastDiv div_period;
    // prepared parameters (mctq_affine_prepare): records {1/s, s, zp bits, (float)zp} per channel and the same values as
    // three arrays [inv | s | zp] of C4 = roundup(C, 4) entries each; NULL for the raw-parameter entry points
    const float4* prep_rec;
    const float* prep_soa;
    const int32_t* prep_flags;   // [0] != 0: some zero point is non-zero
    int64_t C4;
    uint32_t early;              // dependent-launch order: 0 late, 1 early, 2 free (opt-in, see pdl_plan_launch)
    uint32_t tab_early;          // PREP: the parameter blob may be staged before the dependent-launch wait (nobody is writing it)
};

constexpr size_t kPrepHeaderBytes = 16;
inline size_t prep_bytes(int64_t C) { int64_t C4 = (C + 3) & ~(int64_t)3; return kPrepHeaderBytes + (size_t)C * 16 + (size_t)C4 * 12; }

template <bool RINT> struct AffineOp {
    using Args = AffineArgs;
    struct ChanParams { float inv, s, lo, hi; int zp; };
    static constexpr int kSmemFloatsPerChan = 3;

    __device__ static __forceinline__ ChanParams make(float s, int zp, const Args& a) {
        ChanParams p;
        p.s = s;
        p.inv = __fdiv_rn(1.0f, s);                  // IEEE reciprocal of the f32 scale (ATen: 1.0f / scale)
        p.zp = zp;
        if (RINT) { p.lo = (float)a.qmin; p.hi = (float)a.qmax; }
        else { p.lo = small_int_to_float(a.qmin - zp); p.hi = small_int_to_float(a.qmax - zp); }    // |q - zp| <= 2^21 on this path
        return p;
    }
    __device__ static __forceinline__ ChanParams uniform(const Args& a) {
        float s = a.scale ? __ldg(a.scale) : a.scale_val;
        int zp = a.zp ? __ldg(a.zp) : a.zp_val;
        return make(s, zp, a);
    }
    __device__ static __forceinline__ void stage(float* sm, uint32_t W, uint32_t slot, int64_t c, const Args& a) {
        ChanParams p = make(__ldg(a.scale + c), __ldg(a.zp + c), a);
        sm[slot] = p.inv;
        sm[W + slot] = p.s;
        sm[2 * W + slot] = __int_as_float(p.zp);
    }
    __device__ static __forceinline__ ChanParams fetch(const float* sm, uint32_t W, uint32_t slot, const Args& a) {
        ChanParams p;
        p.inv = sm[slot];
        p.s = sm[W + slot];
        p.zp = __float_as_int(sm[2 * W + slot]);
        if (RINT) { p.lo = (float)a.qmin; p.hi = (float)a.qmax; }
        else { p.lo = small_int_to_float(a.qmin - p.zp); p.hi = small_int_to_float(a.qmax - p.zp); }
        return p;
    }
    // prepared record {1/s, s, zp bits, (float)zp}: one 16-byte shared-memory load, no int -> float conversions
    // ((float)(qmin - zp) == (float)qmin - (float)zp exactly: all three are integers below 2^24)
    __device__ static __forceinline__ ChanParams fetch_rec(const float* sm, uint32_t slot, const Args& a) {
        const float4 r = reinterpret_cast<const float4*>(sm)[slot];
        ChanParams p;
        p.inv = r.x;
        p.s = r.y;
        p.zp = __float_as_int(r.z);
        if (RINT) { p.lo = (float)a.qmin; p.hi = (float)a.qmax; }
        else { p.lo = __fsub_rn((float)a.qmin, r.w); p.hi = __fsub_rn((float)a.qmax, r.w); }
        return p;
    }
    // returns y; code receives the clamped integer q
    template <bool WANT_CODE>
    __device__ static __forceinline__ float apply(float x, const ChanParams& p, int& code) {
        float t = __fmul_rn(x, p.inv);
        if (!RINT) {
            // (t + M) - M rounds half-to-even exactly for |t| < 2^22 and stays out of [lo, hi] beyond it;
            // anything that rounds to zero comes out as +0.0, so y never carries the sign of a tiny negative
            // input (ATen subtracts the integer zero point, which has the same effect).  Clamping
            // r to [qmin - zp, qmax - zp] equals clamp(r + zp, qmin, qmax) - zp on integer-valued floats.
            float r = __fsub_rn(__fadd_rn(t, kMagic), kMagic);
            float c = fminf(fmaxf(r, p.lo), p.hi);           // fmaxf(NaN, lo) = lo: NaN -> qmin
            // integer code without F2I (a quarter-rate conversion that made the codes-only bf16 variant issue bound): c is an
            // integer with |c| < 2^22, so the low mantissa bits of c + 1.5 * 2^23 ARE c in two's complement
            if (WANT_CODE) code = __float_as_int(__fadd_rn(c, kMagic)) + (p.zp - 0x4B400000);
            return __fmul_rn(c, p.s);
        } else {
            float zf = (float)p.zp;
            float q = __fadd_rn(rintf(t), zf);
            q = fminf(fmaxf(q, p.lo), p.hi);
            if (WANT_CODE) code = (int)q;
            return __fmul_rn(__fsub_rn(q, zf), p.s);
        }
    }
};

// ------------------------------------------------------------------------------------------ affine kernel
// PREP: the per-channel parameters come from a prepared blob and are staged with 1-D TMA bulk copies (one elected thread,
// one mbarrier) instead of per-thread load / divide / store loops -- the staging cost of a tile that touches hundreds
// of channels (short rows, channel-innermost layouts) drops to a handful of instructions.
// VB: bytes per vector (16, or 8 for 2-byte types in CH_LAST mode: with 16-byte vectors of bf16 a lane needs 8 consecutive
// parameter entries = two LDS.128 at a lane stride of 32 bytes, which is a 2-way bank conflict and made the kernel
// shared-memory bound; 8-byte vectors need one LDS.128 per array at a lane stride of 16 bytes, conflict free).
template <typename T, int CHMODE, int CODE, int UNROLL, bool RINT, bool PREP, int VB = 16>
__global__ void __launch_bounds__(kThreads) fq_affine_kernel(const AffineArgs a) {
    using Op = AffineOp<RINT>;
    constexpr int V = VB / sizeof(T);
    constexpr int WORDS = VB / 4;
    constexpr uint32_t TILE = kThreads * UNROLL * V;
    extern __shared__ __align__(16) float sm_par[];
    __shared__ Window sm_win;
    __shared__ __align__(8) uint64_t sm_bar;

    const uint32_t tid = threadIdx.x;
    const int64_t t0 = (int64_t)blockIdx.x * TILE;
    const int64_t remaining = a.n - t0;
    const bool full = remaining >= (int64_t)TILE;
    const T* xt = reinterpret_cast<const T*>(a.x) + t0;
    bool has_zp = true;
    // PREP: one elected thread arms the mbarrier and hands the tile's channel window to the bulk-copy engine.  When the
    // host knows that the blob is not being written (tab_early) this happens BEFORE the dependent-launch wait, so a CTA
    // scheduled into the predecessor's tail has its parameters in shared memory when the wait returns.
    if constexpr (PREP && CHMODE != CH_PT) {
        auto stage = [&]() {
            if (tid != 0) return;
            mbar_init(&sm_bar, 1);
            if (CHMODE == CH_LAST) {
                // period / C back-to-back copies of each parameter array: entry i = channel i % C
                const uint32_t Cb = (uint32_t)a.C * 4u, reps = a.period / (uint32_t)a.C;
                mbar_arrive_expect_tx(&sm_bar, 3u * a.period * 4u);
                for (uint32_t arr = 0; arr < 3; ++arr)
                    for (uint32_t r = 0; r < reps; ++r)
                        bulk_g2s(sm_par + arr * a.period + r * (uint32_t)a.C, a.prep_soa + arr * a.C4, Cb, &sm_bar);
            } else {
                const int64_t g0 = a.elem_offset + t0;
                const int64_t r0 = g0 / a.inner;
                const int64_t off = g0 - r0 * a.inner;
                Window wv;
                wv.off0 = a.bigrow ? 0u : (uint32_t)off;
                const int64_t sp = a.inner - off;
                wv.split = (uint32_t)(sp > (int64_t)TILE ? (int64_t)TILE + 1 : sp);
                sm_win = wv;
                const uint32_t c0 = (uint32_t)(r0 % a.C);
                const uint32_t n1 = min(a.W, (uint32_t)a.C - c0);          // records before the channel index wraps
                mbar_arrive_expect_tx(&sm_bar, a.W * 16u);
                bulk_g2s(sm_par, a.prep_rec + c0, n1 * 16u, &sm_bar);
                if (n1 < a.W) bulk_g2s(sm_par + 4u * n1, a.prep_rec, (a.W - n1) * 16u, &sm_bar);
            }
        };
        // staging always precedes the tile loads; what moves is the wait (the host only picks an order other than "late"
        // together with tab_early)
        if (!a.tab_early) pdl_enter(0);
        stage();
        if (a.tab_early) pdl_enter(a.early);
    } else {
        pdl_enter(a.early);
    }

    uint32_t w[UNROLL][WORDS];
    if (full) {
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) ld_words<WORDS>(xt + (size_t)(j * kThreads + tid) * V, w[j]);
    } else {
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) {
            int64_t l = (int64_t)(j * kThreads + tid) * V;
            if (l + V <= remaining) ld_words<WORDS>(xt + l, w[j]);
            else {
                T tmp[V];
#pragma unroll
                for (int e = 0; e < V; ++e) tmp[e] = (l + e < remaining) ? xt[l + e] : from_f32<T>(0.0f);
                memcpy(w[j], tmp, VB);
            }
        }
    }
    pdl_loaded(a.early);                                   // the tile is in flight; nothing is written before this point

    typename Op::ChanParams pu;
    Window win;
    uint32_t base_mod = 0;
    if (CHMODE == CH_PT) {
        pu = Op::uniform(a);
    } else if (PREP) {
        // (read after the tile loads are issued: every thread needs it, and a wait in front of the loads would serialise
        // an L2 round trip with them)
        if (CHMODE == CH_LAST || CHMODE == CH_ELEM) has_zp = __ldg(a.prep_flags) != 0;
        if (CHMODE == CH_LAST) base_mod = (uint32_t)((uint64_t)(a.elem_offset + t0) % a.period);
        __syncthreads();                                               // barrier init + window visible to everyone
        if (CHMODE != CH_LAST) win = sm_win;
        mbar_wait(&sm_bar, 0);
    } else if (CHMODE == CH_LAST) {
        // entry i of the period holds the parameters of channel i % C (struct of arrays: inv | s | zp)
        int any_zp = 0;
        for (uint32_t i = tid; i < a.period; i += kThreads) {
            const uint32_t c = i - fdiv_u32(i, a.div_W) * a.div_W.d;              // div_W divides by C here
            Op::stage(sm_par, a.period, i, (int64_t)c, a);
            any_zp |= __ldg(a.zp + c);
        }
        base_mod = (uint32_t)((uint64_t)(a.elem_offset + t0) % a.period);
        // symmetric quantizers have all-zero zero points: then a third of the shared-memory reads can be skipped
        has_zp = __syncthreads_or(any_zp) != 0;
    } else {
        stage_window<Op>(sm_par, &sm_win, a.elem_offset + t0, TILE, a);
        __syncthreads();
        win = sm_win;
    }

    T* yt = reinterpret_cast<T*>(a.y) + t0;
#pragma unroll
    for (int j = 0; j < UNROLL; ++j) {
        const uint32_t l = (uint32_t)(j * kThreads + tid) * V;
        float f[V];
        int code[V];
        Pack<T, V>::unpack(w[j], f);
        if (CHMODE == CH_PT) {
#pragma unroll
            for (int e = 0; e < V; ++e) f[e] = Op::template apply<CODE != 0>(f[e], pu, code[e]);
        } else if (CHMODE == CH_LAST) {
            const uint32_t m = base_mod + l;
            const uint32_t i0 = m - fdiv_u32(m, a.div_period) * a.period;            // multiple of V: vector loads below
            float pinv[V], ps[V], pz[V];
#pragma unroll
            for (int e = 0; e < V; e += 4) {
                *reinterpret_cast<float4*>(&pinv[e]) = *reinterpret_cast<const float4*>(&sm_par[i0 + e]);
                *reinterpret_cast<float4*>(&ps[e]) = *reinterpret_cast<const float4*>(&sm_par[a.period + i0 + e]);
                if (has_zp) *reinterpret_cast<float4*>(&pz[e]) = *reinterpret_cast<const float4*>(&sm_par[2 * a.period + i0 + e]);
                else *reinterpret_cast<float4*>(&pz[e]) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (!has_zp) {
                typename Op::ChanParams p;
                p.zp = 0;
                p.lo = (float)a.qmin;
                p.hi = (float)a.qmax;
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    p.inv = pinv[e];
                    p.s = ps[e];
                    f[e] = Op::template apply<CODE != 0>(f[e], p, code[e]);
                }
            } else {
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    typename Op::ChanParams p;
                    p.inv = pinv[e];
                    p.s = ps[e];
                    p.zp = __float_as_int(pz[e]);
                    if (RINT) { p.lo = (float)a.qmin; p.hi = (float)a.qmax; }
                    else { p.lo = small_int_to_float(a.qmin - p.zp); p.hi = small_int_to_float(a.qmax - p.zp); }
                    f[e] = Op::template apply<CODE != 0>(f[e], p, code[e]);
                }
            }
        } else if (CHMODE == CH_VEC) {
            uint32_t slot, rem;
            locate(l, win, a, slot, rem);
            typename Op::ChanParams p = PREP ? Op::fetch_rec(sm_par, slot, a) : Op::fetch(sm_par, a.W, slot, a);
#pragma unroll
            for (int e = 0; e < V; ++e) f[e] = Op::template apply<CODE != 0>(f[e], p, code[e]);
        } else if (a.inner >= V) {
            // CH_ELEM, rows at least one vector long: the vector straddles at most one row boundary, so two
            // parameter sets and a per-element select replace V shared-memory fetches
            uint32_t slot, rem, k;                  // k = elements of this vector that still belong to the first row
            if (a.bigrow) {
                const bool second = l >= win.split;
                slot = second ? 1u : 0u;
                rem = 0;
                k = second ? (uint32_t)V : min((uint32_t)V, win.split - l);
            } else {
                locate(l, win, a, slot, rem);
                k = a.div_inner.d - rem;
            }
            const uint32_t slot1 = (slot + 1 == a.W) ? 0u : slot + 1;
            const typename Op::ChanParams p0 = PREP ? Op::fetch_rec(sm_par, slot, a) : Op::fetch(sm_par, a.W, slot, a);
            const typename Op::ChanParams p1 = PREP ? Op::fetch_rec(sm_par, slot1, a) : Op::fetch(sm_par, a.W, slot1, a);
            if (PREP && !has_zp) {
                // all zero points are zero (symmetric quantizers): the clamp bounds are the same for every channel, only
                // 1/s and s are selected per element
                typename Op::ChanParams p = p0;
                p.zp = 0;
                p.lo = (float)a.qmin;
                p.hi = (float)a.qmax;
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    const bool first = (uint32_t)e < k;
                    p.inv = first ? p0.inv : p1.inv;
                    p.s = first ? p0.s : p1.s;
                    f[e] = Op::template apply<CODE != 0>(f[e], p, code[e]);
                }
            } else {
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    const bool first = (uint32_t)e < k;
                    typename Op::ChanParams p;
                    p.inv = first ? p0.inv : p1.inv;
                    p.s = first ? p0.s : p1.s;
                    p.lo = first ? p0.lo : p1.lo;
                    p.hi = first ? p0.hi : p1.hi;
                    p.zp = first ? p0.zp : p1.zp;
                    f[e] = Op::template apply<CODE != 0>(f[e], p, code[e]);
                }
            }
        } else {
            // rows shorter than a vector (inner < V, not channel-last): per-element parameter fetch
            uint32_t slot, rem;
            locate(l, win, a, slot, rem);
#pragma unroll
            for (int e = 0; e < V; ++e) {
                typename Op::ChanParams p = PREP ? Op::fetch_rec(sm_par, slot, a) : Op::fetch(sm_par, a.W, slot, a);
                f[e] = Op::template apply<CODE != 0>(f[e], p, code[e]);
                if (++rem == a.div_inner.d) { rem = 0; slot = (slot + 1 == a.W) ? 0 : slot + 1; }
            }
        }
        if (full || (int64_t)l + V <= remaining) {
            if (a.y) { Pack<T, V>::pack(f, w[j]); st_words<WORDS>(yt + l, w[j]); }
            if (CODE != 0) st_codes<V, CODE>(a.codes, t0 + l, code);
        } else if ((int64_t)l < remaining) {
            const int cnt = (int)(remaining - l);
            for (int e = 0; e < V; ++e) {
                if (e < cnt) {
                    if (a.y) yt[l + e] = from_f32<T>(f[e]);
                    if (CODE == MCTQ_CODES_INT8) reinterpret_cast<uint8_t*>(a.codes)[t0 + l + e] = (uint8_t)(code[e] & 0xff);
                }
            }
            if (CODE == MCTQ_CODES_INT4) {
                uint8_t* cp = reinterpret_cast<uint8_t*>(a.codes) + ((t0 + l) >> 1);
                for (int e = 0; e < V; e += 2) {
                    if (e < cnt) {
                        int hi = (e + 1 < cnt) ? code[e + 1] : 0;
                        cp[e >> 1] = (uint8_t)((code[e] & 0xf) | ((hi & 0xf) << 4));
                    }
                }
            }
        }
    }
    pdl_exit(a.early);
}

// ------------------------------------------------------------------------------------------ parameter preparation
// blob = [16-byte header: int32 any_nonzero_zp][records float4 x C][inv C4 | s C4 | zp C4]
__global__ void __launch_bounds__(kThreads) affine_prepare_kernel(const float* __restrict__ scale, const int32_t* __restrict__ zp,
                                                                  int64_t C, int64_t C4, uint8_t* blob) {
    int32_t* flags = reinterpret_cast<int32_t*>(blob);
    float4* rec = reinterpret_cast<float4*>(blob + kPrepHeaderBytes);
    float* soa = reinterpret_cast<float*>(blob + kPrepHeaderBytes + (size_t)C * 16);
    for (int64_t c = (int64_t)blockIdx.x * kThreads + threadIdx.x; c < C4; c += (int64_t)gridDim.x * kThreads) {
        float s = 1.0f;
        int z = 0;
        if (c < C) { s = scale[c]; z = zp[c]; }
        const float inv = __fdiv_rn(1.0f, s);
        if (c < C) rec[c] = make_float4(inv, s, __int_as_float(z), (float)z);
        soa[c] = inv;
        soa[C4 + c] = s;
        soa[2 * C4 + c] = __int_as_float(z);
        if (z != 0) atomicOr(flags, 1);
    }
}

// ------------------------------------------------------------------------------------------ scalar fallbacks
// Misaligned base pointers (views with odd offsets): element-per-thread, still coalesced.
template <typename T, bool RINT>
__global__ void __launch_bounds__(kThreads) fq_affine_scalar_kernel(const AffineArgs a) {
    using Op = AffineOp<RINT>;
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < a.n; i += stride) {
        int64_t c = 0;
        if (a.C > 1) c = ((a.elem_offset + i) / a.inner) % a.C;
        typename Op::ChanParams p = a.scale ? Op::make(__ldg(a.scale + c), __ldg(a.zp + c), a) : Op::make(a.scale_val, a.zp_val, a);
        int code;
        float y = Op::template apply<true>(to_f32<T>(reinterpret_cast<const T*>(a.x)[i]), p, code);
        if (a.y) reinterpret_cast<T*>(a.y)[i] = from_f32<T>(y);
        if (a.codes) reinterpret_cast<int8_t*>(a.codes)[i] = (int8_t)code;   // scalar fallback emits INT8 only
    }
}

// ------------------------------------------------------------------------------------------ dequant of codes
template <int CODE>
__global__ void __launch_bounds__(kThreads) dequant_affine_kernel(const void* codes, int is_signed, float* y, int64_t n,
                                                                  const float* scale, const int32_t* zp, int64_t C,
                                                                  int64_t inner, int64_t elem_offset) {
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
        int q;
        if (CODE == MCTQ_CODES_INT8) {
            uint8_t b = reinterpret_cast<const uint8_t*>(codes)[i];
            q = is_signed ? (int)(int8_t)b : (int)b;
        } else {
            uint8_t b = reinterpret_cast<const uint8_t*>(codes)[i >> 1];
            int nib = (i & 1) ? (b >> 4) : (b & 0xf);
            q = is_signed ? ((nib ^ 8) - 8) : nib;
        }
        int64_t c = C > 1 ? ((elem_offset + i) / inner) % C : 0;
        y[i] = __fmul_rn((float)(q - __ldg(zp + c)), __ldg(scale + c));
    }
}

// Streaming consumer of the code wire format: tile = 256 threads x 4 vectors x V codes, one f32 store per vector; 5 (int8) /
// 4.5 (int4) algorithmic bytes per element.  Code loading, channel walk (MODE 0 / 1 / 2) and stores: codes_tile in
// mctq_common.cuh.  V = 8 (ONE 32-byte store: STG.256) when the whole vector lies in one channel -- half the loads, stores
// and channel look-ups per element.
template <int CODE, int MODE, int V>
__global__ void __launch_bounds__(kThreads) dequant_affine_vec_kernel(const void* codes, int is_signed, float* y, int64_t n,
                                                                      const float* __restrict__ scale, const int32_t* __restrict__ zp,
                                                                      uint32_t C, uint32_t inner, int64_t elem_offset,
                                                                      const FastDiv div_inner, const FastDiv div_C) {
    constexpr int UNROLL = 4;
    constexpr int64_t TILE = (int64_t)kThreads * UNROLL * V;
    pdl_wait();
    pdl_launch_dependents();
    codes_tile<CODE, MODE, V, UNROLL>(reinterpret_cast<const uint8_t*>(codes), y, (int64_t)blockIdx.x * TILE, n, is_signed, C, inner,
                                      elem_offset, div_inner, div_C, AffineCodeOp{scale, zp});
}

// ------------------------------------------------------------------------------------------ multi-tensor
constexpr int kMultiTile = 2048;   // elements per tile, any dtype (8192 measured: ResNet-18 29 -> 29 us, MobileNetV2 10 -> 17 us)

// channel of logical element i: 32-bit arithmetic whenever the tensor has fewer than 2^32 elements
__device__ __forceinline__ int64_t multi_channel(int64_t i, const MctqTensorDesc& d, bool small) {
    if (d.C <= 1) return 0;
    if (small) return (int64_t)(((uint32_t)i / (uint32_t)d.inner) % (uint32_t)d.C);
    return (i / d.inner) % d.C;
}

template <typename T, bool RINT>
__device__ __forceinline__ void multi_tile_body(const MctqTensorDesc& d, int64_t e0) {
    using Op = AffineOp<RINT>;
    constexpr int V = 4;                                   // elements per vector: 16 B (f32) or 8 B (bf16 / f16)
    constexpr int WORDS = V * sizeof(T) / 4;
    constexpr int NV = kMultiTile / (kThreads * V);        // vectors per thread (2)
    const T* x = reinterpret_cast<const T*>(d.x);
    T* y = reinterpret_cast<T*>(d.y);
    const int64_t rem = d.n - e0;
    const bool small = d.n < (1LL << 32) && d.inner < (1LL << 32) && d.C < (1LL << 32);
    AffineArgs a;
    a.qmin = d.qmin;
    a.qmax = d.qmax;
    const bool vec = (d.C <= 1 || d.inner % V == 0) && (reinterpret_cast<uintptr_t>(x) % (V * sizeof(T))) == 0 &&
                     (!y || (reinterpret_cast<uintptr_t>(y) % (V * sizeof(T))) == 0) &&
                     (!d.codes || d.code_mode != MCTQ_CODES_INT8 || (reinterpret_cast<uintptr_t>(d.codes) & 3u) == 0);
    if (vec) {
        // one channel per aligned vector of 4: load both vectors and their parameters first, then one reciprocal per vector
        uint32_t w[NV][WORDS];
        float sc[NV];
        int zp[NV];
        bool whole[NV];
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int64_t l = (int64_t)(j * kThreads + threadIdx.x) * V;
            whole[j] = l + V <= rem;
            if (whole[j]) ld_words<WORDS>(x + e0 + l, w[j]);
            else {
                T tmp[V];
#pragma unroll
                for (int e = 0; e < V; ++e) tmp[e] = (l + e < rem) ? x[e0 + l + e] : from_f32<T>(0.0f);
                memcpy(w[j], tmp, sizeof(tmp));
            }
            const int64_t c = l < rem ? multi_channel(e0 + l, d, small) : 0;
            sc[j] = __ldg(d.scale + c);
            zp[j] = __ldg(d.zp + c);
        }
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int64_t l = (int64_t)(j * kThreads + threadIdx.x) * V;
            if (l >= rem) continue;
            const typename Op::ChanParams p = Op::make(sc[j], zp[j], a);
            float f[V];
            int code[V];
            Pack<T, V>::unpack(w[j], f);
#pragma unroll
            for (int e = 0; e < V; ++e) f[e] = Op::template apply<true>(f[e], p, code[e]);
            if (whole[j]) {
                if (y) { Pack<T, V>::pack(f, w[j]); st_words<WORDS>(y + e0 + l, w[j]); }
                if (d.codes && d.code_mode == MCTQ_CODES_INT8) st_codes<V, MCTQ_CODES_INT8>(d.codes, e0 + l, code);
            } else {
                for (int e = 0; e < V && l + e < rem; ++e) {
                    if (y) y[e0 + l + e] = from_f32<T>(f[e]);
                    if (d.codes && d.code_mode == MCTQ_CODES_INT8) reinterpret_cast<uint8_t*>(d.codes)[e0 + l + e] = (uint8_t)(code[e] & 0xff);
                }
            }
        }
        return;
    }
    // rows that are not a multiple of 4 (depthwise 3x3, first conv ...) or misaligned views: 8 elements per thread,
    // strided by the CTA width so that every access is coalesced; one channel look-up per element
    const int64_t e1 = min(e0 + (int64_t)kMultiTile, d.n);
    float xv[kMultiTile / kThreads];
#pragma unroll
    for (int k = 0; k < kMultiTile / kThreads; ++k) {
        int64_t i = e0 + k * kThreads + threadIdx.x;
        xv[k] = i < e1 ? to_f32<T>(x[i]) : 0.0f;
    }
#pragma unroll
    for (int k = 0; k < kMultiTile / kThreads; ++k) {
        int64_t i = e0 + k * kThreads + threadIdx.x;
        if (i < e1) {
            const int64_t c = multi_channel(i, d, small);
            int code;
            const float out = Op::template apply<true>(xv[k], Op::make(__ldg(d.scale + c), __ldg(d.zp + c), a), code);
            if (y) y[i] = from_f32<T>(out);
            if (d.codes && d.code_mode == MCTQ_CODES_INT8) reinterpret_cast<uint8_t*>(d.codes)[i] = (uint8_t)(code & 0xff);
        }
    }
}

__global__ void __launch_bounds__(kThreads) fq_affine_multi_kernel(const MctqTensorDesc* __restrict__ descs,
                                                                   const int32_t* __restrict__ tile_starts, int n_desc) {
    pdl_wait();
    pdl_launch_dependents();
    // which tensor does this tile belong to?  upper-bound binary search over tile_starts
    const int tile = blockIdx.x;
    int lo = 0, hi = n_desc;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (__ldg(tile_starts + mid) <= tile) lo = mid; else hi = mid;
    }
    const MctqTensorDesc d = descs[lo];
    const int64_t e0 = (int64_t)(tile - __ldg(tile_starts + lo)) * kMultiTile;
    const bool fast = (int64_t)d.qmax - d.qmin < kFastRangeLimit;
    if (d.dtype == MCTQ_F32) { if (fast) multi_tile_body<float, false>(d, e0); else multi_tile_body<float, true>(d, e0); }
    else if (d.dtype == MCTQ_BF16) { if (fast) multi_tile_body<__nv_bfloat16, false>(d, e0); else multi_tile_body<__nv_bfloat16, true>(d, e0); }
    else { if (fast) multi_tile_body<__half, false>(d, e0); else multi_tile_body<__half, true>(d, e0); }
}

// ---- many per-tensor sites, one launch (activation holders whose inputs already exist; SURVEY 8f rank 1 applied to the
// activation side).  54 back-to-back launches of a MobileNetV2 step lose ~1.5 us each to the drain of one grid and the
// ramp of the next even with programmatic dependent launch (4 % of the step); one grid over all sites has neither.
// The site table travels as kernel parameters (constant bank: a binary search of a few LDC, no global look-up in front
// of the tile's loads); every CTA runs the per-tensor body of fq_affine_kernel<T, CH_PT> on one 8 KB tile of its site.
constexpr int kSitesCap = 64;
struct alignas(16) SiteEntry {
    const void* x;
    void* y;
    int64_t n;
    float scale;
    int32_t zp, qmin, qmax;
    int32_t dtype, pad;
};
struct SitesParams {
    int32_t n_sites, pad[3];
    int32_t starts[kSitesCap + 4];              // starts[k] = first tile of site k; starts[n_sites] = number of tiles
    SiteEntry e[kSitesCap];
};
static_assert(sizeof(SitesParams) <= 4096, "kernel parameter space");

template <typename T, bool RINT>
__device__ __forceinline__ void site_tile(const SiteEntry& s, const int64_t tile) {
    using Op = AffineOp<RINT>;
    constexpr int UNROLL = 2, V = 16 / sizeof(T), WORDS = 4;
    constexpr uint32_t TILE = kThreads * UNROLL * V;
    const uint32_t tid = threadIdx.x;
    const int64_t t0 = tile * TILE;
    const int64_t remaining = s.n - t0;
    const bool full = remaining >= (int64_t)TILE;
    const T* xt = reinterpret_cast<const T*>(s.x) + t0;
    T* yt = reinterpret_cast<T*>(s.y) + t0;
    uint32_t w[UNROLL][WORDS];
    if (full) {
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) ld_words<WORDS>(xt + (size_t)(j * kThreads + tid) * V, w[j]);
    } else {
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) {
            int64_t l = (int64_t)(j * kThreads + tid) * V;
            if (l + V <= remaining) ld_words<WORDS>(xt + l, w[j]);
            else {
                T tmp[V];
#pragma unroll
                for (int e = 0; e < V; ++e) tmp[e] = (l + e < remaining) ? xt[l + e] : from_f32<T>(0.0f);
                memcpy(w[j], tmp, 16);
            }
        }
    }
    AffineArgs a;                                   // only the fields AffineOp::make reads
    a.qmin = s.qmin;
    a.qmax = s.qmax;
    const typename Op::ChanParams p = Op::make(s.scale, s.zp, a);
#pragma unroll
    for (int j = 0; j < UNROLL; ++j) {
        const uint32_t l = (uint32_t)(j * kThreads + tid) * V;
        float f[V];
        int code;
        Pack<T, V>::unpack(w[j], f);
#pragma unroll
        for (int e = 0; e < V; ++e) f[e] = Op::template apply<false>(f[e], p, code);
        if (full || (int64_t)l + V <= remaining) {
            Pack<T, V>::pack(f, w[j]);
            st_words<WORDS>(yt + l, w[j]);
        } else if ((int64_t)l < remaining) {
            const int cnt = (int)(remaining - l);
            for (int e = 0; e < V; ++e)
                if (e < cnt) yt[l + e] = from_f32<T>(f[e]);
        }
    }
}

__global__ void __launch_bounds__(kThreads) fq_affine_sites_kernel(const __grid_constant__ SitesParams p) {
    pdl_wait();
    pdl_launch_dependents();
    const int tile = blockIdx.x;
    int lo = 0, hi = p.n_sites;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (p.starts[mid] <= tile) lo = mid; else hi = mid;
    }
    const SiteEntry& s = p.e[lo];
    const int64_t t = (int64_t)(tile - p.starts[lo]);
    const bool fast = (int64_t)s.qmax - s.qmin < kFastRangeLimit;
    if (s.dtype == MCTQ_F32) { if (fast) site_tile<float, false>(s, t); else site_tile<float, true>(s, t); }
    else if (s.dtype == MCTQ_BF16) { if (fast) site_tile<__nv_bfloat16, false>(s, t); else site_tile<__nv_bfloat16, true>(s, t); }
    else { if (fast) site_tile<__half, false>(s, t); else site_tile<__half, true>(s, t); }
}

// ---- 8-bit codes of a [M][K] row-major x and their row sums (integer linear mode, mctq_packed_igemm.cu): one warp per row,
// the per-tensor recipe of fq_affine_kernel (AffineOp<false>::apply), so the codes are those mctq_fq_affine_scalar emits.
// VEC: K % 8 == 0 and x 16-byte aligned: 8 elements per lane and step (one or two 16-byte loads, one 8-byte store).
template <typename T, bool VEC>
__global__ void __launch_bounds__(kThreads) quantize_rows_kernel(const T* __restrict__ x, uint8_t* __restrict__ codes,
                                                                  int32_t* __restrict__ rowsum, int64_t M, int64_t K,
                                                                  float scale, int32_t zp, int32_t qmin, int32_t qmax) {
    using Op = AffineOp<false>;
    AffineArgs a;                                   // only the fields AffineOp::make reads
    a.qmin = qmin;
    a.qmax = qmax;
    const Op::ChanParams p = Op::make(scale, zp, a);
    pdl_wait();
    pdl_launch_dependents();
    const int warps = kThreads / 32, lane = threadIdx.x & 31;
    for (int64_t row = (int64_t)blockIdx.x * warps + (threadIdx.x >> 5); row < M; row += (int64_t)gridDim.x * warps) {
        const T* xr = x + row * K;
        uint8_t* cr = codes + row * K;
        int32_t sum = 0;
        if (VEC) {
            constexpr int W = 8 * sizeof(T) / 4;    // 32-bit words of 8 elements
            for (int64_t k = 8 * lane; k < K; k += 256) {
                uint32_t w[W];
                ld_words<4>(xr + k, w);
                if (W == 8) ld_words<4>(xr + k + 4, w + 4);
                float f[8];
                Pack<T, 8>::unpack(w, f);
                int c[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    Op::template apply<true>(f[e], p, c[e]);
                    sum += c[e];
                }
                st_codes<8, MCTQ_CODES_INT8>(cr, k, c);
            }
        } else {
            for (int64_t k = lane; k < K; k += 32) {
                int c;
                Op::template apply<true>(to_f32<T>(xr[k]), p, c);
                sum += c;
                cr[k] = (uint8_t)(c & 0xff);
            }
        }
        if (rowsum) {
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
            if (lane == 0) rowsum[row] = sum;
        }
    }
}

// ---- NHWC codes of an NCHW x [N][C][HW] and their per-pixel channel sums (integer convolution mode): the recipe of
// quantize_rows_kernel as a tiled transpose through shared memory.  A CTA takes 32 pixels of one image and walks the
// channels 64 at a time: warp w reads channels w, w + 8, .. of the 32 pixels (coalesced along W), then the CTA writes the
// 64 channel codes of 4 pixels per pass (coalesced along C).
template <typename T>
__global__ void __launch_bounds__(kThreads) quantize_nhwc_kernel(const T* __restrict__ x, uint8_t* __restrict__ codes,
                                                                  int32_t* __restrict__ psum, int64_t N, int64_t C, int64_t HW,
                                                                  float scale, int32_t zp, int32_t qmin, int32_t qmax) {
    using Op = AffineOp<false>;
    AffineArgs a;                                   // only the fields AffineOp::make reads
    a.qmin = qmin;
    a.qmax = qmax;
    const Op::ChanParams p = Op::make(scale, zp, a);
    __shared__ uint8_t tile[64][33];                // [channel][pixel]; the odd row length spreads the column reads
    __shared__ int32_t sums[kThreads / 32][32];
    pdl_wait();
    pdl_launch_dependents();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t ptiles = (HW + 31) / 32;
    for (int64_t t = blockIdx.x; t < N * ptiles; t += gridDim.x) {
        const int64_t b = t / ptiles, p0 = (t - b * ptiles) * 32;
        const T* xb = x + b * C * HW;
        uint8_t* cb = codes + b * HW * C;
        int32_t sum = 0;
        for (int64_t c0 = 0; c0 < C; c0 += 64) {
#pragma unroll
            for (int i = 0; i < 64 / (kThreads / 32); ++i) {
                const int cl = ty + (kThreads / 32) * i;
                const int64_t c = c0 + cl, px = p0 + tx;
                int q = 0;
                if (c < C && px < HW) {
                    Op::template apply<true>(to_f32<T>(xb[c * HW + px]), p, q);
                    sum += q;
                }
                tile[cl][tx] = (uint8_t)(q & 0xff);
            }
            __syncthreads();
#pragma unroll
            for (int i = 0; i < 32 / (kThreads / 64); ++i) {
                const int pl = (kThreads / 64) * i + (threadIdx.x >> 6), cl = threadIdx.x & 63;
                const int64_t px = p0 + pl, c = c0 + cl;
                if (px < HW && c < C) cb[px * C + c] = tile[cl][pl];
            }
            __syncthreads();
        }
        if (psum) {
            sums[ty][tx] = sum;
            __syncthreads();
            if (ty == 0 && p0 + tx < HW) {
                int32_t s = 0;
#pragma unroll
                for (int j = 0; j < kThreads / 32; ++j) s += sums[j][tx];
                psum[b * HW + p0 + tx] = s;
            }
            __syncthreads();
        }
    }
}

// ---- padded codes (integer modes for row lengths and channel counts off the GEMM's granule, DESIGN §7f): the recipe of
// quantize_rows_kernel, the pad columns / channels holding the code of zx and counted in the sums.
// Rows: qx [M][ldc] of x [M][K], ldc % 4 == 0.  G lanes (a power of two <= 32) share a row, each writing whole 32-bit
// words, so that short rows (a channels_last stem: K = 3, ldc = 4) still give one row per thread and coalesced stores.
template <typename T>
__global__ void __launch_bounds__(kThreads) quantize_rows_pad_kernel(const T* __restrict__ x, uint8_t* __restrict__ codes,
                                                                      int32_t* __restrict__ rowsum, int64_t M, int64_t K,
                                                                      int64_t ldc, int G, float scale, int32_t zp,
                                                                      int32_t qmin, int32_t qmax) {
    using Op = AffineOp<false>;
    AffineArgs a;                                   // only the fields AffineOp::make reads
    a.qmin = qmin;
    a.qmax = qmax;
    const Op::ChanParams p = Op::make(scale, zp, a);
    pdl_wait();
    pdl_launch_dependents();
    const int sub = threadIdx.x & (G - 1);
    const int64_t per_cta = kThreads / G, words = ldc / 4;
    // the row loop is uniform across the CTA: every lane reaches the shuffles
    for (int64_t base = (int64_t)blockIdx.x * per_cta; base < M; base += (int64_t)gridDim.x * per_cta) {
        const int64_t row = base + threadIdx.x / G;
        int32_t sum = 0;
        if (row < M) {
            const T* xr = x + row * K;
            uint32_t* cr = reinterpret_cast<uint32_t*>(codes + row * ldc);
            for (int64_t w = sub; w < words; w += G) {
                uint32_t word = 0;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    int c = zp;
                    if (4 * w + e < K) Op::template apply<true>(to_f32<T>(xr[4 * w + e]), p, c);
                    sum += c;
                    word |= (uint32_t)(c & 0xff) << (8 * e);
                }
                cr[w] = word;
            }
        }
        if (rowsum) {
            for (int d = G >> 1; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
            if (row < M && sub == 0) rowsum[row] = sum;
        }
    }
}

// NHWC codes with a channel pitch Cp of an NCHW x [N][C][HW]: one pixel per thread, V codes per store (V = Cp for Cp 4 / 8,
// else 16: Cp % 16 == 0).  Each channel's load runs along HW across the warp and each store along the pixels, so both
// sides stay coalesced for tiny C; P[pixel] is the sum over all Cp codes.
template <typename T, int V>
__global__ void __launch_bounds__(kThreads) quantize_nhwc_pad_kernel(const T* __restrict__ x, uint8_t* __restrict__ codes,
                                                                      int32_t* __restrict__ psum, int64_t N, int64_t C,
                                                                      int64_t HW, int64_t Cp, float scale, int32_t zp,
                                                                      int32_t qmin, int32_t qmax) {
    using Op = AffineOp<false>;
    AffineArgs a;                                   // only the fields AffineOp::make reads
    a.qmin = qmin;
    a.qmax = qmax;
    const Op::ChanParams p = Op::make(scale, zp, a);
    pdl_wait();
    pdl_launch_dependents();
    const int64_t ptiles = (HW + kThreads - 1) / kThreads;
    for (int64_t t = blockIdx.x; t < N * ptiles; t += gridDim.x) {
        const int64_t b = t / ptiles, px = (t - b * ptiles) * kThreads + threadIdx.x;
        if (px >= HW) continue;
        const T* xp = x + b * C * HW + px;
        uint8_t* cp = codes + (b * HW + px) * Cp;
        int32_t sum = 0;
        for (int64_t c0 = 0; c0 < Cp; c0 += V) {
            uint32_t w[V / 4];
#pragma unroll
            for (int i = 0; i < V / 4; ++i) w[i] = 0;
#pragma unroll
            for (int e = 0; e < V; ++e) {
                int q = zp;
                if (c0 + e < C) Op::template apply<true>(to_f32<T>(xp[(c0 + e) * HW]), p, q);
                sum += q;
                w[e / 4] |= (uint32_t)(q & 0xff) << (8 * (e % 4));
            }
            if constexpr (V == 4) *reinterpret_cast<uint32_t*>(cp + c0) = w[0];
            else if constexpr (V == 8) *reinterpret_cast<uint2*>(cp + c0) = make_uint2(w[0], w[1]);
            else *reinterpret_cast<uint4*>(cp + c0) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        if (psum) psum[b * HW + px] = sum;
    }
}

// ---- depthwise convolution of Q's codes (integer convolution mode, mctq_packed_dwconv2d_i8): x is read once as floats and
// quantized in registers by the recipe of quantize_rows_kernel; only qx - zx reaches shared memory (0 for taps outside the
// image), and the centred sum needs neither Sx nor Sw.  A work unit is S "slots" times a TH x TW tile of output pixels:
//   NCHW  a slot is one (b, c) plane, S consecutive planes per unit (S > 1 for small planes); loads run along W
//   NHWC  a slot is one channel of image b, S consecutive channels; loads run along C
// The window tile [IH][IW][SB] holds the slots innermost (SB: S rounded to an odd number of 32-bit words, so that the
// transposing stores of the NCHW path spread over the banks).  Each unit then walks the channel multiplier t: the m output
// channels o = c * m + t of every slot reuse the staged tile, their kh * kw codes decoded once into qw - zw.
struct DwArgs {
    const void* x;
    void* y;
    const uint8_t* codes;            // weight codes / LUT indices [Cout][K]
    const int32_t* w_zp;             // affine: zw [1 or Cout]; LUT: null (zw = 0)
    const float* factor;             // f [1 or Cout]
    const void* bias;                // [Cout] of T, or null
    int64_t units, groups, nplanes;  // work units; slot groups; N * C
    int32_t H, W, C, Cout, Ho, Wo, m, K, kh, kw, sh, sw, dh, dw, pt, pl;
    int32_t S, SB, TH, TW, IH, IW, tiles_x, tiles_y;
    int32_t kind, w_signed, per_channel;
    float x_scale;
    int32_t x_zp, x_qmin, x_qmax;
    FastDiv div_S, div_npix, div_IW, div_nout, div_TW;
    int8_t lut[256];                 // LUT kinds: the centroid codes (by value: no device copy)
};

// qw - zw of weight element i (LUT kinds: the centroid code of its index, zw = 0)
__device__ __forceinline__ int dw_weight(const DwArgs& a, int64_t i, int32_t zw) {
    const bool nib = a.kind == MCTQ_PACK_AFFINE_I4 || a.kind == MCTQ_PACK_LUT_I4;
    const uint32_t byte = __ldg(a.codes + (nib ? i >> 1 : i));
    const uint32_t u = nib ? ((i & 1) ? byte >> 4 : byte & 15u) : byte;
    if (a.kind == MCTQ_PACK_LUT_U8 || a.kind == MCTQ_PACK_LUT_I4) return a.lut[u];
    const int q = !a.w_signed ? (int)u : nib ? (int)(u ^ 8u) - 8 : (int)(int8_t)u;
    return q - zw;
}

// KS: 3 for a 3x3 kernel (taps unrolled, the thread's weights held in registers), 0 for any other kernel.  At most 40
// registers, so that six CTAs share an SM and hide each other's staging (eight would spill)
template <typename T, bool NHWC, int KS>
__global__ void __launch_bounds__(kThreads, 6) packed_dwconv_kernel(const __grid_constant__ DwArgs a) {
    using Op = AffineOp<false>;
    AffineArgs aa;                                  // only the fields AffineOp::make reads
    aa.qmin = a.x_qmin;
    aa.qmax = a.x_qmax;
    const Op::ChanParams p = Op::make(a.x_scale, a.x_zp, aa);
    extern __shared__ __align__(16) uint8_t dw_smem[];
    int64_t* soff = reinterpret_cast<int64_t*>(dw_smem);      // [S] y offset of slot s's output plane / channel
    float* sf = reinterpret_cast<float*>(soff + a.S);           // [S] f[o]
    float* sbias = sf + a.S;                                    // [S] bias[o]
    int32_t* so = reinterpret_cast<int32_t*>(sbias + a.S);      // [S] o, or -1 for a slot past the last plane / channel
    int32_t* ws = so + a.S;                                     // [K][S] qw - zw
    int16_t* xs = reinterpret_cast<int16_t*>(ws + (size_t)a.K * a.S);    // [IH * IW][SB] qx - zx
    pdl_wait();
    pdl_launch_dependents();
    const T* x = reinterpret_cast<const T*>(a.x);
    T* y = reinterpret_cast<T*>(a.y);
    const int KH = KS ? KS : a.kh, KW = KS ? KS : a.kw;
    const uint32_t S = (uint32_t)a.S, npix = (uint32_t)(a.IH * a.IW), nout = (uint32_t)(a.TH * a.TW);
    const int64_t per_group = (int64_t)a.tiles_y * a.tiles_x, HW = (int64_t)a.H * a.W;
    for (int64_t u = blockIdx.x; u < a.units; u += gridDim.x) {
        const int64_t g = u / per_group;
        const int32_t t2 = (int32_t)(u - g * per_group), ty = t2 / a.tiles_x, tx = t2 - ty * a.tiles_x;
        const int32_t ho0 = ty * a.TH, wo0 = tx * a.TW;
        const int64_t h0 = (int64_t)ho0 * a.sh - a.pt, w0 = (int64_t)wo0 * a.sw - a.pl;
        int64_t b = 0, first;                        // NHWC: image b and its first channel; NCHW: the first plane
        if (NHWC) {
            const int64_t cblocks = (a.C + a.S - 1) / a.S;
            b = g / cblocks;
            first = (g - b * cblocks) * a.S;
        } else {
            first = g * a.S;
        }
        const int64_t nslots = min((int64_t)a.S, (NHWC ? (int64_t)a.C : a.nplanes) - first);
        __syncthreads();                             // the previous unit is done with the shared tiles
        for (uint32_t e = threadIdx.x; e < npix * S; e += kThreads) {
            uint32_t s, pix;
            if (NHWC) { pix = fdiv_u32(e, a.div_S); s = e - pix * S; }           // channels innermost: coalesced along C
            else { s = fdiv_u32(e, a.div_npix); pix = e - s * npix; }            // columns innermost: coalesced along W
            const uint32_t iy = fdiv_u32(pix, a.div_IW), ix = pix - iy * (uint32_t)a.IW;
            const int64_t h = h0 + iy, w = w0 + ix;
            int v = 0;
            if ((int64_t)s < nslots && h >= 0 && h < a.H && w >= 0 && w < a.W) {
                const int64_t off = NHWC ? ((b * a.H + h) * a.W + w) * a.C + first + s : (first + s) * HW + h * a.W + w;
                int q;
                Op::template apply<true>(to_f32<T>(x[off]), p, q);
                v = q - a.x_zp;
            }
            xs[pix * a.SB + s] = (int16_t)v;
        }
        for (int32_t t = 0; t < a.m; ++t) {
            if (threadIdx.x < S) {
                const uint32_t s = threadIdx.x;
                int32_t o = -1;
                if ((int64_t)s < nslots) {
                    const int64_t plane = first + s;
                    const int64_t bb = NHWC ? b : plane / a.C, c = NHWC ? plane : plane - bb * a.C;
                    o = (int32_t)(c * a.m + t);
                    const int ch = a.per_channel ? o : 0;
                    soff[s] = NHWC ? (int64_t)o : (bb * a.Cout + o) * ((int64_t)a.Ho * a.Wo);
                    sf[s] = __ldg(a.factor + ch);
                    sbias[s] = a.bias ? to_f32<T>(reinterpret_cast<const T*>(a.bias)[o]) : 0.0f;
                }
                so[s] = o;
            }
            __syncthreads();                         // slot parameters set; the tile is staged (t = 0)
            for (uint32_t e = threadIdx.x; e < (uint32_t)a.K * S; e += kThreads) {
                const uint32_t k = fdiv_u32(e, a.div_S), s = e - k * S;
                const int32_t o = so[s];
                int v = 0;
                if (o >= 0) v = dw_weight(a, (int64_t)o * a.K + k, a.w_zp ? __ldg(a.w_zp + (a.per_channel ? o : 0)) : 0);
                ws[e] = v;
            }
            __syncthreads();
            int wr[KS ? KS * KS : 1];
            uint32_t wslot = 0xffffffffu;
            for (uint32_t q = threadIdx.x; q < nout * S; q += kThreads) {
                uint32_t s, pix;
                if (NHWC) { pix = fdiv_u32(q, a.div_S); s = q - pix * S; }        // lanes along C: coalesced NHWC stores
                else { s = fdiv_u32(q, a.div_nout); pix = q - s * nout; }          // lanes along W: coalesced plane stores
                const uint32_t oy = fdiv_u32(pix, a.div_TW), ox = pix - oy * (uint32_t)a.TW;
                const int32_t ho = ho0 + (int32_t)oy, wo = wo0 + (int32_t)ox;
                if (so[s] < 0 || ho >= a.Ho || wo >= a.Wo) continue;
                const int16_t* xw = xs + ((size_t)oy * a.sh * a.IW + (size_t)ox * a.sw) * a.SB + s;
                int32_t acc = 0;
                if (KS) {
                    if (s != wslot) {
#pragma unroll
                        for (int k = 0; k < KS * KS; ++k) wr[k] = ws[k * S + s];
                        wslot = s;
                    }
#pragma unroll
                    for (int r = 0; r < KS; ++r)
#pragma unroll
                        for (int c = 0; c < KS; ++c)
                            acc += (int)xw[((size_t)r * a.dh * a.IW + (size_t)c * a.dw) * a.SB] * wr[r * KS + c];
                } else {
                    for (int r = 0; r < KH; ++r)
                        for (int c = 0; c < KW; ++c)
                            acc += (int)xw[((size_t)r * a.dh * a.IW + (size_t)c * a.dw) * a.SB] * ws[(r * KW + c) * S + s];
                }
                float v = __fmul_rn(__int2float_rn(acc), sf[s]);
                if (a.bias) v = __fadd_rn(v, sbias[s]);
                const int64_t pix_off = NHWC ? ((b * a.Ho + ho) * a.Wo + wo) * a.Cout : (int64_t)ho * a.Wo + wo;
                y[soff[s] + pix_off] = from_f32<T>(v);
            }
            __syncthreads();                         // the weights of t are read
        }
    }
}

}  // namespace mctq

using namespace mctq;

namespace {

int check_codes(int32_t qmin, int32_t qmax, int code_mode, const void* codes) {
    if (code_mode == MCTQ_CODES_NONE) return 0;
    if (!codes) return MCTQ_E_BADARG;
    if (code_mode == MCTQ_CODES_INT8) {
        if ((qmin >= -128 && qmax <= 127) || (qmin >= 0 && qmax <= 255)) return 0;
        return MCTQ_E_RANGE;
    }
    if (code_mode == MCTQ_CODES_INT4) {
        if ((qmin >= -8 && qmax <= 7) || (qmin >= 0 && qmax <= 15)) return 0;
        return MCTQ_E_RANGE;
    }
    return MCTQ_E_BADARG;
}

// bytes per vector: 16, except channel-innermost layouts of 2-byte types (8: see fq_affine_kernel)
template <typename T, int CHMODE> constexpr int vec_bytes() { return (CHMODE == CH_LAST && sizeof(T) == 2) ? 8 : 16; }

template <typename T, int CHMODE, int CODE, int UNROLL_IN, bool RINT, bool PREP = false>
int launch_affine_tiles(const AffineArgs& a_in, cudaStream_t st) {
    constexpr int VB = vec_bytes<T, CHMODE>();
    constexpr int UNROLL = UNROLL_IN * 16 / VB;            // same bytes in flight per thread
    constexpr int V = VB / sizeof(T);
    constexpr uint32_t TILE = kThreads * UNROLL * V;
    AffineArgs a = a_in;
    size_t smem = 0;
    if (CHMODE == CH_LAST) {
        a.div_W = make_fastdiv((uint32_t)a.C);
        a.div_period = make_fastdiv(a.period);
        smem = (size_t)a.period * 3 * sizeof(float);
        int rc = ensure_smem(fq_affine_kernel<T, CHMODE, CODE, UNROLL, RINT, PREP, VB>, smem);
        if (rc) return rc;
    } else if (CHMODE != CH_PT) {
        set_window(a, TILE);
        smem = (size_t)a.W * (PREP ? 4 : 3) * sizeof(float);
        int rc = ensure_smem(fq_affine_kernel<T, CHMODE, CODE, UNROLL, RINT, PREP, VB>, smem);
        if (rc) return rc;
    }
    int64_t tiles = (a.n + TILE - 1) / TILE;
    if (tiles > 0x7fffffffLL) return MCTQ_E_BADARG;
    const IoSpan in[1] = {{a.x, (size_t)a.n * sizeof(T)}};
    const IoSpan out[2] = {{a.y, (size_t)a.n * sizeof(T)}, {a.codes, CODE == MCTQ_CODES_INT4 ? (size_t)(a.n + 1) / 2 : (size_t)a.n}};
    if (PREP && CHMODE != CH_PT) {
        const IoSpan tables = {a.prep_flags, prep_bytes(a.C)};            // the blob starts with its flags word
        a.early = (uint32_t)pdl_plan_launch(st, in, 1, out, CODE != 0 ? 2 : 1, &tables, &a.tab_early);
        if (!a.tab_early) a.early = 0;
    } else {
        a.early = (uint32_t)pdl_plan_launch(st, in, 1, out, CODE != 0 ? 2 : 1);
    }
    return launch_planned(fq_affine_kernel<T, CHMODE, CODE, UNROLL, RINT, PREP, VB>, (unsigned)tiles, smem, st, a);
}

// prepared parameters: TMA-staged variants (fast range, unroll 4, every code mode)
template <typename T, int CHMODE>
int launch_affine_prepared(const AffineArgs& a, int code_mode, cudaStream_t st) {
    switch (code_mode) {
        case MCTQ_CODES_INT8: return launch_affine_tiles<T, CHMODE, MCTQ_CODES_INT8, 4, false, true>(a, st);
        case MCTQ_CODES_INT4: return launch_affine_tiles<T, CHMODE, MCTQ_CODES_INT4, 4, false, true>(a, st);
        default: return launch_affine_tiles<T, CHMODE, MCTQ_CODES_NONE, 4, false, true>(a, st);
    }
}

// 16-byte vectors in flight per thread: 8 KB tiles for plain per-tensor fake-quant (nothing to stage per tile;
// tools/stream_probe.cu measures +2 % over 16 KB tiles), 16 KB tiles otherwise.  (4 KB tiles were measured in round 2 and
// are slower at every size: 74 MB 5.72 -> 5.16 TB/s queued, 295 MB 6.63 -> 5.94, 1 GB 6.91 -> 6.16 for bf16; the ~3 us a
// mid-size launch loses are drain + ramp, not tile granularity.)
template <int CHMODE, int CODE, bool RINT> constexpr int affine_unroll() { return CHMODE == CH_PT && CODE == MCTQ_CODES_NONE && !RINT ? 2 : 4; }

template <typename T, int CHMODE, bool RINT>
int launch_affine_code(const AffineArgs& a, int code_mode, cudaStream_t st) {
    switch (code_mode) {
        case MCTQ_CODES_INT8: return launch_affine_tiles<T, CHMODE, MCTQ_CODES_INT8, affine_unroll<CHMODE, MCTQ_CODES_INT8, RINT>(), RINT>(a, st);
        case MCTQ_CODES_INT4: return launch_affine_tiles<T, CHMODE, MCTQ_CODES_INT4, affine_unroll<CHMODE, MCTQ_CODES_INT4, RINT>(), RINT>(a, st);
        default: return launch_affine_tiles<T, CHMODE, MCTQ_CODES_NONE, affine_unroll<CHMODE, MCTQ_CODES_NONE, RINT>(), RINT>(a, st);
    }
}

template <typename T>
int launch_affine_typed(const AffineArgs& a, int code_mode, cudaStream_t st) {
    constexpr int V = 16 / sizeof(T);
    const bool rint_path = !(a.qmax - (int64_t)a.qmin < kFastRangeLimit);
    // vector path needs 16-byte aligned x / y and suitably aligned codes
    bool vec_ok = aligned16(a.x) && (!a.y || aligned16(a.y));
    if (code_mode != MCTQ_CODES_NONE) vec_ok = vec_ok && (reinterpret_cast<uintptr_t>(a.codes) & 7u) == 0;
    if (!vec_ok) {
        if (code_mode == MCTQ_CODES_INT4) return MCTQ_E_BADARG;
        int64_t blocks = (a.n + kThreads - 1) / kThreads;
        if (blocks > 148 * 64) blocks = 148 * 64;
        if (rint_path) fq_affine_scalar_kernel<T, true><<<(unsigned)blocks, kThreads, 0, st>>>(a);
        else fq_affine_scalar_kernel<T, false><<<(unsigned)blocks, kThreads, 0, st>>>(a);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return cuda_rc(cudaGetLastError());
    }
    int chmode;
    AffineArgs a2 = a;
    if (a.C == 1) chmode = CH_PT;
    else if (a.inner % V == 0 && a.elem_offset % V == 0) chmode = CH_VEC;
    else {
        chmode = CH_ELEM;
        constexpr int VL = vec_bytes<T, CH_LAST>() / sizeof(T);       // elements per vector in CH_LAST mode
        if (a.inner == 1 && a.elem_offset % VL == 0 && a.C <= 4096) {
            // channel-innermost layout: one period of the channel pattern (lcm(C, VL) entries, <= 48 KB) in shared memory
            uint64_t g = (uint64_t)a.C, h = VL;
            while (h) { uint64_t t = g % h; g = h; h = t; }
            const uint64_t period = (uint64_t)a.C / g * VL;
            if (period <= 4096) { chmode = CH_LAST; a2.period = (uint32_t)period; }
        }
    }
    if (a.prep_rec && !rint_path) {
        // prepared blob: bulk-copy staging needs 16-byte granules (CH_LAST: whole arrays of C floats)
        if (chmode == CH_VEC) return launch_affine_prepared<T, CH_VEC>(a2, code_mode, st);
        if (chmode == CH_ELEM) return launch_affine_prepared<T, CH_ELEM>(a2, code_mode, st);
        if (chmode == CH_LAST && a.C % 4 == 0) return launch_affine_prepared<T, CH_LAST>(a2, code_mode, st);
    }
#define MCTQ_DISPATCH_AFF(CM)                                                                   \
    return rint_path ? launch_affine_code<T, CM, true>(a2, code_mode, st) : launch_affine_code<T, CM, false>(a2, code_mode, st)
    if (chmode == CH_PT) { MCTQ_DISPATCH_AFF(CH_PT); }
    if (chmode == CH_VEC) { MCTQ_DISPATCH_AFF(CH_VEC); }
    if (chmode == CH_LAST) { MCTQ_DISPATCH_AFF(CH_LAST); }
    MCTQ_DISPATCH_AFF(CH_ELEM);
#undef MCTQ_DISPATCH_AFF
}

int launch_affine(const AffineArgs& a, int x_dtype, int code_mode, cudaStream_t st) {
    if (a.n < 0 || a.C < 1 || a.inner < 1 || a.elem_offset < 0 || !a.x || (!a.y && code_mode == MCTQ_CODES_NONE))
        return MCTQ_E_BADARG;
    if (a.qmin > a.qmax) return MCTQ_E_RANGE;
    int rc = check_codes(a.qmin, a.qmax, code_mode, a.codes);
    if (rc) return rc;
    if (a.n == 0) return 0;
    switch (x_dtype) {
        case MCTQ_F32: return launch_affine_typed<float>(a, code_mode, st);
        case MCTQ_BF16: return launch_affine_typed<__nv_bfloat16>(a, code_mode, st);
        case MCTQ_F16: return launch_affine_typed<__half>(a, code_mode, st);
        default: return MCTQ_E_DTYPE;
    }
}

// shared-memory bytes of packed_dwconv_kernel for the tile in `a`
size_t dw_smem_bytes(const DwArgs& a) {
    return (size_t)a.S * (8 + 4 + 4 + 4) + (size_t)a.K * a.S * 4 + (size_t)a.IH * a.IW * a.SB * 2;
}

// the tile of a work unit: about 2048 outputs, S slots, shrunk until the window tile fits shared memory (0, or MCTQ_E_RANGE
// for a dilated window too wide even for one output row of one slot)
int dw_plan(DwArgs& a, bool nhwc) {
    constexpr int64_t kOut = 2048;
    const int64_t plane = (int64_t)a.Ho * a.Wo;
    if (nhwc) {
        a.S = 32;
        a.TW = (int32_t)std::min<int64_t>(a.Wo, 16);
        a.TH = (int32_t)std::min<int64_t>(a.Ho, 8);
    } else {
        a.S = (int32_t)std::max<int64_t>(1, std::min<int64_t>({32, kOut / plane, a.nplanes}));
        a.TW = (int32_t)std::min<int64_t>(a.Wo, 64);
        a.TH = (int32_t)std::min<int64_t>(a.Ho, std::max<int64_t>(1, kOut / ((int64_t)a.S * a.TW)));
    }
    for (;;) {
        const int64_t ih = (int64_t)(a.TH - 1) * a.sh + (int64_t)(a.kh - 1) * a.dh + 1;
        const int64_t iw = (int64_t)(a.TW - 1) * a.sw + (int64_t)(a.kw - 1) * a.dw + 1;
        a.SB = 2 * (((a.S + 1) / 2) | 1);
        if (ih * iw * a.SB < (1LL << 31)) {
            a.IH = (int32_t)ih;
            a.IW = (int32_t)iw;
            if (dw_smem_bytes(a) <= 200 * 1024) return 0;
        }
        if (a.TH > 1) a.TH = (a.TH + 1) / 2;
        else if (a.S > 1) a.S = (a.S + 1) / 2;
        else if (a.TW > 1) a.TW = (a.TW + 1) / 2;
        else return MCTQ_E_RANGE;
    }
}

// the geometry checks of mctq_packed_dwconv2d_i8 and its plan query
int dw_check_geometry(const MctqConv2dGeom* g, int64_t Cout, int x_nhwc) {
    if (!g) return MCTQ_E_BADARG;
    if (g->N < 0 || g->H < 1 || g->W < 1 || g->Cin < 1 || g->Ho < 1 || g->Wo < 1 || g->kh < 1 || g->kw < 1 || g->sh < 1 ||
        g->sw < 1 || g->dh < 1 || g->dw < 1 || g->pt < 0 || g->pb < 0 || g->pl < 0 || g->pr < 0 || (x_nhwc != 0 && x_nhwc != 1))
        return MCTQ_E_BADARG;
    if (Cout < 1 || Cout % g->Cin != 0) return MCTQ_E_BADARG;
    return 0;
}

// the geometry fields of DwArgs that dw_plan reads, on a zeroed `a`
void dw_set_geometry(DwArgs& a, const MctqConv2dGeom* g, int64_t Cout) {
    memset(&a, 0, sizeof(a));
    a.nplanes = (int64_t)g->N * g->Cin;
    a.H = g->H; a.W = g->W; a.C = g->Cin; a.Cout = (int32_t)Cout; a.Ho = g->Ho; a.Wo = g->Wo;
    a.m = (int32_t)(Cout / g->Cin); a.K = (int32_t)((int64_t)g->kh * g->kw); a.kh = g->kh; a.kw = g->kw;   // K <= 33025
    a.sh = g->sh; a.sw = g->sw; a.dh = g->dh; a.dw = g->dw; a.pt = g->pt; a.pl = g->pl;
}

}  // namespace

extern "C" {

int mctq_fq_affine(const void* x, void* y, void* codes, int64_t n, int x_dtype, const float* scale, const int32_t* zp,
                   int64_t C, int64_t inner, int64_t elem_offset, int32_t qmin, int32_t qmax, int code_mode,
                   void* stream) {
    MCTQ_NVTX("mctq_fq_affine");
    if (!scale || !zp) return MCTQ_E_BADARG;
    AffineArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.y = y; a.codes = codes; a.n = n; a.scale = scale; a.zp = zp;
    a.C = C; a.inner = C == 1 ? 1 : inner; a.elem_offset = C == 1 ? 0 : elem_offset; a.qmin = qmin; a.qmax = qmax;
    return launch_affine(a, x_dtype, code_mode, (cudaStream_t)stream);
}

size_t mctq_affine_prepared_bytes(int64_t C) { return C < 1 ? 0 : prep_bytes(C); }

int mctq_affine_prepare(const float* scale, const int32_t* zp, int64_t C, void* prepared_dev, size_t prepared_bytes, void* stream) {
    MCTQ_NVTX("mctq_affine_prepare");
    if (!scale || !zp || !prepared_dev || C < 1 || prepared_bytes < prep_bytes(C) || !aligned16(prepared_dev)) return MCTQ_E_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(prepared_dev, 0, kPrepHeaderBytes, st);
    if (e != cudaSuccess) return (int)e;
    const int64_t C4 = (C + 3) & ~(int64_t)3;
    int64_t blocks = (C4 + kThreads - 1) / kThreads;
    if (blocks > 148 * 8) blocks = 148 * 8;
    pdl_note_prepare(st, prepared_dev, prep_bytes(C));              // launches that follow stage this blob only after their wait
    affine_prepare_kernel<<<(unsigned)blocks, kThreads, 0, st>>>(scale, zp, C, C4, reinterpret_cast<uint8_t*>(prepared_dev));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cuda_rc(cudaGetLastError());
}

int mctq_fq_affine_prepared(const void* x, void* y, void* codes, int64_t n, int x_dtype, const void* prepared_dev, int64_t C,
                            int64_t inner, int64_t elem_offset, int32_t qmin, int32_t qmax, int code_mode, void* stream) {
    MCTQ_NVTX("mctq_fq_affine_prepared");
    if (!prepared_dev || C < 1 || !aligned16(prepared_dev)) return MCTQ_E_BADARG;
    const uint8_t* blob = reinterpret_cast<const uint8_t*>(prepared_dev);
    AffineArgs a;
    memset(&a, 0, sizeof(a));
    a.C4 = (C + 3) & ~(int64_t)3;
    a.prep_flags = reinterpret_cast<const int32_t*>(blob);
    a.prep_rec = reinterpret_cast<const float4*>(blob + kPrepHeaderBytes);
    a.prep_soa = reinterpret_cast<const float*>(blob + kPrepHeaderBytes + (size_t)C * 16);
    // the arrays inside the blob double as the raw parameters for the variants that do not use bulk staging
    a.scale = a.prep_soa + a.C4;
    a.zp = reinterpret_cast<const int32_t*>(a.prep_soa + 2 * a.C4);
    a.x = x; a.y = y; a.codes = codes; a.n = n;
    a.C = C; a.inner = C == 1 ? 1 : inner; a.elem_offset = C == 1 ? 0 : elem_offset; a.qmin = qmin; a.qmax = qmax;
    return launch_affine(a, x_dtype, code_mode, (cudaStream_t)stream);
}

int mctq_fq_affine_scalar(const void* x, void* y, void* codes, int64_t n, int x_dtype, float scale, int32_t zp,
                          int32_t qmin, int32_t qmax, int code_mode, void* stream) {
    MCTQ_NVTX("mctq_fq_affine_scalar");
    AffineArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.y = y; a.codes = codes; a.n = n; a.scale = nullptr; a.zp = nullptr; a.scale_val = scale; a.zp_val = zp;
    a.C = 1; a.inner = 1; a.elem_offset = 0; a.qmin = qmin; a.qmax = qmax;
    return launch_affine(a, x_dtype, code_mode, (cudaStream_t)stream);
}

int mctq_quantize_rows_i8(const void* x, int x_dtype, int64_t M, int64_t K, float scale, int32_t zp, int32_t qmin,
                          int32_t qmax, void* codes, int32_t* rowsum, void* stream) {
    MCTQ_NVTX("mctq_quantize_rows_i8");
    if (!x || !codes || M < 0 || K < 1) return MCTQ_E_BADARG;
    if (x_dtype != MCTQ_F32 && x_dtype != MCTQ_BF16 && x_dtype != MCTQ_F16) return MCTQ_E_DTYPE;
    if (qmin > qmax) return MCTQ_E_RANGE;
    if (int rc = check_codes(qmin, qmax, MCTQ_CODES_INT8, codes)) return rc;
    if (M == 0) return 0;
    const int64_t blocks = std::min<int64_t>((M + kThreads / 32 - 1) / (kThreads / 32), 148 * 16);
    const bool vec = K % 8 == 0 && aligned16(x) && (reinterpret_cast<uintptr_t>(codes) & 7u) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    auto run = [&](auto type) {
        using T = typename decltype(type)::type;
        const T* xt = reinterpret_cast<const T*>(x);
        uint8_t* c = reinterpret_cast<uint8_t*>(codes);
        if (vec) return launch_streaming(quantize_rows_kernel<T, true>, (unsigned)blocks, 0, st, xt, c, rowsum, M, K, scale, zp, qmin, qmax);
        return launch_streaming(quantize_rows_kernel<T, false>, (unsigned)blocks, 0, st, xt, c, rowsum, M, K, scale, zp, qmin, qmax);
    };
    if (x_dtype == MCTQ_F32) return run(PackType<float>{});
    if (x_dtype == MCTQ_BF16) return run(PackType<__nv_bfloat16>{});
    return run(PackType<__half>{});
}

int mctq_quantize_nhwc_i8(const void* x, int x_dtype, int64_t N, int64_t C, int64_t H, int64_t W, float scale, int32_t zp,
                          int32_t qmin, int32_t qmax, void* codes, int32_t* P, void* stream) {
    MCTQ_NVTX("mctq_quantize_nhwc_i8");
    if (!x || !codes || N < 0 || C < 1 || H < 1 || W < 1) return MCTQ_E_BADARG;
    if (x_dtype != MCTQ_F32 && x_dtype != MCTQ_BF16 && x_dtype != MCTQ_F16) return MCTQ_E_DTYPE;
    if (qmin > qmax) return MCTQ_E_RANGE;
    if (int rc = check_codes(qmin, qmax, MCTQ_CODES_INT8, codes)) return rc;
    if (N == 0) return 0;
    const int64_t HW = H * W;
    const int64_t blocks = std::min<int64_t>(N * ((HW + 31) / 32), 148 * 16);
    cudaStream_t st = (cudaStream_t)stream;
    auto run = [&](auto type) {
        using T = typename decltype(type)::type;
        return launch_streaming(quantize_nhwc_kernel<T>, (unsigned)blocks, 0, st, reinterpret_cast<const T*>(x),
                                reinterpret_cast<uint8_t*>(codes), P, N, C, HW, scale, zp, qmin, qmax);
    };
    if (x_dtype == MCTQ_F32) return run(PackType<float>{});
    if (x_dtype == MCTQ_BF16) return run(PackType<__nv_bfloat16>{});
    return run(PackType<__half>{});
}

int mctq_quantize_rows_i8_padded(const void* x, int x_dtype, int64_t M, int64_t K, int64_t ldc, float scale, int32_t zp,
                                 int32_t qmin, int32_t qmax, void* codes, int32_t* rowsum, void* stream) {
    MCTQ_NVTX("mctq_quantize_rows_i8_padded");
    if (!x || !codes || M < 0 || K < 1 || ldc < K || ldc % 4 != 0 || (reinterpret_cast<uintptr_t>(codes) & 3u) != 0)
        return MCTQ_E_BADARG;
    if (x_dtype != MCTQ_F32 && x_dtype != MCTQ_BF16 && x_dtype != MCTQ_F16) return MCTQ_E_DTYPE;
    if (qmin > qmax) return MCTQ_E_RANGE;
    if (int rc = check_codes(qmin, qmax, MCTQ_CODES_INT8, codes)) return rc;
    if (zp < qmin || zp > qmax) return MCTQ_E_RANGE;             // the pad columns hold zp as a code
    if (M == 0) return 0;
    int G = 1;
    while (G < 32 && 4 * G < ldc) G *= 2;
    const int64_t blocks = std::min<int64_t>((M + kThreads / G - 1) / (kThreads / G), 148 * 16);
    cudaStream_t st = (cudaStream_t)stream;
    auto run = [&](auto type) {
        using T = typename decltype(type)::type;
        return launch_streaming(quantize_rows_pad_kernel<T>, (unsigned)blocks, 0, st, reinterpret_cast<const T*>(x),
                                reinterpret_cast<uint8_t*>(codes), rowsum, M, K, ldc, G, scale, zp, qmin, qmax);
    };
    if (x_dtype == MCTQ_F32) return run(PackType<float>{});
    if (x_dtype == MCTQ_BF16) return run(PackType<__nv_bfloat16>{});
    return run(PackType<__half>{});
}

int mctq_quantize_nhwc_i8_padded(const void* x, int x_dtype, int64_t N, int64_t C, int64_t H, int64_t W, int64_t Cp,
                                 float scale, int32_t zp, int32_t qmin, int32_t qmax, void* codes, int32_t* P, void* stream) {
    MCTQ_NVTX("mctq_quantize_nhwc_i8_padded");
    if (!x || !codes || N < 0 || C < 1 || H < 1 || W < 1 || Cp < C || !aligned16(codes)) return MCTQ_E_BADARG;
    if (Cp != 4 && Cp != 8 && Cp % 16 != 0) return MCTQ_E_BADARG;
    if (x_dtype != MCTQ_F32 && x_dtype != MCTQ_BF16 && x_dtype != MCTQ_F16) return MCTQ_E_DTYPE;
    if (qmin > qmax) return MCTQ_E_RANGE;
    if (int rc = check_codes(qmin, qmax, MCTQ_CODES_INT8, codes)) return rc;
    if (zp < qmin || zp > qmax) return MCTQ_E_RANGE;
    if (N == 0) return 0;
    const int64_t HW = H * W;
    const int64_t blocks = std::min<int64_t>(N * ((HW + kThreads - 1) / kThreads), 148 * 16);
    cudaStream_t st = (cudaStream_t)stream;
    auto run = [&](auto type) {
        using T = typename decltype(type)::type;
        const T* xt = reinterpret_cast<const T*>(x);
        uint8_t* c = reinterpret_cast<uint8_t*>(codes);
        if (Cp == 4) return launch_streaming(quantize_nhwc_pad_kernel<T, 4>, (unsigned)blocks, 0, st, xt, c, P, N, C, HW, Cp, scale, zp, qmin, qmax);
        if (Cp == 8) return launch_streaming(quantize_nhwc_pad_kernel<T, 8>, (unsigned)blocks, 0, st, xt, c, P, N, C, HW, Cp, scale, zp, qmin, qmax);
        return launch_streaming(quantize_nhwc_pad_kernel<T, 16>, (unsigned)blocks, 0, st, xt, c, P, N, C, HW, Cp, scale, zp, qmin, qmax);
    };
    if (x_dtype == MCTQ_F32) return run(PackType<float>{});
    if (x_dtype == MCTQ_BF16) return run(PackType<__nv_bfloat16>{});
    return run(PackType<__half>{});
}

int mctq_packed_dwconv2d_i8(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cout, const void* x, int x_dtype,
                            int x_nhwc, float x_scale, int32_t x_zero_point, int32_t x_qmin, int32_t x_qmax,
                            const float* factor, const void* bias, void* y, const int8_t* lut_codes_host, void* stream) {
    MCTQ_NVTX("mctq_packed_dwconv2d_i8");
    if (!w || !g || !factor) return MCTQ_E_BADARG;
    if (const int rc = dw_check_geometry(g, Cout, x_nhwc)) return rc;
    const int64_t K = (int64_t)g->kh * g->kw;
    // the weight as a [Cout][kh * kw] matrix: kind, dtype, extent, parameter layout, pointers
    if (const int rc = packed_linear_check(w, Cout, K, x, x_dtype, g->N, y)) return rc;
    if (pack_is_lut(w->kind) != (lut_codes_host != nullptr)) return MCTQ_E_BADARG;
    if (x_qmin > x_qmax) return MCTQ_E_RANGE;
    if (int rc = check_codes(x_qmin, x_qmax, MCTQ_CODES_INT8, x)) return rc;
    if (x_zero_point < x_qmin || x_zero_point > x_qmax || K > 33025) return MCTQ_E_RANGE;    // |qx - zx|, |qw - zw| <= 255
    if (g->N == 0) return 0;

    DwArgs a;
    dw_set_geometry(a, g, Cout);
    a.x = x;
    a.y = y;
    a.codes = reinterpret_cast<const uint8_t*>(w->codes);
    a.w_zp = pack_is_lut(w->kind) ? nullptr : w->zp;
    a.factor = factor;
    a.bias = bias;
    a.kind = w->kind; a.w_signed = w->is_signed ? 1 : 0; a.per_channel = w->C != 1;
    a.x_scale = x_scale; a.x_zp = x_zero_point; a.x_qmin = x_qmin; a.x_qmax = x_qmax;
    if (lut_codes_host) memcpy(a.lut, lut_codes_host, (size_t)w->K);
    if (const int rc = dw_plan(a, x_nhwc != 0)) return rc;
    a.tiles_y = (a.Ho + a.TH - 1) / a.TH;
    a.tiles_x = (a.Wo + a.TW - 1) / a.TW;
    a.groups = x_nhwc ? (int64_t)g->N * ((a.C + a.S - 1) / a.S) : (a.nplanes + a.S - 1) / a.S;
    a.units = a.groups * a.tiles_y * a.tiles_x;
    a.div_S = make_fastdiv((uint32_t)a.S);
    a.div_npix = make_fastdiv((uint32_t)(a.IH * a.IW));
    a.div_IW = make_fastdiv((uint32_t)a.IW);
    a.div_nout = make_fastdiv((uint32_t)(a.TH * a.TW));
    a.div_TW = make_fastdiv((uint32_t)a.TW);
    const size_t smem = dw_smem_bytes(a);
    const unsigned blocks = (unsigned)std::min<int64_t>(a.units, 148 * 8);
    cudaStream_t st = (cudaStream_t)stream;
    const bool k3 = g->kh == 3 && g->kw == 3;
    auto run = [&](auto type) {
        using T = typename decltype(type)::type;
        auto kernel = x_nhwc ? (k3 ? packed_dwconv_kernel<T, true, 3> : packed_dwconv_kernel<T, true, 0>)
                             : (k3 ? packed_dwconv_kernel<T, false, 3> : packed_dwconv_kernel<T, false, 0>);
        if (const int rc = ensure_smem(kernel, smem)) return rc;
        return launch_streaming(kernel, blocks, smem, st, a);
    };
    if (x_dtype == MCTQ_F32) return run(PackType<float>{});
    if (x_dtype == MCTQ_BF16) return run(PackType<__nv_bfloat16>{});
    return run(PackType<__half>{});
}

int mctq_packed_dwconv2d_i8_plan(const MctqConv2dGeom* g, int64_t Cout, int x_nhwc, MctqDwPlan* out) {
    if (!out) return MCTQ_E_BADARG;
    if (const int rc = dw_check_geometry(g, Cout, x_nhwc)) return rc;
    if ((int64_t)g->kh * g->kw > 33025) return MCTQ_E_RANGE;
    DwArgs a;
    dw_set_geometry(a, g, Cout);
    if (const int rc = dw_plan(a, x_nhwc != 0)) return rc;
    out->S = a.S;
    out->TH = a.TH;
    out->TW = a.TW;
    out->IH = a.IH;
    out->IW = a.IW;
    out->smem_bytes = (int32_t)dw_smem_bytes(a);
    return 0;
}

int mctq_dequant_affine(const void* codes, int code_mode, int is_signed, float* y, int64_t n, const float* scale,
                        const int32_t* zp, int64_t C, int64_t inner, int64_t elem_offset, void* stream) {
    MCTQ_NVTX("mctq_dequant_affine");
    if (!codes || !y || !scale || !zp || n < 0 || C < 1 || inner < 1) return MCTQ_E_BADARG;
    if (n == 0) return 0;
    if (code_mode != MCTQ_CODES_INT8 && code_mode != MCTQ_CODES_INT4) return MCTQ_E_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (aligned16(y) && (reinterpret_cast<uintptr_t>(codes) & 3u) == 0 && C < (1LL << 32) && inner < (1LL << 32)) {
        const int mode = C == 1 ? 0 : ((inner % 4 == 0 && elem_offset % 4 == 0) ? 1 : 2);
        // 8 codes per vector (32-byte aligned y, the vector inside one channel) only where it measured faster on the B200:
        // per-channel int4 (5.63 -> 6.14 TB/s; the channel look-up per vector halves).  Per-tensor and int8 variants are
        // at 6.3-6.4 TB/s with 4-code vectors and lose ~3 % with 8.
        const bool v8 = mode == 1 && code_mode == MCTQ_CODES_INT4 && aligned32(y) && inner % 8 == 0 && elem_offset % 8 == 0;
        const int64_t tile = (int64_t)kThreads * 4 * (v8 ? 8 : 4);
        const int64_t tiles = (n + tile - 1) / tile;
        if (tiles > 0x7fffffffLL) return MCTQ_E_BADARG;
        const uint32_t C32 = (uint32_t)C, in32 = (uint32_t)(C == 1 ? 1 : inner);
        const FastDiv di = make_fastdiv(in32), dc = make_fastdiv(C32);
#define MCTQ_DQ(CM, MD, VV) launch_streaming(dequant_affine_vec_kernel<CM, MD, VV>, (unsigned)tiles, 0, st, codes, is_signed, y, n, scale, zp, C32, in32, elem_offset, di, dc)
        if (code_mode == MCTQ_CODES_INT8)
            return mode == 0 ? MCTQ_DQ(MCTQ_CODES_INT8, 0, 4) : mode == 1 ? MCTQ_DQ(MCTQ_CODES_INT8, 1, 4) : MCTQ_DQ(MCTQ_CODES_INT8, 2, 4);
        if (v8) return MCTQ_DQ(MCTQ_CODES_INT4, 1, 8);
        return mode == 0 ? MCTQ_DQ(MCTQ_CODES_INT4, 0, 4) : mode == 1 ? MCTQ_DQ(MCTQ_CODES_INT4, 1, 4) : MCTQ_DQ(MCTQ_CODES_INT4, 2, 4);
#undef MCTQ_DQ
    }
    int64_t blocks = (n + kThreads - 1) / kThreads;
    if (blocks > 148 * 32) blocks = 148 * 32;
    if (code_mode == MCTQ_CODES_INT8)
        dequant_affine_kernel<MCTQ_CODES_INT8><<<(unsigned)blocks, kThreads, 0, st>>>(codes, is_signed, y, n, scale, zp, C, inner, elem_offset);
    else if (code_mode == MCTQ_CODES_INT4)
        dequant_affine_kernel<MCTQ_CODES_INT4><<<(unsigned)blocks, kThreads, 0, st>>>(codes, is_signed, y, n, scale, zp, C, inner, elem_offset);
    else return MCTQ_E_BADARG;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cuda_rc(cudaGetLastError());
}

int64_t mctq_multi_tile_elems(void) { return kMultiTile; }

int64_t mctq_multi_plan(const MctqTensorDesc* descs, int n_desc, int32_t* tile_starts) {
    if (!descs || !tile_starts || n_desc < 0) return MCTQ_E_BADARG;
    int64_t t = 0;
    for (int k = 0; k < n_desc; ++k) {
        if (descs[k].n < 0) return MCTQ_E_BADARG;
        tile_starts[k] = (int32_t)t;
        t += (descs[k].n + kMultiTile - 1) / kMultiTile;
        if (t > 0x7fffffffLL) return MCTQ_E_BADARG;
    }
    tile_starts[n_desc] = (int32_t)t;
    return t;
}

int mctq_fq_affine_multi(const MctqTensorDesc* descs_dev, const int32_t* tile_starts_dev, int n_desc,
                         int64_t total_tiles, void* stream) {
    MCTQ_NVTX("mctq_fq_affine_multi");
    if (!descs_dev || !tile_starts_dev || n_desc < 1 || total_tiles < 0 || total_tiles > 0x7fffffffLL) return MCTQ_E_BADARG;
    if (total_tiles == 0) return 0;
    return launch_streaming(fq_affine_multi_kernel, (unsigned)total_tiles, 0, (cudaStream_t)stream, descs_dev, tile_starts_dev, n_desc);
}

int mctq_fq_affine_scalar_multi(const MctqSiteDesc* sites, int n_sites, void* stream) {
    MCTQ_NVTX("mctq_fq_affine_scalar_multi");
    if (n_sites < 0 || (n_sites > 0 && !sites)) return MCTQ_E_BADARG;
    for (int k = 0; k < n_sites; ++k) {                     // validate everything before anything is launched
        const MctqSiteDesc& d = sites[k];
        if (d.n < 0 || (d.n > 0 && (!d.x || !d.y))) return MCTQ_E_BADARG;
        if (d.dtype != MCTQ_F32 && d.dtype != MCTQ_BF16 && d.dtype != MCTQ_F16) return MCTQ_E_DTYPE;
        if (d.qmin > d.qmax) return MCTQ_E_RANGE;
        if (d.n > 0 && (!aligned16(d.x) || !aligned16(d.y))) return MCTQ_E_BADARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    SitesParams p;
    int k = 0;
    while (k < n_sites) {
        memset(&p, 0, sizeof(p));
        int64_t tiles = 0;
        int m = 0;
        for (; k < n_sites && m < kSitesCap; ++k) {
            const MctqSiteDesc& d = sites[k];
            if (d.n == 0) continue;
            const int64_t tile_elems = (int64_t)kThreads * 2 * (d.dtype == MCTQ_F32 ? 4 : 8);
            const int64_t t = (d.n + tile_elems - 1) / tile_elems;
            if (tiles + t > 0x7fffffffLL) { if (m == 0) return MCTQ_E_BADARG; break; }       // next launch takes it
            SiteEntry& e = p.e[m];
            e.x = d.x; e.y = d.y; e.n = d.n; e.scale = d.scale; e.zp = d.zp; e.qmin = d.qmin; e.qmax = d.qmax; e.dtype = d.dtype;
            p.starts[m] = (int32_t)tiles;
            tiles += t;
            ++m;
        }
        if (m == 0) continue;
        p.n_sites = m;
        p.starts[m] = (int32_t)tiles;
        int rc = launch_streaming(fq_affine_sites_kernel, (unsigned)tiles, 0, st, p);
        if (rc) return rc;
    }
    return 0;
}

}  // extern "C"
