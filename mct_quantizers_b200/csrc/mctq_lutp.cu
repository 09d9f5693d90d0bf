// mctq_lutp.cu -- "prepared" LUT fake-quant: per-channel decision tables in the x domain.
//
// The reference normalises every element (x / (thr + eps)), scales, clips and runs an argmin over the centroids
// (mct_quantizers/pytorch/quantizer_utils.py:95-170).  All of that is a monotone function of x per channel, so the
// result is decided by which of the K - 1 per-channel thresholds X[c][j] = sup{x : normalised(x) <= tau_j} the element
// exceeds.  mctq_lut_prepare computes those thresholds EXACTLY, once per quantizer, by bisection over f32 bit patterns
// through the reference's own arithmetic (IEEE division, optional rounding to bf16 / f16, first-minimum thresholds
// of the search table).  The dequantised output is (lut_sorted[pos] / 2^(bw-s)) * thr_c: the quotients are a small
// channel-independent table, the product is one multiply per element (a first version staged the products per channel,
// which doubled the record: for rows of 64 elements the tables were then more L2 traffic than the data).
// The hot kernel then needs no division and no search loop: an approximate cell index (one saturating FMA)
// selects the single threshold that can still matter, one exact compare decides, one shared-memory load fetches y.
#include <algorithm>
#include <cmath>
#include <type_traits>
#include <utility>
#include <vector>

#include "mctq_common.cuh"
#include "mctq_lut_table.cuh"
#include "mctq_plan.cuh"

namespace mctq {

constexpr uint32_t kPrepMagic = 0x32515050u;   // 'PPQ2'
constexpr int kCellsPerUnitMax = 4;            // finest cell width = 1/4 of a step of the normalised grid (always valid)
constexpr float kCellSlop = 0.02f;             // cells; >> the 1e-4 cell error of the approximate index
constexpr float kMagicRound = 12582912.0f;     // 1.5 * 2^23
constexpr int kXyP = 16;                       // xy records: 16 thresholds + 16 outputs (centroid lists of <= 16 entries)
constexpr int kXyRecFloats = 2 * kXyP + 4;     // X[16] | Y[16] | s' thr d pad   (144 bytes)
constexpr int64_t kXyMaxC = 65536;             // xy records are built for quantizers of up to this many channels (9 MB)

// Layout of the prepared blob (device memory):
//   header | tau[P] | FRONT = consts(16 B: NCf, c0, NCd, -) cq[P] orig[P] cells[NC + 1] | thin records C x rec_floats | xy records C x 36
// FRONT is what every CTA stages: its length depends on the number of cells actually used (header.front_bytes).
struct LutPrepHeader {      // 96 bytes
    uint32_t magic;
    int32_t K, P, NC;       // centroids, padded table size, number of cells IN USE
    int64_t C;
    float mult;
    int32_t round_dtype;    // 0 none, 1 bf16, 2 f16 (activation flavour with half-precision inputs)
    int32_t pos0;           // sorted position of original index 0 (NaN inputs)
    int32_t rec_floats;     // floats per thin channel record: X[P] s' thr d pad
    int32_t off_tau, off_front, off_rec, off_xy;   // byte offsets into the blob (off_xy == 0: no xy records)
    int32_t orig_identity;  // sorted position == original LUT index for every reachable position
    int32_t front_bytes;    // bytes of FRONT that are in use (multiple of 16)
    int32_t cells_per_unit; // 1, 2 or 4 ...
    float cell_offset;      // cells are shifted by this fraction of a cell against the integer grid
    int32_t cells_shift;    // ... divided by 2^cells_shift (grids of more than 10 bits: cells coarser than the integer grid)
    int32_t reserved[5];
};
static_assert(sizeof(LutPrepHeader) == 96, "header layout");

struct PrepGeom {
    int P, NC, rec_floats;                      // NC = cell CAPACITY (finest geometry)
    size_t off_tau, off_front, off_rec, off_xy, bytes;
    uint32_t rel_cq, rel_orig, rel_cells, front_cap;     // offsets inside FRONT; its capacity in bytes
};

static inline int64_t cells_needed(int cells_per_unit, int64_t mult, int shift = 0) { return (((int64_t)cells_per_unit * 2 * mult) >> shift) + 8; }
constexpr int64_t kMaxCells = 4200;            // the byte-wide cell table has to fit comfortably in shared memory
// smallest shift for which the finest geometry (kCellsPerUnitMax >> shift cells per step) fits: 0 for grids of <= 10 bits
static inline int finest_shift(int64_t mult) {
    int sh = 0;
    while (cells_needed(kCellsPerUnitMax, mult, sh) > kMaxCells) ++sh;
    return sh;
}

static int prep_geometry(int K, int bw, int is_signed, int64_t C, PrepGeom* g) {
    int L;
    if (lut_geometry_from_K(K, &g->P, &L)) return MCTQ_E_LUT;
    if (bw < 1 || bw > 16 || C < 1) return MCTQ_E_LUT;
    const int64_t mult = 1LL << (bw - (is_signed ? 1 : 0));
    // grids of more than 10 bits: the cell grid is coarser than the integer grid (mctq_lut_prepare then checks that the
    // centroid list is sparse enough for it and returns MCTQ_E_RANGE otherwise)
    g->NC = (int)cells_needed(kCellsPerUnitMax, mult, finest_shift(mult));
    // everything the hot kernels stage with 16-byte bulk copies (FRONT, channel records) starts on a 16-byte boundary and
    // is a multiple of 16 bytes long, also for tables of one or two entries
    g->rec_floats = (g->P + 4 + 3) & ~3;
    auto up16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
    size_t o = sizeof(LutPrepHeader);
    g->off_tau = o; o = up16(o + (size_t)g->P * 4);
    g->off_front = o;
    g->rel_cq = 16;
    g->rel_orig = g->rel_cq + (uint32_t)up16((size_t)g->P * 4);
    g->rel_cells = g->rel_orig + (uint32_t)up16((size_t)g->P);
    g->front_cap = g->rel_cells + (uint32_t)up16((size_t)g->NC + 1);
    o += g->front_cap;
    g->off_rec = o; o += (size_t)C * g->rec_floats * 4;
    g->off_xy = 0;
    if (g->P <= kXyP && C <= kXyMaxC) { g->off_xy = o; o += (size_t)C * kXyRecFloats * 4; }
    g->bytes = o;
    return 0;
}

__host__ __device__ inline float round_like(float q, int round_dtype) {
    if (round_dtype == 1) return __bfloat162float(__float2bfloat16_rn(q));
    if (round_dtype == 2) return __half2float(__float2half_rn(q));
    return q;
}

__host__ __device__ inline int32_t f2ord(float f) {
    int32_t i = (int32_t)
#ifdef __CUDA_ARCH__
        __float_as_int(f);
#else
        [](float v) { int32_t r; memcpy(&r, &v, 4); return r; }(f);
#endif
    return i < 0 ? (int32_t)(0x80000000u - (uint32_t)i) : i;
}
__host__ __device__ inline float ord2f(int32_t o) {
    int32_t i = o < 0 ? (int32_t)(0x80000000u - (uint32_t)o) : o;
#ifdef __CUDA_ARCH__
    return __int_as_float(i);
#else
    float f; memcpy(&f, &i, 4); return f;
#endif
}

// ---- prepare kernel: one thread per (channel, table position)
__global__ void __launch_bounds__(kThreads) lut_prepare_kernel(uint8_t* blob, const float* thr, float eps, int scalar_mode,
                                                               float divisor, float thr_f32) {
    const LutPrepHeader h = *reinterpret_cast<const LutPrepHeader*>(blob);
    const float* tau = reinterpret_cast<const float*>(blob + h.off_tau);
    const float* cq = reinterpret_cast<const float*>(blob + h.off_front + 16);
    float* rec = reinterpret_cast<float*>(blob + h.off_rec);
    float* xy = h.off_xy ? reinterpret_cast<float*>(blob + h.off_xy) : nullptr;
    const int64_t total = h.C * h.P;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < total; i += (int64_t)gridDim.x * kThreads) {
        const int64_t c = i / h.P;
        const int j = (int)(i - c * h.P);
        float d, t;
        if (scalar_mode) { d = divisor; t = thr_f32; }
        else { t = thr[c]; d = __fadd_rn(t, eps); }
        float* r = rec + c * h.rec_floats;
        if (j == 0) {
            // approximate cell scale: u = x * s' + 0.5, cell = round(u * NC)
            const float cm = __fmul_rn(ldexpf((float)h.cells_per_unit, -h.cells_shift), h.mult);       // power-of-two factors: exact
            r[h.P] = (scalar_mode == 2 ? __fmul_rn(cm, d) : __fdiv_rn(cm, d)) / (float)h.NC;
            r[h.P + 1] = t;                                                 // y = cq[pos] * thr_c (thr WITHOUT eps)
            r[h.P + 2] = d;
            if (xy) {
                float* q = xy + c * kXyRecFloats;
                q[2 * kXyP] = r[h.P];
                q[2 * kXyP + 1] = t;
                q[2 * kXyP + 2] = d;
                q[2 * kXyP + 3] = 0.0f;
                for (int k = h.P; k < kXyP; ++k) { q[k] = INFINITY; q[kXyP + k] = 0.0f; }
            }
        }
        float X = INFINITY;
        if (j < h.P - 1) {
            const float tj = tau[j];
            if (tj == -INFINITY) X = -INFINITY;
            else if (tj != INFINITY) {
                // P(x) := round_like(x / d) > tau_j is monotone in x (d > 0); X = largest x for which it is false
                // scalar_mode 2: d is the multiplier f32(1 / (thr + eps)) of the reference's CUDA flavour (monotone as well)
                auto above = [&](float x) { return round_like(scalar_mode == 2 ? __fmul_rn(x, d) : __fdiv_rn(x, d), h.round_dtype) > tj; };
                const float big = 3.4028234663852886e38f;
                if (above(-big)) X = -INFINITY;
                else if (!above(big)) X = big;
                else {
                    int64_t lo = f2ord(-big), hi = f2ord(big);
                    while (hi - lo > 1) {
                        int64_t mid = lo + (hi - lo) / 2;
                        if (above(ord2f((int32_t)mid))) hi = mid; else lo = mid;
                    }
                    X = ord2f((int32_t)lo);
                }
            }
        }
        r[j] = X;
        if (xy) {
            float* q = xy + c * kXyRecFloats;
            q[j] = X;
            q[kXyP + j] = __fmul_rn(cq[j], t);                              // the product the thin kernel forms per element
        }
    }
}

// ---- hot kernel
struct LutPArgs {
    const void* x;
    float* y;
    void* idx;
    int64_t n;
    const uint8_t* blob;
    int32_t P, NC, rec_floats;                 // NC: cell capacity (shared-memory sizing); the cells in use come with FRONT
    int32_t off_front, off_rec, off_xy;
    uint32_t rel_cq, rel_orig, rel_cells, front_cap;
    int64_t C, inner, elem_offset;
    FastDiv div_inner, div_W;
    uint32_t W, bigrow;
    uint32_t early;          // dependent-launch order: 0 late, 1 early, 2 free (opt-in, see pdl_plan_launch)
    uint32_t tab_early;      // the tables may be staged before the dependent-launch wait (the blob is not being written)
};

__device__ __forceinline__ float fma_sat(float a, float b, float c) {
    float r;
    asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// V: elements per vector.  4 everywhere (8-byte loads of 2-byte types, one 16-byte f32 store), or 8 for 2-byte types when
// the whole vector lies in one channel (CH_PT, CH_VEC with rows that are a multiple of 8): one 16-byte load, one 32-byte
// store (STG.256), half the per-vector bookkeeping per element -- the 2-byte kernels are instruction-issue bound, not HBM bound.
// One tile per CTA: sm_bar is initialised once and used for a single phase.
template <typename T, int CHMODE, int CODE, int UNROLL, int V>
__device__ __forceinline__ void lutp_tile(const LutPArgs& a, const int64_t tile_index) {
    constexpr int WORDS_IN = V * sizeof(T) / 4;
    constexpr uint32_t TILE = kThreads * UNROLL * V;
    static_assert(V == 4 || (V == 8 && sizeof(T) == 2 && CHMODE != CH_ELEM), "vector width");
    extern __shared__ __align__(16) float sm_dyn[];                   // [records W * rec_floats][cq P (+pad)][cells NC + 1 (+pad)][orig P]
    __shared__ Window sm_win;
    __shared__ __align__(8) uint64_t sm_bar;

    const uint32_t tid = threadIdx.x;
    const int64_t t0 = tile_index * TILE;
    const int64_t remaining = a.n - t0;
    const bool full = remaining >= (int64_t)TILE;
    const T* xt = reinterpret_cast<const T*>(a.x) + t0;
    // Stage the decision tables with the bulk-copy engine (1-D TMA): the blob already holds them in the layout the
    // CTA wants -- [cells | orig] contiguous and channel records back to back -- so one elected thread arms the
    // mbarrier and issues at most three cp.async.bulk copies (cells + orig, records c0 .. C-1, wrapped records 0 ..);
    // they complete while every thread's streaming loads of the data tile are in flight.  When the host knows that the
    // blob is not being written (tab_early) this happens BEFORE the dependent-launch wait: a CTA that was scheduled
    // into the predecessor's tail has its tables in shared memory by the time the wait returns.
    const uint32_t Wn = CHMODE == CH_PT ? 1u : a.W;
    float* sm_rec = sm_dyn;
    float* sm_front = sm_dyn + (size_t)Wn * a.rec_floats;             // consts | cq | orig | cells
    auto stage = [&]() {
        if (tid != 0) return;
        const uint32_t tab_bytes = (uint32_t)__ldg(&reinterpret_cast<const LutPrepHeader*>(a.blob)->front_bytes);   // bytes of FRONT in use
        mbar_init(&sm_bar, 1);
        uint32_t c0 = 0;
        if (CHMODE != CH_PT) {
            const int64_t g0 = a.elem_offset + t0;
            const int64_t r0 = g0 / a.inner;
            const int64_t off = g0 - r0 * a.inner;
            Window wv;
            wv.off0 = a.bigrow ? 0u : (uint32_t)off;
            const int64_t sp = a.inner - off;
            wv.split = (uint32_t)(sp > (int64_t)TILE ? (int64_t)TILE + 1 : sp);
            sm_win = wv;
            c0 = (uint32_t)(r0 % a.C);
        }
        const uint32_t rec_bytes = (uint32_t)a.rec_floats * 4u;
        const uint32_t n1 = min(Wn, (uint32_t)a.C - c0);            // records before the channel index wraps
        mbar_arrive_expect_tx(&sm_bar, tab_bytes + Wn * rec_bytes);
        bulk_g2s(sm_front, a.blob + a.off_front, tab_bytes, &sm_bar);
        bulk_g2s(sm_rec, a.blob + a.off_rec + (size_t)c0 * rec_bytes, n1 * rec_bytes, &sm_bar);
        if (n1 < Wn) bulk_g2s(reinterpret_cast<char*>(sm_rec) + (size_t)n1 * rec_bytes, a.blob + a.off_rec, (Wn - n1) * rec_bytes, &sm_bar);
    };
    // staging always precedes the tile loads (few registers are live here); what moves is the wait.  The host only picks
    // an order other than "late" together with tab_early.
    if (!a.tab_early) pdl_enter(0);
    stage();
    if (a.tab_early) pdl_enter(a.early);

    uint32_t w[UNROLL][WORDS_IN];
    if (full) {
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) ld_words<WORDS_IN>(xt + (size_t)(j * kThreads + tid) * V, w[j]);
    } else {
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) {
            int64_t l = (int64_t)(j * kThreads + tid) * V;
            if (l + V <= remaining) ld_words<WORDS_IN>(xt + l, w[j]);
            else {
                T tmp[V];
#pragma unroll
                for (int e = 0; e < V; ++e) tmp[e] = (l + e < remaining) ? xt[l + e] : from_f32<T>(0.0f);
                memcpy(w[j], tmp, sizeof(tmp));
            }
        }
    }

    pdl_loaded(a.early);                                                  // the tile is in flight; nothing is written before this point
    __syncthreads();                                                  // barrier init + window visible to everyone
    Window win;
    if (CHMODE != CH_PT) win = sm_win;
    mbar_wait(&sm_bar, 0);

    // Everything below addresses shared memory through 32-bit shared-window addresses: the element loop is
    //   u = sat(x * s' + 0.5); cell = low bits of fma(u, NC, 1.5 * 2^23); b = cells[cell]          (candidate threshold)
    //   px = rec + 4 b; X = [px]; pos = b + (x > X); y = cq[pos] * thr_c                           (record = X[P] | s' | thr_c ...)
    const uint32_t front_s = smem_u32(sm_front);
    const float NCf = lds_f32(front_s);                               // cells in use and the additive constant of the cell index
    const float c0f = lds_f32(front_s + 4u);
    const uint32_t rec_bytes = (uint32_t)a.rec_floats * 4u;
    const uint32_t xbytes = (uint32_t)a.P * 4u;                       // s' sits right behind the P thresholds, thr_c behind it
    const uint32_t rec_base = smem_u32(sm_rec);
    const uint32_t cq_s = front_s + a.rel_cq;
    const uint32_t cells_s = front_s + a.rel_cells;
    const uint32_t orig_s = front_s + a.rel_orig;
    float* yt = a.y + t0;
    // Index emission: when the centroid list is already sorted and free of duplicates the sorted position IS the LUT index
    // (flag in the blob header) and the look-up of the original index disappears from the element loop.
    auto run = [&](auto ident_tag) {
        constexpr bool IDENT = decltype(ident_tag)::value;
    #pragma unroll
        for (int j = 0; j < UNROLL; ++j) {
            const uint32_t l = (uint32_t)(j * kThreads + tid) * V;
            float f[V];
            int code[V];
            Pack<T, V>::unpack(w[j], f);
            uint32_t slot = 0, rem = 0;
            if (CHMODE != CH_PT) locate(l, win, a, slot, rem);
            uint32_t rec = rec_base + slot * rec_bytes;
            float sp = lds_f32(rec + xbytes);
            float th = lds_f32(rec + xbytes + 4u);
            float nan_probe = f[0] + f[1];                             // NaN iff some element is NaN (or inf - inf)
    #pragma unroll
            for (int e = 2; e < V; e += 2) nan_probe += f[e] + f[e + 1];
            // CH_ELEM: a vector of 4 straddles row boundaries.  Rows of at least 4 elements: at most one boundary, so the
            // record pointer / cell scale of the second row are selected per element; shorter rows advance per element.
            const bool two_rows = CHMODE == CH_ELEM && a.inner >= V;
            uint32_t k = V;                                             // elements of this vector in the first row
            uint32_t rec1 = rec;
            float sp1 = sp, th1 = th;
            if (two_rows) {
                if (a.bigrow) {
                    const bool second = l >= win.split;
                    slot = second ? 1u : 0u;
                    rec = rec_base + slot * rec_bytes;
                    sp = lds_f32(rec + xbytes);
                    th = lds_f32(rec + xbytes + 4u);
                    k = second ? (uint32_t)V : min((uint32_t)V, win.split - l);
                } else {
                    k = a.div_inner.d - rem;
                }
                const uint32_t slot1 = (slot + 1 == a.W) ? 0u : slot + 1;
                rec1 = rec_base + slot1 * rec_bytes;
                sp1 = lds_f32(rec1 + xbytes);
                th1 = lds_f32(rec1 + xbytes + 4u);
            }
    #pragma unroll
            for (int e = 0; e < V; ++e) {
                uint32_t r = rec;
                float s = sp, t = th;
                if (CHMODE == CH_ELEM) {
                    if (two_rows) {
                        const bool first = (uint32_t)e < k;
                        r = first ? rec : rec1;
                        s = first ? sp : sp1;
                        t = first ? th : th1;
                    } else {
                        r = rec_base + slot * rec_bytes;
                        s = lds_f32(r + xbytes);
                        t = lds_f32(r + xbytes + 4u);
                    }
                }
                const float x = f[e];
                const float u = fma_sat(x, s, c0f);                         // saturates to [0, 1]; NaN -> 0
                const float cf = __fmaf_rn(u, NCf, kMagicRound);            // integer cell index in the low mantissa bits
                const uint32_t cell = __float_as_uint(cf) & 0x1fffu;
                const uint32_t b = lds_u8(cells_s + cell);                  // index of the candidate threshold
                const uint32_t b4 = b << 2;
                const float X = lds_f32(r + b4);
                const bool above = x > X;
                f[e] = __fmul_rn(lds_f32(cq_s + b4 + (above ? 4u : 0u)), t);     // 16 consecutive words: never a bank conflict
                if (CODE != 0) code[e] = IDENT ? (int)(b + (above ? 1u : 0u)) : (int)lds_u8(orig_s + b + (above ? 1u : 0u));
                if (CHMODE == CH_ELEM && !two_rows) {
                    if (++rem == a.div_inner.d) { rem = 0; slot = (slot + 1 == a.W) ? 0 : slot + 1; }
                }
            }
            if (nan_probe != nan_probe) {
                // rare: torch.argmin over all-NaN distances returns index 0
                const uint32_t pos0 = (uint32_t)__ldg(&reinterpret_cast<const LutPrepHeader*>(a.blob)->pos0);
                float g[V];
                Pack<T, V>::unpack(w[j], g);
                uint32_t slot2 = 0, rem2 = 0;
                if (CHMODE != CH_PT) locate(l, win, a, slot2, rem2);
                for (int e = 0; e < V; ++e) {
                    if (CHMODE == CH_ELEM && a.bigrow) {
                        uint32_t jrow = (l + e) >= win.split ? 1u : 0u;
                        slot2 = jrow >= a.W ? jrow - a.W : jrow;
                    }
                    if (g[e] != g[e]) {
                        f[e] = __fmul_rn(lds_f32(cq_s + 4u * pos0), lds_f32(rec_base + slot2 * rec_bytes + xbytes + 4u));
                        if (CODE != 0) code[e] = (int)lds_u8(orig_s + pos0);
                    }
                    if (CHMODE == CH_ELEM && !a.bigrow) {
                        if (++rem2 == a.div_inner.d) { rem2 = 0; slot2 = (slot2 + 1 == a.W) ? 0 : slot2 + 1; }
                    }
                }
            }
            if (full || (int64_t)l + V <= remaining) {
                if (a.y) {
                    uint32_t o[V];
                    Pack<float, V>::pack(f, o);
                    if (V == 8) st_stream256(yt + l, o);        // 32 contiguous bytes per lane in one store
                    else st_words<4>(yt + l, o);
                }
                if (CODE != 0) st_codes<V, CODE>(a.idx, t0 + l, code);
            } else if ((int64_t)l < remaining) {
                const int cnt = (int)(remaining - l);
                for (int e = 0; e < V; ++e) {
                    if (e < cnt) {
                        if (a.y) yt[l + e] = f[e];
                        if (CODE == MCTQ_CODES_INT8) reinterpret_cast<uint8_t*>(a.idx)[t0 + l + e] = (uint8_t)code[e];
                    }
                }
                if (CODE == MCTQ_CODES_INT4) {
                    uint8_t* cp = reinterpret_cast<uint8_t*>(a.idx) + ((t0 + l) >> 1);
                    for (int e = 0; e < V; e += 2) {
                        if (e < cnt) {
                            int hi = (e + 1 < cnt) ? code[e + 1] : 0;
                            cp[e >> 1] = (uint8_t)((code[e] & 0xf) | ((hi & 0xf) << 4));
                        }
                    }
                }
            }
        }
    };
    if (CODE != 0 && __ldg(&reinterpret_cast<const LutPrepHeader*>(a.blob)->orig_identity) != 0) run(std::true_type{});
    else run(std::false_type{});
    pdl_exit(a.early);
}

// ---- xy variant: per-tensor thresholds or rows at least one tile long (a tile touches at most two channels), centroid
// lists of <= 16 entries.  Channel records are {X[16] | Y[16] | s'} with Y[k] = cq[k] * thr_c formed at prepare time, so
// the element loop is  u = sat(x * s' + c0);  cell address = bits of fma(u, NCd, base)  [subnormal arithmetic: NCd = NC
// ulps of 2^-149, base = the shared-memory address of cells[] in the same units -- no mask, no add];  b = cells[..];
// X = rec[b];  y = rec[16 + b + (x > X)]  (two predicated loads at immediate offsets 64 / 68) -- 9 issue slots and
// 3 shared-memory reads per element, against 15 + 4 in lutp_tile.  NaN inputs (index 0 of the original list, as
// torch.argmin) are found by a packed probe of the raw words and patched on a cold path.
template <typename T> struct NanProbe;
template <> struct NanProbe<float> {
    template <int WORDS> __device__ static __forceinline__ bool any(const uint32_t* w) {
        float s = __uint_as_float(w[0]);
#pragma unroll
        for (int i = 1; i < WORDS; ++i) s += __uint_as_float(w[i]);
        return s != s;                                                // NaN iff some element is NaN (or inf - inf: re-checked)
    }
};
template <> struct NanProbe<__nv_bfloat16> {
    template <int WORDS> __device__ static __forceinline__ bool any(const uint32_t* w) {
        __nv_bfloat162 s = *reinterpret_cast<const __nv_bfloat162*>(&w[0]);
#pragma unroll
        for (int i = 1; i < WORDS; ++i) s = __hadd2(s, *reinterpret_cast<const __nv_bfloat162*>(&w[i]));
        return __hisnan(s.x) || __hisnan(s.y);
    }
};
template <> struct NanProbe<__half> {
    template <int WORDS> __device__ static __forceinline__ bool any(const uint32_t* w) {
        __half2 s = *reinterpret_cast<const __half2*>(&w[0]);
#pragma unroll
        for (int i = 1; i < WORDS; ++i) s = __hadd2(s, *reinterpret_cast<const __half2*>(&w[i]));
        return __hisnan(s.x) || __hisnan(s.y);
    }
};

// y = (x > X) ? [addr + 68] : [addr + 64] with X = [addr]: one compare, two predicated loads (one executes)
__device__ __forceinline__ float xy_select(float x, uint32_t addr, bool& above) {
    float y;
    uint32_t p;
    asm volatile("{\n\t.reg .pred q;\n\t.reg .f32 t;\n\t"
                 "ld.shared.f32 t, [%2];\n\t"
                 "setp.gt.f32 q, %3, t;\n\t"
                 "@q ld.shared.f32 %0, [%2+68];\n\t"
                 "@!q ld.shared.f32 %0, [%2+64];\n\t"
                 "selp.u32 %1, 1, 0, q;\n\t}"
                 : "=f"(y), "=r"(p) : "r"(addr), "f"(x));
    above = p != 0;
    return y;
}
__device__ __forceinline__ float xy_select(float x, uint32_t addr) {
    float y;
    asm volatile("{\n\t.reg .pred q;\n\t.reg .f32 t;\n\t"
                 "ld.shared.f32 t, [%1];\n\t"
                 "setp.gt.f32 q, %2, t;\n\t"
                 "@q ld.shared.f32 %0, [%1+68];\n\t"
                 "@!q ld.shared.f32 %0, [%1+64];\n\t}"
                 : "=f"(y) : "r"(addr), "f"(x));
    return y;
}

template <typename T, int CHMODE, int CODE, int UNROLL, int V>
__device__ __forceinline__ void lutx_tile(const LutPArgs& a, const int64_t tile_index) {
    constexpr int WORDS_IN = V * sizeof(T) / 4;
    constexpr uint32_t TILE = kThreads * UNROLL * V;
    constexpr uint32_t REC = kXyRecFloats * 4u;
    static_assert(CHMODE == CH_PT || CHMODE == CH_VEC, "xy records: per-tensor or whole-vector channels");
    extern __shared__ __align__(16) float sm_dyn[];                   // [records W * 36 floats][FRONT]
    __shared__ Window sm_win;
    __shared__ __align__(8) uint64_t sm_bar;

    const uint32_t tid = threadIdx.x;
    const int64_t t0 = tile_index * TILE;
    const int64_t remaining = a.n - t0;
    const bool full = remaining >= (int64_t)TILE;
    const T* xt = reinterpret_cast<const T*>(a.x) + t0;
    const uint32_t Wn = CHMODE == CH_PT ? 1u : a.W;                   // channel slots (rows a tile can touch; <= kXyMaxW)
    float* sm_rec = sm_dyn;
    float* sm_front = sm_dyn + Wn * kXyRecFloats;
    auto stage = [&]() {                                              // see lutp_tile: before the dependent-launch wait when legal
        if (tid != 0) return;
        const uint32_t tab_bytes = (uint32_t)__ldg(&reinterpret_cast<const LutPrepHeader*>(a.blob)->front_bytes);
        mbar_init(&sm_bar, 1);
        uint32_t c0 = 0;
        if (CHMODE != CH_PT) {
            const int64_t g0 = a.elem_offset + t0;
            const int64_t r0 = g0 / a.inner;
            const int64_t off = g0 - r0 * a.inner;
            Window wv;
            wv.off0 = a.bigrow ? 0u : (uint32_t)off;
            const int64_t sp = a.inner - off;                         // elements of this tile in its first row
            wv.split = (uint32_t)(sp > (int64_t)TILE ? (int64_t)TILE + 1 : sp);
            sm_win = wv;
            c0 = (uint32_t)(r0 % a.C);
        }
        const uint32_t n1 = min(Wn, (uint32_t)a.C - c0);              // records before the channel index wraps
        mbar_arrive_expect_tx(&sm_bar, tab_bytes + Wn * REC);
        bulk_g2s(sm_front, a.blob + a.off_front, tab_bytes, &sm_bar);
        bulk_g2s(sm_rec, a.blob + a.off_xy + (size_t)c0 * REC, n1 * REC, &sm_bar);
        if (n1 < Wn) bulk_g2s(reinterpret_cast<char*>(sm_rec) + (size_t)n1 * REC, a.blob + a.off_xy, (Wn - n1) * REC, &sm_bar);
    };
    // staging always precedes the tile loads (few registers are live here); what moves is the wait.  The host only picks
    // an order other than "late" together with tab_early.
    if (!a.tab_early) pdl_enter(0);
    stage();
    if (a.tab_early) pdl_enter(a.early);

    uint32_t w[UNROLL][WORDS_IN];
    if (full) {
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) ld_words<WORDS_IN>(xt + (size_t)(j * kThreads + tid) * V, w[j]);
    } else {
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) {
            int64_t l = (int64_t)(j * kThreads + tid) * V;
            if (l + V <= remaining) ld_words<WORDS_IN>(xt + l, w[j]);
            else {
                T tmp[V];
#pragma unroll
                for (int e = 0; e < V; ++e) tmp[e] = (l + e < remaining) ? xt[l + e] : from_f32<T>(0.0f);
                memcpy(w[j], tmp, sizeof(tmp));
            }
        }
    }

    pdl_loaded(a.early);                                                  // the tile is in flight; nothing is written before this point
    __syncthreads();                                                  // barrier init + window visible to everyone
    Window win;
    if (CHMODE != CH_PT) win = sm_win;
    mbar_wait(&sm_bar, 0);

    const uint32_t front_s = smem_u32(sm_front);
    const uint32_t rec_s = smem_u32(sm_rec);
    const float c0f = lds_f32(front_s + 4u);
    const float NCd = lds_f32(front_s + 8u);                          // NC * 2^-149
    const float based = __uint_as_float(front_s + a.rel_cells);       // &cells[0] * 2^-149
    const uint32_t orig_s = front_s + a.rel_orig;
    float* yt = a.y + t0;
    // Index emission packs as it goes: element e adds pos << (4e) (nibbles) or pos << (8 (e & 3)) (bytes) to a 32-bit
    // accumulator -- one shift-add per element, no per-element code registers (a first version kept V codes and masked /
    // shifted / or-ed them at the end: 21 instructions per element and 58-64 registers for bf16).  When the centroid list
    // is sorted and free of duplicates the sorted position IS the LUT index (flag in the blob header).
    auto run = [&](auto ident_tag) {
        constexpr bool IDENT = decltype(ident_tag)::value;
        constexpr int CW = CODE == MCTQ_CODES_INT8 ? V / 4 : 1;
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) {
            const uint32_t l = (uint32_t)(j * kThreads + tid) * V;
            float f[V];
            uint32_t cw[CW];
#pragma unroll
            for (int i = 0; i < CW; ++i) cw[i] = 0;
            Pack<T, V>::unpack(w[j], f);
            uint32_t slot = 0, rem = 0;
            if (CHMODE != CH_PT) locate(l, win, a, slot, rem);
            const uint32_t rec = rec_s + slot * REC;
            const float sp = lds_f32(rec + 2u * kXyP * 4u);
            // staged so that the V independent look-up chains of a vector are in flight together
            uint32_t ca[V], bb[V];
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const float u = fma_sat(f[e], sp, c0f);                           // saturates to [0, 1]; NaN -> 0
                ca[e] = __float_as_uint(__fmaf_rn(u, NCd, based));                // address of this element's cell
            }
#pragma unroll
            for (int e = 0; e < V; ++e) bb[e] = lds_u8(ca[e]);                    // index of the candidate threshold
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const uint32_t ea = rec + (bb[e] << 2);
                if (CODE != 0) {
                    bool above;
                    f[e] = xy_select(f[e], ea, above);
                    uint32_t pos = bb[e] + (above ? 1u : 0u);
                    if (!IDENT) pos = lds_u8(orig_s + pos);
                    if (CODE == MCTQ_CODES_INT4) cw[0] += pos << (4 * e);
                    else cw[e >> 2] += pos << (8 * (e & 3));
                } else {
                    f[e] = xy_select(f[e], ea);
                }
            }
            if (NanProbe<T>::template any<WORDS_IN>(w[j])) {
                // rare: torch.argmin over all-NaN distances returns index 0 of the ORIGINAL centroid list
                const uint32_t pos0 = (uint32_t)__ldg(&reinterpret_cast<const LutPrepHeader*>(a.blob)->pos0);
                float g[V];
                Pack<T, V>::unpack(w[j], g);
                for (int e = 0; e < V; ++e) {
                    if (g[e] != g[e]) {
                        f[e] = lds_f32(rec + (kXyP + pos0) * 4u);
                        if (CODE == MCTQ_CODES_INT4) cw[0] = (cw[0] & ~(0xfu << (4 * e))) | (lds_u8(orig_s + pos0) << (4 * e));
                        if (CODE == MCTQ_CODES_INT8) cw[e >> 2] = (cw[e >> 2] & ~(0xffu << (8 * (e & 3)))) | (lds_u8(orig_s + pos0) << (8 * (e & 3)));
                    }
                }
            }
            if (full || (int64_t)l + V <= remaining) {
                if (a.y) {
                    uint32_t o[V];
                    Pack<float, V>::pack(f, o);
                    if (V == 8) st_stream256(yt + l, o);
                    else st_words<4>(yt + l, o);
                }
                if (CODE == MCTQ_CODES_INT8) {
                    uint8_t* cp = reinterpret_cast<uint8_t*>(a.idx) + t0 + l;
                    if (V == 4) st_stream(reinterpret_cast<uint32_t*>(cp), cw[0]);
                    else st_stream(reinterpret_cast<uint2*>(cp), make_uint2(cw[0], cw[CW - 1]));
                } else if (CODE == MCTQ_CODES_INT4) {
                    uint8_t* cp = reinterpret_cast<uint8_t*>(a.idx) + ((t0 + l) >> 1);
                    if (V == 4) st_stream(reinterpret_cast<uint16_t*>(cp), (uint16_t)cw[0]);
                    else st_stream(reinterpret_cast<uint32_t*>(cp), cw[0]);
                }
            } else if ((int64_t)l < remaining) {
                const int cnt = (int)(remaining - l);
                for (int e = 0; e < V; ++e) {
                    if (e < cnt) {
                        if (a.y) yt[l + e] = f[e];
                        if (CODE == MCTQ_CODES_INT8) reinterpret_cast<uint8_t*>(a.idx)[t0 + l + e] = (uint8_t)(cw[e >> 2] >> (8 * (e & 3)));
                    }
                }
                if (CODE == MCTQ_CODES_INT4) {
                    uint8_t* cp = reinterpret_cast<uint8_t*>(a.idx) + ((t0 + l) >> 1);
                    for (int e = 0; e < V; e += 2) {
                        if (e < cnt) {
                            const uint32_t lo4 = (cw[0] >> (4 * e)) & 0xfu;
                            const uint32_t hi4 = (e + 1 < cnt) ? (cw[0] >> (4 * e + 4)) & 0xfu : 0u;
                            cp[e >> 1] = (uint8_t)(lo4 | (hi4 << 4));
                        }
                    }
                }
            }
        }
    };
    if (CODE != 0 && __ldg(&reinterpret_cast<const LutPrepHeader*>(a.blob)->orig_identity) == 0) run(std::false_type{});
    else run(std::true_type{});
    pdl_exit(a.early);
}

template <typename T, int CHMODE, int CODE, int UNROLL, int V>
__global__ void __launch_bounds__(kThreads) fq_lutx_kernel(const __grid_constant__ LutPArgs a) {
    lutx_tile<T, CHMODE, CODE, UNROLL, V>(a, (int64_t)blockIdx.x);
}

template <typename T, int CHMODE, int CODE, int UNROLL, int V>
__global__ void __launch_bounds__(kThreads) fq_lutp_kernel(const __grid_constant__ LutPArgs a) {
    lutp_tile<T, CHMODE, CODE, UNROLL, V>(a, (int64_t)blockIdx.x);
}

// ---- many tensors, one launch (whole-model LUT weight quantization).  The per-tensor argument blocks and the first tile
// of every tensor travel as KERNEL PARAMETERS (a __grid_constant__ struct): a CTA finds its tensor by a binary search over
// the constant bank and reads that tensor's arguments with register-indexed LDC -- a few tens of cycles, no global loads
// and no barrier before the data loads can be issued (a first version kept the table in global memory: the dependent
// look-ups cost every CTA ~1000 cycles of idle residency and 15-20 % of the bandwidth).  No launch gaps and no per-launch
// tails between the tensors.
// Every launch is SPECIALISED for one kernel variant (dtype, channel mode, vector width, thin / xy records): the host plan
// groups the tensors by variant.  The first version ran every variant out of one kernel (64 registers, 4 CTAs per SM, four
// tiles per CTA to amortise the dispatch) and reached 6.3 TB/s on Llama-7B where the single-tensor kernels run at 6.6-6.7;
// a specialised launch has the single-tensor kernel's registers and one tile per CTA.
struct LutPMultiVariant {
    int32_t dtype, chmode, v, xy, pad[3];
};
// The parameter block is copied by every launch, so its capacity is a template parameter: 16 / 64 tensors (2.5 / 10 KB).
template <int CAP>
using LutPMultiParamsT = PlanChunk<LutPMultiVariant, LutPArgs, CAP>;

// 2-D grid: blockIdx.y = tensor, blockIdx.x = tile of that tensor (CTAs past a tensor's last tile exit at once; the host
// only puts tensors of similar size into one launch).  No search: a first version found the tensor by a binary search
// over prefix sums in the constant bank -- seven dependent LDC round trips in front of every CTA's first load, which cost
// the Llama-7B launch 5 % against the single-tensor kernel.
template <typename T, int CHMODE, int V, bool XY, int CAP>
__global__ void __launch_bounds__(kThreads) fq_lut_multi_kernel(const __grid_constant__ LutPMultiParamsT<CAP> p) {
    const uint32_t k = blockIdx.y;
    if ((int32_t)blockIdx.x >= p.tiles[k]) return;
    const LutPArgs& a = p.e[k];
    if constexpr (XY) lutx_tile<T, CHMODE, MCTQ_CODES_NONE, 4, V>(a, (int64_t)blockIdx.x);
    else lutp_tile<T, CHMODE, MCTQ_CODES_NONE, 4, V>(a, (int64_t)blockIdx.x);
}

}  // namespace mctq

using namespace mctq;

namespace {

// variant selection shared by the single-tensor and the multi-tensor entry points
void lutp_variant(const LutPArgs& a, size_t esz, int idx_mode, int* chmode, int* v) {
    // 8-element vectors for 2-byte inputs: 16-byte aligned x, 32-byte aligned y, 8-byte aligned int8 indices, rows a multiple of 8
    bool v8 = esz == 2 && aligned16(a.x) && (!a.y || aligned32(a.y)) &&
              (idx_mode != MCTQ_CODES_INT8 || (reinterpret_cast<uintptr_t>(a.idx) & 7u) == 0);
    if (a.C == 1) *chmode = CH_PT;
    else if (a.inner % 4 == 0 && a.elem_offset % 4 == 0) {
        *chmode = CH_VEC;
        v8 = v8 && a.inner % 8 == 0 && a.elem_offset % 8 == 0;
    } else {
        *chmode = CH_ELEM;
        v8 = false;
    }
    *v = v8 ? 8 : 4;
}

// channel-window geometry and dynamic shared memory of one tensor for tiles of kThreads * 4 * v elements
int lutp_finish_args(LutPArgs& a, int chmode, int v, size_t* smem_out) {
    const uint32_t tile = kThreads * 4 * (uint32_t)v;
    uint32_t W = 1;
    if (chmode != CH_PT) { set_window(a, tile); W = a.W; }
    const size_t smem = (size_t)W * a.rec_floats * 4 + (size_t)a.front_cap;                // records + FRONT (capacity)
    if (smem > 64 * 1024) return MCTQ_E_RANGE;            // caller falls back to the generic kernel
    *smem_out = smem;
    return 0;
}

// declares the launch's inputs / outputs to the dependent-launch bookkeeping; 1 = the early order may be used
template <typename T, int CODE>
void lut_pdl_order(LutPArgs& a, cudaStream_t st) {
    const IoSpan in[1] = {{a.x, (size_t)a.n * sizeof(T)}};
    const IoSpan out[2] = {{a.y, (size_t)a.n * 4}, {a.idx, CODE == MCTQ_CODES_INT4 ? (size_t)(a.n + 1) / 2 : (size_t)a.n}};
    const IoSpan tables = {a.blob, (size_t)a.off_rec + (size_t)a.C * a.rec_floats * 4 + (a.off_xy ? (size_t)a.C * kXyRecFloats * 4 : 0)};
    a.early = (uint32_t)pdl_plan_launch(st, in, 1, out, CODE != 0 ? 2 : 1, &tables, &a.tab_early);
    if (!a.tab_early) a.early = 0;         // tables after the wait: only the late order has that shape (right after a prepare call)
}

template <typename T, int CHMODE, int CODE, int V>
int launch_lutp_tiles(const LutPArgs& a_in, cudaStream_t st) {
    constexpr int UNROLL = 4;
    constexpr uint32_t TILE = kThreads * UNROLL * V;
    LutPArgs a = a_in;
    size_t smem = 0;
    int rc = lutp_finish_args(a, CHMODE, V, &smem);
    if (rc) return rc;
    rc = ensure_smem(fq_lutp_kernel<T, CHMODE, CODE, UNROLL, V>, smem);
    if (rc) return rc;
    int64_t tiles = (a.n + TILE - 1) / TILE;
    if (tiles > 0x7fffffffLL) return MCTQ_E_BADARG;
    lut_pdl_order<T, CODE>(a, st);
    return launch_planned(fq_lutp_kernel<T, CHMODE, CODE, UNROLL, V>, (unsigned)tiles, smem, st, a);
}

// xy variant eligible: records exist, per-tensor thresholds or whole-vector channels whose tiles touch at most kXyMaxW rows
// (144-byte records: for shorter rows the thin 72-byte records keep the table traffic below the data traffic).
// Call after lutp_finish_args (a.W = rows a tile can touch).
constexpr uint32_t kXyMaxW = 8;
bool lutx_eligible(const LutPArgs& a, int chmode, int v) {
    (void)v;
    if (a.off_xy == 0 || a.P > kXyP) return false;
    if (chmode == CH_PT) return true;
    return chmode == CH_VEC && a.W <= kXyMaxW;
}
size_t lutx_smem(const LutPArgs& a, int chmode) { return (size_t)(chmode == CH_PT ? 1u : a.W) * kXyRecFloats * 4 + a.front_cap; }

// (half-size tiles, UNROLL = 2, were measured on the B200 and are slower: f32 6717 -> 6320 GB/s, bf16 6836 -> 6599, Llama-7B
// per-layer bf16 6110 -> 5839 -- the per-tile staging and barrier outweigh the finer tail)
template <typename T, int CHMODE, int CODE, int V>
int launch_lutx_tiles(const LutPArgs& a_in, cudaStream_t st) {
    constexpr int UNROLL = 4;
    constexpr uint32_t TILE = kThreads * UNROLL * V;
    LutPArgs a = a_in;
    const size_t smem = lutx_smem(a, CHMODE);
    int rc = ensure_smem(fq_lutx_kernel<T, CHMODE, CODE, UNROLL, V>, smem);
    if (rc) return rc;
    int64_t tiles = (a.n + TILE - 1) / TILE;
    if (tiles > 0x7fffffffLL) return MCTQ_E_BADARG;
    lut_pdl_order<T, CODE>(a, st);
    return launch_planned(fq_lutx_kernel<T, CHMODE, CODE, UNROLL, V>, (unsigned)tiles, smem, st, a);
}

template <typename T, int CHMODE, int V>
int launch_lutx_code(const LutPArgs& a, int idx_mode, cudaStream_t st) {
    switch (idx_mode) {
        case MCTQ_CODES_INT8: return launch_lutx_tiles<T, CHMODE, MCTQ_CODES_INT8, V>(a, st);
        case MCTQ_CODES_INT4: return launch_lutx_tiles<T, CHMODE, MCTQ_CODES_INT4, V>(a, st);
        default: return launch_lutx_tiles<T, CHMODE, MCTQ_CODES_NONE, V>(a, st);
    }
}

template <typename T, int CHMODE, int V>
int launch_lutp_code(const LutPArgs& a, int idx_mode, cudaStream_t st) {
    switch (idx_mode) {
        case MCTQ_CODES_INT8: return launch_lutp_tiles<T, CHMODE, MCTQ_CODES_INT8, V>(a, st);
        case MCTQ_CODES_INT4: return launch_lutp_tiles<T, CHMODE, MCTQ_CODES_INT4, V>(a, st);
        default: return launch_lutp_tiles<T, CHMODE, MCTQ_CODES_NONE, V>(a, st);
    }
}

template <typename T>
int launch_lutp_typed(const LutPArgs& a, int idx_mode, cudaStream_t st) {
    constexpr int V8 = sizeof(T) == 2 ? 8 : 4;
    int chmode, v;
    lutp_variant(a, sizeof(T), idx_mode, &chmode, &v);
    LutPArgs ax = a;
    size_t smem_thin = 0;
    if (lutp_finish_args(ax, chmode, v, &smem_thin) == 0 && lutx_eligible(ax, chmode, v)) {
        if (chmode == CH_PT) return v == 8 ? launch_lutx_code<T, CH_PT, V8>(ax, idx_mode, st) : launch_lutx_code<T, CH_PT, 4>(ax, idx_mode, st);
        return v == 8 ? launch_lutx_code<T, CH_VEC, V8>(ax, idx_mode, st) : launch_lutx_code<T, CH_VEC, 4>(ax, idx_mode, st);
    }
    if (chmode == CH_PT) return v == 8 ? launch_lutp_code<T, CH_PT, V8>(a, idx_mode, st) : launch_lutp_code<T, CH_PT, 4>(a, idx_mode, st);
    if (chmode == CH_VEC) return v == 8 ? launch_lutp_code<T, CH_VEC, V8>(a, idx_mode, st) : launch_lutp_code<T, CH_VEC, 4>(a, idx_mode, st);
    return launch_lutp_code<T, CH_ELEM, 4>(a, idx_mode, st);
}

// argument block of one prepared-LUT tensor (validated); shared by mctq_fq_lut_prepared and the multi-tensor plan
int lutp_make_args(const void* x, float* y, void* idx, int64_t n, int x_dtype, const void* prepared_dev, int K, int bw, int is_signed,
                   int64_t C, int64_t inner, int64_t elem_offset, int idx_mode, LutPArgs* out) {
    if (!x || !prepared_dev || n < 0 || C < 1 || inner < 1 || elem_offset < 0 || (!y && idx_mode == MCTQ_CODES_NONE)) return MCTQ_E_BADARG;
    if (idx_mode != MCTQ_CODES_NONE && !idx) return MCTQ_E_BADARG;
    if (x_dtype < 0 || x_dtype > 2) return MCTQ_E_DTYPE;
    PrepGeom g;
    int rc = prep_geometry(K, bw, is_signed, C, &g);
    if (rc) return rc;
    if (idx_mode == MCTQ_CODES_INT4 && g.P > 16) return MCTQ_E_RANGE;
    const size_t esz = x_dtype == MCTQ_F32 ? 4 : 2;
    bool vec_ok = (reinterpret_cast<uintptr_t>(x) % (4 * esz)) == 0 && (!y || aligned16(y));
    if (idx_mode != MCTQ_CODES_NONE) vec_ok = vec_ok && (reinterpret_cast<uintptr_t>(idx) & 3u) == 0;
    if (!aligned16(prepared_dev)) vec_ok = false;  // the tables are staged with 16-byte bulk copies
    if (!vec_ok) return MCTQ_E_BADARG;             // caller uses the generic entry point for misaligned views
    LutPArgs a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.y = y; a.idx = idx; a.n = n; a.blob = reinterpret_cast<const uint8_t*>(prepared_dev);
    a.P = g.P; a.NC = g.NC; a.rec_floats = g.rec_floats;
    a.off_front = (int32_t)g.off_front; a.off_rec = (int32_t)g.off_rec; a.off_xy = (int32_t)g.off_xy;
    a.rel_cq = g.rel_cq; a.rel_orig = g.rel_orig; a.rel_cells = g.rel_cells; a.front_cap = g.front_cap;
    a.C = C; a.inner = C == 1 ? 1 : inner; a.elem_offset = C == 1 ? 0 : elem_offset;
    *out = a;
    return 0;
}

}  // namespace

extern "C" {

size_t mctq_lut_prepared_bytes(int K, int lut_values_bitwidth, int is_signed, int64_t C) {
    PrepGeom g;
    if (prep_geometry(K, lut_values_bitwidth, is_signed, C, &g)) return 0;
    return g.bytes;
}

int mctq_lut_prepare(const void* table_host, int K, const float* thr_dev, int64_t C, float eps, int scalar_mode,
                     float divisor, float thr_f32, int round_dtype, void* prepared_dev, size_t prepared_bytes, void* stream) {
    MCTQ_NVTX("mctq_lut_prepare");
    if (!table_host || !prepared_dev || C < 1 || (!scalar_mode && !thr_dev) || round_dtype < 0 || round_dtype > 2 || scalar_mode < 0 || scalar_mode > 2) return MCTQ_E_BADARG;
    if (scalar_mode && C != 1) return MCTQ_E_BADARG;
    const LutTableHeader* th = reinterpret_cast<const LutTableHeader*>(table_host);
    if (th->magic != kLutMagic || th->K != K) return MCTQ_E_LUT;
    PrepGeom g;
    int rc = prep_geometry(K, th->bw, th->is_signed, C, &g);
    if (rc) return rc;
    if (prepared_bytes < g.bytes) return MCTQ_E_BADARG;
    const int P = g.P;
    const float* tau = reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(table_host) + sizeof(LutTableHeader));
    const float* cq = tau + (P - 1);
    const uint8_t* orig = reinterpret_cast<const uint8_t*>(cq + P);
    // channel-independent front of the blob, assembled on the host
    std::vector<uint8_t> front(g.off_rec, 0);
    LutPrepHeader* h = reinterpret_cast<LutPrepHeader*>(front.data());
    h->magic = kPrepMagic; h->K = K; h->P = P; h->C = C; h->mult = th->mult; h->round_dtype = round_dtype;
    h->pos0 = th->pos_of_idx0; h->rec_floats = g.rec_floats;
    h->orig_identity = 1;
    for (int i = 0; i < th->Ks; ++i) if (orig[i] != i) h->orig_identity = 0;
    h->off_tau = (int32_t)g.off_tau; h->off_front = (int32_t)g.off_front; h->off_rec = (int32_t)g.off_rec; h->off_xy = (int32_t)g.off_xy;
    float* ftau = reinterpret_cast<float*>(front.data() + g.off_tau);
    float* fcq = reinterpret_cast<float*>(front.data() + g.off_front + g.rel_cq);
    for (int j = 0; j < P; ++j) { ftau[j] = j < P - 1 ? tau[j] : INFINITY; fcq[j] = cq[j]; }
    memcpy(front.data() + g.off_front + g.rel_orig, orig, P);
    // effective thresholds in the unrounded q domain (rounding to bf16 / f16 moves them to the rounding boundary)
    std::vector<double> E(P - 1 > 0 ? P - 1 : 0);
    for (int j = 0; j < P - 1; ++j) {
        float tj = tau[j];
        double e;
        if (tj == INFINITY) e = INFINITY;
        else if (tj == -INFINITY) e = -INFINITY;
        else if (round_dtype == 0) e = tj;
        else {
            // largest f32 q with round_like(q) <= tau_j
            int64_t lo = f2ord(-3.0e38f), hi = f2ord(3.0e38f);
            if (round_like(ord2f((int32_t)lo), round_dtype) > tj) e = -INFINITY;
            else if (!(round_like(ord2f((int32_t)hi), round_dtype) > tj)) e = INFINITY;
            else {
                while (hi - lo > 1) {
                    int64_t mid = lo + (hi - lo) / 2;
                    if (round_like(ord2f((int32_t)mid), round_dtype) > tj) hi = mid; else lo = mid;
                }
                e = ord2f((int32_t)lo);
            }
        }
        E[j] = e;
    }
    // Cell geometry: the coarsest of {1, 2, 4} cells per step of the normalised grid for which every cell -- widened by
    // the slop of the approximate index -- holds at most ONE threshold (then the candidate + one exact compare decide).
    // Integer centroids put their thresholds on the half-integer grid at least one step apart, so one cell per step,
    // shifted by a quarter cell so that neither integers nor half-integers sit on a cell boundary, is enough: 264 cells
    // for 8-bit grids instead of 2048 -- the byte-wide cell look-up then touches < 32 words for typical data and is all
    // but free of bank conflicts (ncu: 53-77 conflicts per 1000 elements with 2048 cells).
    // Grids of more than 10 bits (round 2): the finest geometry that fits is COARSER than the integer grid (1 / 2^shift cells
    // per step), so it is no longer valid for every centroid list -- lists whose thresholds are closer than a cell are
    // refused (MCTQ_E_RANGE: the caller uses the generic kernel); k-means centroid lists on 12- or 16-bit grids are sparse
    // and pass.  Candidates run from 16 x coarser than the finest to the finest.
    const int sh0 = finest_shift((int64_t)th->mult);
    struct Cand { int cpu, shift; };
    std::vector<Cand> cands;
    if (sh0 == 0) cands = {{1, 0}, {2, 0}, {kCellsPerUnitMax, 0}};
    else for (int k = 4; k >= 0; --k) cands.push_back({kCellsPerUnitMax, sh0 + k});
    int cpu = kCellsPerUnitMax, shift = 0, NC = g.NC;
    double off = 0.0;
    bool found = false;
    std::vector<double> V(E.size());
    for (const Cand& cand : cands) {
        const bool finest = cand.cpu == kCellsPerUnitMax && cand.shift == sh0;
        const int nc = (int)cells_needed(cand.cpu, (int64_t)th->mult, cand.shift);
        if (nc < 40 && !finest) continue;
        const double per_unit = std::ldexp((double)cand.cpu, -cand.shift);
        const double o = (finest && sh0 == 0) ? 0.0 : 0.25;
        bool ok = true;
        for (size_t j = 0; j < E.size(); ++j) V[j] = E[j] * per_unit * (double)th->mult + 0.5 * nc + o;
        for (size_t j = 0; ok && j + 1 < E.size(); ++j) {
            if (!std::isfinite(V[j]) || !std::isfinite(V[j + 1])) continue;
            // two thresholds share a widened cell iff some integer k has k - 0.5 - slop <= V[j] and V[j + 1] <= k + 0.5 + slop
            const double k_lo = std::ceil(V[j + 1] - 0.5 - kCellSlop), k_hi = std::floor(V[j] + 0.5 + kCellSlop);
            if (k_lo <= k_hi) ok = false;
        }
        // (4 cells per step of the integer grid are always valid: thresholds of integer centroids are >= half a step apart)
        if (ok || (finest && sh0 == 0)) { cpu = cand.cpu; shift = cand.shift; NC = nc; off = o; found = true; break; }
    }
    if (!found) return MCTQ_E_RANGE;
    h->NC = NC;
    h->cells_per_unit = cpu;
    h->cells_shift = shift;
    h->cell_offset = (float)off;
    h->front_bytes = (int32_t)(g.rel_cells + (((uint32_t)NC + 1 + 15) & ~15u));
    float* consts = reinterpret_cast<float*>(front.data() + g.off_front);
    consts[0] = (float)NC;
    consts[1] = (float)(0.5 + off / NC);
    {   // NC as a multiple of the smallest subnormal: fma(u, NCd, base) then IS the shared-memory address of the cell
        const uint32_t bits = (uint32_t)NC;
        memcpy(&consts[2], &bits, 4);
    }
    uint8_t* cells = front.data() + g.off_front + g.rel_cells;
    for (int k = 0; k <= NC; ++k) {
        int b = 0;
        for (int j = 0; j < P - 1; ++j) if (V[j] < (double)k - 0.5 - kCellSlop) ++b;
        cells[k] = (uint8_t)b;
    }
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyAsync(prepared_dev, front.data(), g.off_rec, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return (int)e;
    e = cudaStreamSynchronize(st);                 // `front` is pageable and goes out of scope; this call is one-off setup
    if (e != cudaSuccess) return (int)e;
    int64_t total = C * P;
    int64_t blocks = (total + kThreads - 1) / kThreads;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pdl_note_prepare(st, prepared_dev, g.bytes);                  // launches that follow stage this blob only after their wait
    lut_prepare_kernel<<<(unsigned)blocks, kThreads, 0, st>>>(reinterpret_cast<uint8_t*>(prepared_dev), thr_dev, eps, scalar_mode, divisor, thr_f32);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cuda_rc(cudaGetLastError());
}

int mctq_fq_lut_prepared(const void* x, float* y, void* idx, int64_t n, int x_dtype, const void* prepared_dev, int K,
                         int lut_values_bitwidth, int is_signed, int64_t C, int64_t inner, int64_t elem_offset,
                         int idx_mode, void* stream) {
    MCTQ_NVTX("mctq_fq_lut_prepared");
    LutPArgs a;
    int rc = lutp_make_args(x, y, idx, n, x_dtype, prepared_dev, K, lut_values_bitwidth, is_signed, C, inner, elem_offset, idx_mode, &a);
    if (rc) return rc;
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    switch (x_dtype) {
        case MCTQ_F32: return launch_lutp_typed<float>(a, idx_mode, st);
        case MCTQ_BF16: return launch_lutp_typed<__nv_bfloat16>(a, idx_mode, st);
        default: return launch_lutp_typed<__half>(a, idx_mode, st);
    }
}

}  // extern "C"

namespace {

using LutMultiPlan = Plan<LutPMultiVariant, LutPArgs, 0x4d514c4du>;   // 'MQLM'

template <typename T, int CHMODE, int V, bool XY, int CAP>
int launch_multi_variant(LutPMultiParamsT<CAP>& p, size_t smem, cudaStream_t st) {
    int rc = ensure_smem(fq_lut_multi_kernel<T, CHMODE, V, XY, CAP>, smem);
    if (rc) return rc;
    // ranges "unknown" (late order); the tables of all tensors may be staged before the wait unless a prepare kernel is in flight
    uint32_t te = 0;
    const IoSpan any_blob = {nullptr, 0};
    pdl_plan_launch(st, nullptr, 0, nullptr, 0, &any_blob, &te);
    for (int i = 0; i < p.n_desc; ++i) p.e[i].tab_early = te;
    return launch_planned(fq_lut_multi_kernel<T, CHMODE, V, XY, CAP>, dim3((unsigned)p.tiles[CAP], (unsigned)p.n_desc), smem, st, p);
}

template <typename T, int CAP>
int launch_multi_typed(LutPMultiParamsT<CAP>& c, size_t smem, cudaStream_t st) {
    constexpr int V8 = sizeof(T) == 2 ? 8 : 4;
    const bool wide = c.var.v == 8 && V8 == 8;
    if (c.var.xy) {
        if (c.var.chmode == CH_PT) return wide ? launch_multi_variant<T, CH_PT, V8, true, CAP>(c, smem, st) : launch_multi_variant<T, CH_PT, 4, true, CAP>(c, smem, st);
        return wide ? launch_multi_variant<T, CH_VEC, V8, true, CAP>(c, smem, st) : launch_multi_variant<T, CH_VEC, 4, true, CAP>(c, smem, st);
    }
    if (c.var.chmode == CH_PT) return wide ? launch_multi_variant<T, CH_PT, V8, false, CAP>(c, smem, st) : launch_multi_variant<T, CH_PT, 4, false, CAP>(c, smem, st);
    if (c.var.chmode == CH_VEC) return wide ? launch_multi_variant<T, CH_VEC, V8, false, CAP>(c, smem, st) : launch_multi_variant<T, CH_VEC, 4, false, CAP>(c, smem, st);
    return launch_multi_variant<T, CH_ELEM, 4, false, CAP>(c, smem, st);
}

template <int CAP>
int launch_multi_chunk(LutPMultiParamsT<CAP>& c, size_t smem, cudaStream_t st) {
    if (c.var.dtype == MCTQ_F32) return launch_multi_typed<float, CAP>(c, smem, st);
    if (c.var.dtype == MCTQ_BF16) return launch_multi_typed<__nv_bfloat16, CAP>(c, smem, st);
    return launch_multi_typed<__half, CAP>(c, smem, st);
}

// argument block, variant, tiles and shared memory of one tensor (validated); 0 or MCTQ_E_*
int multi_describe(const MctqLutTensorDesc& d, LutMultiPlan::Item& it) {
    if (d.n < 1 || !d.y) return MCTQ_E_BADARG;         // empty tensors do not belong in a plan
    LutPArgs& a = it.args;
    int rc = lutp_make_args(d.x, d.y, nullptr, d.n, d.dtype, d.prepared_dev, d.K, d.lut_values_bitwidth, d.is_signed, d.C, d.inner,
                            0, MCTQ_CODES_NONE, &a);
    if (rc) return rc;
    int chmode, v;
    lutp_variant(a, d.dtype == MCTQ_F32 ? 4 : 2, MCTQ_CODES_NONE, &chmode, &v);
    rc = lutp_finish_args(a, chmode, v, &it.smem);
    if (rc) return rc;
    const int xy = lutx_eligible(a, chmode, v) ? 1 : 0;
    if (xy) it.smem = lutx_smem(a, chmode);
    it.var = {d.dtype, chmode, v, xy, {}};
    const int64_t per_tile = (int64_t)kThreads * 4 * v;
    it.tiles = (d.n + per_tile - 1) / per_tile;
    return 0;
}

}  // namespace

extern "C" {

size_t mctq_lut_multi_plan_bytes(const MctqLutTensorDesc* descs, int n_desc) {
    LutMultiPlan plan;
    return plan.compile(descs, n_desc, multi_describe) ? 0 : plan.bytes();
}

int64_t mctq_lut_multi_plan(const MctqLutTensorDesc* descs, int n_desc, void* plan_host_out, size_t plan_bytes) {
    LutMultiPlan plan;
    if (const int rc = plan.compile(descs, n_desc, multi_describe)) return rc;
    plan.h.tiles_per_cta = 1;
    return plan.write(plan_host_out, plan_bytes);
}

int mctq_fq_lut_prepared_multi(const void* plan_host, void* stream) {
    MCTQ_NVTX("mctq_fq_lut_prepared_multi");
    return LutMultiPlan::run<16>(plan_host, 1, [&](auto& p, const PlanHeader& h) {
        return launch_multi_chunk(p, (size_t)h.smem_bytes, (cudaStream_t)stream);
    });
}

}  // extern "C"
