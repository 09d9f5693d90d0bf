// mctq_packed_igemm.cu -- integer linear mode: y = T(((acc - corrections) * f) + b) with acc = sum_k qx[n,k] * qw[o,k] an
// exact int32 product of 8-bit activation codes and packed int8 / int4 weight codes on the tensor cores
// (tcgen05 MMA kind::i8, s32 accumulator in tensor memory).  Packed nn.Linear wrappers in integer mode
// (pytorch/packed_weights.py) call it after mctq_quantize_rows_i8 has turned their input into codes.
//
// The tensor-core frame (TMEM, MMA issue and commit, split-K tile and reduction, launches over row ranges) is that of
// mctq_tcgen05.cuh, shared with mctq_packed_gemm.cu.  Shape: output features are the MMA's M (128 per CTA), batch rows its N (nt, a multiple of 16 up
// to 256; more rows run as further CTAs along grid.y).  A CTA walks its share of the row length in chunks of 128 codes (one
// 128-byte swizzle row) through a ring of `stages` shared-memory stages with a full and an empty mbarrier each:
//   warps 0-3  producers: thread 0 arms the stage's full barrier and copies the x codes (and int8 weight codes) with 2-D TMA
//              (SWIZZLE_128B, zero fill outside the tensor: tail rows and columns are zero codes); for int4 weights the 128
//              producer threads each load one weight row's nibbles and expand them to bytes into the stage (sign extension
//              for signed codes) and arrive on the full barrier
//   warp 4     lane 0 issues the stage's four MMAs (K = 32 each) and commits them onto the stage's empty barrier
//   all warps  the epilogue: tcgen05.ld, one output feature per thread, corrections and scaling in the fixed formula
//              c = acc - zw[o] * Sx[n] - zx * Sw[o] + K * zx * zw[o]  (int64),   y = T(fl(fl((float)c * f[o]) + b[o]))
// There is no CTA-wide barrier in the main loop.  Split-K: the S CTAs of a cluster take consecutive chunk ranges and rank 0
// adds the int32 partial sums of the others (distributed shared memory); integer sums are exact, so the result does not
// depend on S or on the tiling.
//
// Integer convolution mode (packed_iconv_kernel, mctq_packed_conv2d_i8) is the same GEMM with batch rows = output pixels
// (b, ho, wo) and row length K = (r, s, c) taps of the window.  Only the source of the x operand differs: warps 0-3 gather
// it from NHWC codes.  Each producer thread owns rows tid and tid + 128 of the CTA and decomposes their window origins
// once; Cin % 16 == 0, so each 16-byte granule of a stage row is 16 channels of one input pixel, copied with a 16-byte
// cp.async (a tap outside the image is a splat of zx, rows >= M and columns >= K are zero).  The copies of kIConvAhead
// stages stay in flight (cp.async groups); a stage's full barrier gets the producers' arrivals once its group has landed.
// The epilogue writes row-major [M][Cout] (NHWC) or NCHW planes.
//
// Padded codes (mctq_packed_conv2d_i8_padded, DESIGN §7f): the NHWC codes have a pixel pitch Cp >= Cin whose pad channels
// hold zx.  Cp % 16 == 0 is the gather above with Cin := Cp.  Cp = 4 / 8 (packed_iconv_narrow_kernel) is the narrow gather:
// a 16-byte granule holds 16 / Cp consecutive taps, each one cp.async of Cp bytes (a tap outside the image is a Cp-byte
// store of zx); the row length is kh * kw * Cp rounded up to 16 (32 for 4-bit codes), and taps at or beyond kh * kw form
// a row tail of zero codes that the correction does not count.
#include <cuda.h>               // CUtensorMap and the cuTensorMapEncodeTiled types (the entry point is fetched at run time)

#include <algorithm>

#include "mctq_tcgen05.cuh"

namespace mctq {

constexpr int kIChunk = 128;          // codes of the row length per stage
constexpr int kIMinStages = 4, kIMaxStages = 8;
constexpr int kIMaxSplit = 8;         // portable cluster size
constexpr int kIProducers = 128;      // warps 0-3
constexpr int kIMmaWarp = 4;
constexpr int kIConvAhead = 3;        // stages of gathered x in flight per producer (<= kIMinStages - 1)

struct IgemmArgs {
    CUtensorMap tm_x;                 // x codes [M_total][K], box [nt][128]
    CUtensorMap tm_w;                 // int8 weight codes [N][K], box [128][128] (int4 weights: unused)
    const uint8_t* codes;             // int4 weight codes, two per byte
    const int32_t* w_zp;              // zw[C]
    const int32_t* x_rowsum;          // Sx[M_total], or null when every zw is 0
    const int32_t* w_rowsum;          // Sw[N], or null when zx is 0
    const float* factor;              // f[C]
    const void* bias;                 // [N] of T, or null
    void* y;                          // [M_total] rows of ldy elements
    int64_t ldy;
    int64_t m0;                       // first row of this launch
    int64_t M;                        // rows of this launch
    int32_t N, K;
    int32_t per_channel, x_zp;
    int32_t nt, nchunks, stages;
    uint32_t stage_bytes, tmem_cols, idesc;
    // integer convolution mode only
    const uint8_t* x_nhwc;            // x codes [N][H][W][Cin]
    MctqConv2dGeom g;
    FastDiv div_howo, div_wo, div_cin, div_kw;
    int32_t y_nchw;                   // y as NCHW planes instead of [M][Cout]
    uint32_t zx_splat;                // the byte of zx, four times
    // LUT weights only: the int8 codes of the centroids, lut[i] in byte i % 4 of word i / 4 (by value: no device pointer)
    uint32_t lut[64];
};

// how the weight operand reaches a stage: int8 affine codes by TMA, int4 affine codes or LUT indices through the producers
enum class WFmt { I8, I4, LUT4, LUT8 };
__host__ __device__ constexpr bool producer_written(WFmt f) { return f != WFmt::I8; }
__host__ __device__ constexpr bool is_lut(WFmt f) { return f == WFmt::LUT4 || f == WFmt::LUT8; }
constexpr uint32_t kLut8TableBytes = 256 * 32;   // the table of 8-bit indices, one copy per lane

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" :: "r"(dst), "l"(src) : "memory");
}

// the Cp = 4 / 8 bytes of one tap of the narrow gather, and its splat of zx (or zeros)
template <int N>
__device__ __forceinline__ void cp_async_n(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" :: "r"(dst), "l"(src), "n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void st_shared_n(uint32_t addr, uint32_t v) {
    if constexpr (N == 4) asm volatile("st.shared.b32 [%0], %1;" :: "r"(addr), "r"(v) : "memory");
    else asm volatile("st.shared.v2.b32 [%0], {%1,%2};" :: "r"(addr), "r"(v), "r"(v) : "memory");
}

__device__ __forceinline__ void tma_2d(const CUtensorMap* map, uint32_t dst, int32_t c0, int32_t c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}

// 8 nibbles (element 2j in the low nibble of byte j) -> 8 bytes, sign-extended when SIGNED
template <bool SIGNED>
__device__ __forceinline__ void expand8(uint32_t w, uint32_t& lo, uint32_t& hi) {
    const uint32_t ev = w & 0x0F0F0F0Fu, od = (w >> 4) & 0x0F0F0F0Fu;
    lo = __byte_perm(ev, od, 0x5140);
    hi = __byte_perm(ev, od, 0x7362);
    if (SIGNED) {
        lo |= (lo & 0x08080808u) * 0x1Eu;                                // 0x08 * 0x1E = 0xF0: no carry between bytes
        hi |= (hi & 0x08080808u) * 0x1Eu;
    }
}

// 8 nibbles (element 2j in the low nibble of byte j) -> the 8 bytes lut[nibble] of a 16-entry table in t[0..3]: the low
// three bits of a nibble select among entries 0-7 and 8-15 (two byte permutations), its bit 3 picks one of the two bytes
__device__ __forceinline__ void lut8(uint32_t w, const uint32_t* t, uint32_t& lo, uint32_t& hi) {
    const uint32_t s_lo = w & 0x7777u, s_hi = (w >> 16) & 0x7777u;
    const uint32_t pick_lo = 0x3210u | ((w >> 1) & 0x4444u), pick_hi = 0x3210u | ((w >> 17) & 0x4444u);
    lo = __byte_perm(__byte_perm(t[0], t[1], s_lo), __byte_perm(t[2], t[3], s_lo), pick_lo);
    hi = __byte_perm(__byte_perm(t[0], t[1], s_hi), __byte_perm(t[2], t[3], s_hi), pick_hi);
}

// int4 weight codes of one row, chunk c (128 codes = 64 bytes), or zeros outside the weight
__device__ __forceinline__ void load_w4(const uint8_t* wrow, int64_t o, int64_t N, int64_t K, int c, uint4* v) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {                                        // 32 codes per 16 bytes; K % 32 == 0
        const int64_t k = (int64_t)c * kIChunk + 32 * j;
        v[j] = (o < N && k < K) ? ld_stream(reinterpret_cast<const uint4*>(wrow + (k >> 1))) : make_uint4(0, 0, 0, 0);
    }
}
// row `row` of the weight operand of a stage: the 128 codes of v expanded to bytes (LUT: the table codes t[] of the indices)
template <bool WSIGNED, bool LUT = false>
__device__ __forceinline__ void store_w4(uint32_t st, uint32_t row, const uint4* v, const uint32_t* t = nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t words[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
        uint32_t g[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if constexpr (LUT) lut8(words[q], t, g[2 * q], g[2 * q + 1]);
            else expand8<WSIGNED>(words[q], g[2 * q], g[2 * q + 1]);
        }
        st_shared_v4(st + sw128_off(row, 2 * j), g);
        st_shared_v4(st + sw128_off(row, 2 * j + 1), g + 4);
    }
}

// 8-bit LUT indices of one row, chunk c (128 indices), or zeros outside the weight
__device__ __forceinline__ void load_w8(const uint8_t* wrow, int64_t o, int64_t N, int64_t K, int c, uint4* v) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {                                        // 16 indices per 16 bytes; K % 16 == 0
        const int64_t k = (int64_t)c * kIChunk + 16 * j;
        v[j] = (o < N && k < K) ? ld_stream(reinterpret_cast<const uint4*>(wrow + k)) : make_uint4(0, 0, 0, 0);
    }
}
// row `row` of the weight operand of a stage: the table codes of the 128 indices of v.  `tab` is this lane's column of the
// replicated table: entry e at byte (e / 4) * 128 + e % 4, so that the 32 lanes of a warp read 32 different banks
__device__ __forceinline__ void store_w8(uint32_t st, uint32_t row, const uint4* v, const uint8_t* tab) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint32_t words[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
        uint32_t g[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint32_t e = (words[q] >> (8 * i)) & 0xFFu;
                b[i] = tab[((e & 0xFCu) << 5) | (e & 3u)];
            }
            g[q] = __byte_perm(__byte_perm(b[0], b[1], 0x0040u), __byte_perm(b[2], b[3], 0x0040u), 0x5410u);
        }
        st_shared_v4(st + sw128_off(row, (uint32_t)j), g);
    }
}

// the weight operand's row `row` of chunk c, by format: load_w into registers (one chunk ahead), store_w into a stage.  t: the
// 16-entry table in four registers (LUT4); tab: this lane's column of the shared-memory table (LUT8)
template <WFmt F>
__device__ __forceinline__ void load_w(const uint8_t* wrow, int64_t o, int64_t N, int64_t K, int c, uint4* v) {
    if constexpr (F == WFmt::LUT8) load_w8(wrow, o, N, K, c, v);
    else load_w4(wrow, o, N, K, c, v);
}
template <WFmt F, bool WSIGNED>
__device__ __forceinline__ void store_w(uint32_t st, uint32_t row, const uint4* v, const uint32_t* t, const uint8_t* tab) {
    if constexpr (F == WFmt::LUT8) store_w8(st, row, v, tab);
    else if constexpr (F == WFmt::LUT4) store_w4<false, true>(st, row, v, t);
    else store_w4<WSIGNED>(st, row, v);
}

template <WFmt F, bool WSIGNED, typename T, bool CONV, int CP = 0>
__device__ __forceinline__ void igemm_body(const IgemmArgs& a) {
    constexpr bool INT4 = producer_written(F);     // the producers write the weight operand (int4 codes, LUT indices)
    extern __shared__ __align__(1024) uint8_t dsm[];
    __shared__ uint64_t bar_full[kIMaxStages], bar_empty[kIMaxStages];
    __shared__ uint64_t bar_done;
    __shared__ uint32_t tmem_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nt = a.nt, nst = a.stages;
    const uint32_t a_bytes = kTcRows * 128, stage_bytes = a.stage_bytes;
    const uint32_t sbase = (smem_u32(dsm) + 1023u) & ~1023u;             // swizzle atoms need 1024-byte alignment

    pdl_wait();                 // x codes may be the output of the previous launch; TMEM is taken only after the wait
    pdl_launch_dependents();
    tmem_alloc(warp, &tmem_slot, a.tmem_cols);
    if (tid == 0) {
        for (int s = 0; s < nst; ++s) {
            mbar_init(&bar_full[s], CONV ? (INT4 ? 0 : 1) + kIProducers : INT4 ? 1 + kIProducers : 1);
            mbar_init(&bar_empty[s], 1);
        }
        mbar_init(&bar_done, 1);
    }
    if constexpr (F == WFmt::LUT8) {                 // behind the ring: 32 copies of the table, word e / 4 of copy l at 32 e / 4 + l
        uint32_t* tab = reinterpret_cast<uint32_t*>(dsm + (sbase - smem_u32(dsm)) + (uint32_t)nst * stage_bytes);
        for (int i = tid; i < (int)(kLut8TableBytes / 4); i += kThreads) tab[i] = a.lut[i >> 5];
    }
    const uint32_t tmem = tmem_address(&tmem_slot);

    const int64_t N = a.N, K = a.K;
    const TcTile tile = tc_tile(a, nt);
    const int64_t o0 = tile.o0, n0 = tile.n0, rows = tile.rows;           // n0: first row of this CTA inside the launch
    const int c_begin = tile.c_begin, nloc = tile.c_end - tile.c_begin;

    constexpr int NV = F == WFmt::LUT8 ? 8 : 4;     // 16-byte words of weight codes per row and chunk
    uint32_t t[4];
    if constexpr (F == WFmt::LUT4) {
#pragma unroll
        for (int i = 0; i < 4; ++i) t[i] = a.lut[i];
    }
    const uint8_t* tab = dsm + (sbase - smem_u32(dsm)) + (uint32_t)nst * stage_bytes + 4 * lane;
    if (warp < 4) {
        // ---- producers
        if (CONV) {
            const MctqConv2dGeom& g = a.g;
            const int64_t o = o0 + tid;
            const uint8_t* wrow = a.codes + o * (F == WFmt::LUT8 ? K : K >> 1);
            uint4 cur[NV], nxt[NV];
            if (INT4 && nloc > 0) load_w<F>(wrow, o, N, K, c_begin, cur);
            // the window origins of this thread's rows tid and tid + 128; `have_row`: the row is in the stage (r < nt),
            // `live`: it is an output pixel (r < rows)
            bool have_row[2], live[2];
            int32_t ih0[2], iw0[2];
            const uint8_t* img[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int r = tid + kIProducers * q;
                have_row[q] = r < nt;
                live[q] = r < rows;
                const uint32_t pix = live[q] ? (uint32_t)(a.m0 + n0 + r) : 0u;             // M < 2^31
                const uint32_t b = fdiv_u32(pix, a.div_howo), rem = pix - b * (uint32_t)(g.Ho * g.Wo);
                const uint32_t ho = fdiv_u32(rem, a.div_wo), wo = rem - ho * (uint32_t)g.Wo;
                ih0[q] = (int32_t)ho * g.sh - g.pt;
                iw0[q] = (int32_t)wo * g.sw - g.pl;
                img[q] = a.x_nhwc + (int64_t)b * g.H * g.W * g.Cin;
            }
            const uint32_t zero[4] = {0u, 0u, 0u, 0u}, pad[4] = {a.zx_splat, a.zx_splat, a.zx_splat, a.zx_splat};
            for (int i = 0; i < nloc; ++i) {
                const int c = c_begin + i, s = i % nst;
                const uint32_t st = sbase + (uint32_t)s * stage_bytes;
                if (INT4 && i + 1 < nloc) load_w<F>(wrow, o, N, K, c + 1, nxt);
                if (i >= nst) mbar_wait(&bar_empty[s], (uint32_t)((i / nst - 1) & 1));
                if (!INT4 && tid == 0) {
                    mbar_arrive_expect_tx(&bar_full[s], a_bytes);
                    tma_2d(&a.tm_w, st, c * kIChunk, (int32_t)o0, &bar_full[s]);
                }
                if (INT4) store_w<F, WSIGNED>(st, (uint32_t)tid, cur, t, tab);
#pragma unroll
                for (int j = 0; j < kIChunk / 16; ++j) {
                    const int32_t k = c * kIChunk + 16 * j;
                    if constexpr (CP != 0) {                 // narrow gather: taps k / CP .. k / CP + 16 / CP - 1
#pragma unroll
                        for (int u = 0; u < 16 / CP; ++u) {
                            const uint32_t tap = (uint32_t)(k / CP + u);
                            const bool in_k = tap < (uint32_t)(g.kh * g.kw);
                            const uint32_t rr = fdiv_u32(tap, a.div_kw), ss = tap - rr * (uint32_t)g.kw;
                            const int32_t dy = (int32_t)rr * g.dh, dx = (int32_t)ss * g.dw;
#pragma unroll
                            for (int q = 0; q < 2; ++q) {
                                if (!have_row[q]) continue;
                                const uint32_t dst =
                                    st + a_bytes + sw128_off((uint32_t)(tid + kIProducers * q), (uint32_t)j) + CP * u;
                                const int32_t ih = ih0[q] + dy, iw = iw0[q] + dx;
                                if (live[q] && in_k && ih >= 0 && ih < g.H && iw >= 0 && iw < g.W)
                                    cp_async_n<CP>(dst, img[q] + ((int64_t)ih * g.W + iw) * CP);
                                else
                                    st_shared_n<CP>(dst, live[q] && in_k ? a.zx_splat : 0u);
                            }
                        }
                        continue;
                    }
                    const bool in_k = k < K;
                    const uint32_t tap = fdiv_u32((uint32_t)k, a.div_cin), ch = (uint32_t)k - tap * (uint32_t)g.Cin;
                    const uint32_t rr = fdiv_u32(tap, a.div_kw), ss = tap - rr * (uint32_t)g.kw;
                    const int32_t dy = (int32_t)rr * g.dh, dx = (int32_t)ss * g.dw;
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        if (!have_row[q]) continue;
                        const uint32_t dst = st + a_bytes + sw128_off((uint32_t)(tid + kIProducers * q), (uint32_t)j);
                        const int32_t ih = ih0[q] + dy, iw = iw0[q] + dx;
                        if (live[q] && in_k && ih >= 0 && ih < g.H && iw >= 0 && iw < g.W)
                            cp_async16(dst, img[q] + ((int64_t)ih * g.W + iw) * g.Cin + ch);
                        else
                            st_shared_v4(dst, live[q] && in_k ? pad : zero);
                    }
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                if (i >= kIConvAhead) {                                  // stage i - kIConvAhead has landed: publish it
                    asm volatile("cp.async.wait_group %0;" :: "n"(kIConvAhead) : "memory");
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    mbar_arrive(&bar_full[(i - kIConvAhead) % nst]);
                }
                if (INT4) {
#pragma unroll
                    for (int j = 0; j < NV; ++j) cur[j] = nxt[j];
                }
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            for (int i = nloc > kIConvAhead ? nloc - kIConvAhead : 0; i < nloc; ++i) mbar_arrive(&bar_full[i % nst]);
        } else if (INT4) {
            const int64_t o = o0 + tid;
            const uint8_t* wrow = a.codes + o * (F == WFmt::LUT8 ? K : K >> 1);
            uint4 cur[NV], nxt[NV];
            if (nloc > 0) load_w<F>(wrow, o, N, K, c_begin, cur);
            for (int i = 0; i < nloc; ++i) {
                const int c = c_begin + i, s = i % nst;
                const uint32_t st = sbase + (uint32_t)s * stage_bytes;
                if (i + 1 < nloc) load_w<F>(wrow, o, N, K, c + 1, nxt);  // in flight while this stage is filled
                if (i >= nst) mbar_wait(&bar_empty[s], (uint32_t)((i / nst - 1) & 1));
                if (tid == 0) {
                    mbar_arrive_expect_tx(&bar_full[s], (uint32_t)nt * 128u);
                    tma_2d(&a.tm_x, st + a_bytes, c * kIChunk, (int32_t)(a.m0 + n0), &bar_full[s]);
                }
                store_w<F, WSIGNED>(st, (uint32_t)tid, cur, t, tab);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy stores -> tensor-core reads
                mbar_arrive(&bar_full[s]);
#pragma unroll
                for (int j = 0; j < NV; ++j) cur[j] = nxt[j];
            }
        } else if (tid == 0) {
            for (int i = 0; i < nloc; ++i) {
                const int c = c_begin + i, s = i % nst;
                const uint32_t st = sbase + (uint32_t)s * stage_bytes;
                if (i >= nst) mbar_wait(&bar_empty[s], (uint32_t)((i / nst - 1) & 1));
                mbar_arrive_expect_tx(&bar_full[s], a_bytes + (uint32_t)nt * 128u);
                tma_2d(&a.tm_w, st, c * kIChunk, (int32_t)o0, &bar_full[s]);
                tma_2d(&a.tm_x, st + a_bytes, c * kIChunk, (int32_t)(a.m0 + n0), &bar_full[s]);
            }
        }
    } else if (warp == kIMmaWarp && lane == 0) {
        // ---- MMA issuer
        for (int i = 0; i < nloc; ++i) {
            const int s = i % nst;
            const uint32_t st = sbase + (uint32_t)s * stage_bytes;
            mbar_wait(&bar_full[s], (uint32_t)((i / nst) & 1));
            tc_fence_after();
#pragma unroll
            for (int ks = 0; ks < kIChunk / 32; ++ks) {
                const uint64_t ad = sw128_desc(st + 32 * ks), bd = sw128_desc(st + a_bytes + 32 * ks);
                tc_mma<true>(tmem, ad, bd, a.idesc, (i > 0 || ks > 0) ? 1u : 0u);
            }
            tc_commit(&bar_empty[s]);
        }
        if (nloc > 0) tc_commit(&bar_done);
    }
    __syncwarp();
    if (nloc > 0) mbar_wait(&bar_done, 0);
    tc_fence_after();

    // epilogue (one output feature o per thread): the split-K sum in int32, then the corrections and the scaling
    const TcEpilogue e = tc_epilogue(tile, nt, tmem, sbase, tid);
    const int64_t o = o0 + e.r;
    splitk_park<int32_t>(e, tile);
    if (tile.rank == 0) {
        const bool live = o < N;
        const int64_t ch = a.per_channel ? o : 0;
        const float f = live ? __ldg(a.factor + ch) : 0.0f;
        const int32_t zw = !is_lut(F) && live ? __ldg(a.w_zp + ch) : 0;     // LUT codes: zw = 0
        const int64_t sw = live && a.w_rowsum ? (int64_t)__ldg(a.w_rowsum + o) : 0;
        int64_t Kc = K;                                                    // the counted columns
        if constexpr (CP != 0) Kc = (int64_t)a.g.kh * a.g.kw * CP;         // narrow gather: the row tail is not counted
        const int64_t fixed = Kc * (int64_t)a.x_zp * zw - (int64_t)a.x_zp * sw;    // K zx zw - zx Sw[o]
        const float b = a.bias && live ? to_f32<T>(reinterpret_cast<const T*>(a.bias)[o]) : 0.0f;
        const int64_t g0 = a.m0 + n0;                                      // first global row of this CTA
        T* y = reinterpret_cast<T*>(a.y);
        for (int cb = e.cb0; cb < e.nblocks; cb += 2) {
            int32_t v[16];
            splitk_sum(e, tile, cb, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int64_t n = cb * 16 + j;
                if (!live || n >= rows) continue;
                int64_t c = (int64_t)v[j] + fixed;
                if (zw != 0 && a.x_rowsum) c -= (int64_t)zw * __ldg(a.x_rowsum + g0 + n);
                float s = __fmul_rn(__ll2float_rn(c), f);
                if (a.bias) s = __fadd_rn(s, b);
                if (CONV && a.y_nchw) {                                  // pixel g of image b: plane (b, o)
                    const uint32_t g = (uint32_t)(g0 + n), howo = (uint32_t)(a.g.Ho * a.g.Wo);
                    const uint32_t img = fdiv_u32(g, a.div_howo);
                    y[((int64_t)img * N + o) * howo + (g - img * howo)] = from_f32<T>(s);
                } else {
                    y[(g0 + n) * a.ldy + o] = from_f32<T>(s);
                }
            }
        }
    }
    splitk_release();
    tmem_dealloc(warp, tmem, a.tmem_cols);
}

template <WFmt F, bool WSIGNED, typename T>
__global__ void __launch_bounds__(kThreads, 1) packed_igemm_kernel(const __grid_constant__ IgemmArgs a) {
    igemm_body<F, WSIGNED, T, false>(a);
}

template <WFmt F, bool WSIGNED, typename T>
__global__ void __launch_bounds__(kThreads, 1) packed_iconv_kernel(const __grid_constant__ IgemmArgs a) {
    igemm_body<F, WSIGNED, T, true>(a);
}

template <WFmt F, bool WSIGNED, typename T, int CP>
__global__ void __launch_bounds__(kThreads, 1) packed_iconv_narrow_kernel(const __grid_constant__ IgemmArgs a) {
    igemm_body<F, WSIGNED, T, true, CP>(a);
}

}  // namespace mctq

using namespace mctq;

namespace {

using EncodeTiled = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_fn(EncodeTiled* out) {
    static EncodeTiled fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiled>(p);
    }();
    *out = fn;
    return fn ? 0 : (int)cudaErrorSymbolNotFound;
}

// a [rows][K] uint8 matrix (rows K bytes apart) read in boxes of [box_rows][128] bytes, 128-byte swizzle, zeros outside
int encode_codes(EncodeTiled fn, CUtensorMap* map, const void* base, int64_t K, int64_t rows, uint32_t box_rows) {
    const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)K};
    const cuuint32_t box[2] = {(cuuint32_t)kIChunk, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

template <WFmt F, bool WSIGNED, typename T, bool CONV, int CP = 0>
int launch_igemm(const IgemmArgs& a, int64_t M, cudaStream_t st) {
    auto kernel = [] {
        if constexpr (CP != 0) return packed_iconv_narrow_kernel<F, WSIGNED, T, CP>;
        else return CONV ? packed_iconv_kernel<F, WSIGNED, T> : packed_igemm_kernel<F, WSIGNED, T>;
    }();
    const size_t smem = tc_ring_smem(a.stages, a.stage_bytes, a.tmem_cols) + (F == WFmt::LUT8 ? kLut8TableBytes : 0);
    int rc = ensure_smem(kernel, smem);
    if (rc) return rc;
    const int64_t tiles = (a.N + kTcRows - 1) / kTcRows;
    const int64_t ntiles = (M + a.nt - 1) / a.nt;
    // split-K: as many CTAs as fit the GPU at once (one wave), at least one chunk per CTA.  The ring's shared memory decides
    // how many CTAs an SM holds: two for small row tiles, one from nt = 96 on (four stages of 28 KB and more)
    int sms = 0, per_sm = 0;
    if ((rc = sm_count(&sms)) || (rc = cuda_rc(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem))))
        return rc;
    int64_t S = (int64_t)std::max(per_sm, 1) * sms / (tiles * ntiles);
    S = S < 1 ? 1 : S > kIMaxSplit ? kIMaxSplit : S;
    if (S > a.nchunks) S = a.nchunks;
    // the TMA maps and x_rowsum index global rows: a launch gets its range as m0, M
    return tc_launch_rows(kernel, a, M, a.nt, tiles, S, smem, st, [](IgemmArgs& b, int64_t m0, int64_t m) {
        b.m0 = m0;
        b.M = m;
    });
}

// largest in_features whose int32 sum of code products cannot overflow, per (weight, x) signedness
int64_t igemm_max_k(bool w_signed, bool x_signed) {
    if (w_signed && x_signed) return 131071;            // 128 * 128 * K < 2^31
    if (w_signed || x_signed) return 65793;             // 255 * 128 * K < 2^31
    return 33025;                                       // 255 * 255 * K < 2^31
}

// the checks every entry point makes after its shape checks: factors, Sw when zx != 0, aligned codes, zx and K in range
// (w_signed: the signedness of the weight codes the tensor cores multiply)
int igemm_check(const MctqPackedDesc* w, bool w_signed, int64_t K, const void* x_codes, int x_signed, int32_t x_zero_point,
                const int32_t* w_rowsum, const float* factor) {
    if (!factor || (x_zero_point != 0 && !w_rowsum)) return MCTQ_E_BADARG;
    if (!aligned16(x_codes) || !aligned16(w->codes)) return MCTQ_E_BADARG;
    if (x_signed ? (x_zero_point < -128 || x_zero_point > 127) : (x_zero_point < 0 || x_zero_point > 255)) return MCTQ_E_RANGE;
    if (K > igemm_max_k(w_signed, x_signed != 0)) return MCTQ_E_RANGE;
    return 0;
}

// the launch arguments shared by both modes: tiling of M rows, ring, TMEM, instruction descriptor, pointers
void igemm_prepare(IgemmArgs& a, const MctqPackedDesc* w, int64_t N, int64_t K, int64_t M, int x_signed, int32_t x_zero_point,
                   const int32_t* x_rowsum, const int32_t* w_rowsum, const float* factor, const void* bias, void* y) {
    memset(&a, 0, sizeof(a));
    // the table of 8-bit LUT indices (8 KB) and four stages of 256 rows exceed the 200 KB a launch may take: 240 rows fit
    a.nt = tc_row_tile(M, w->kind == MCTQ_PACK_LUT_U8 ? 240 : 256);
    a.nchunks = (int32_t)((K + kIChunk - 1) / kIChunk);
    a.stage_bytes = (uint32_t)(kTcRows * 128 + a.nt * 128);
    // deep rings for the HBM-bound small-batch shapes, while two CTAs still fit an SM's shared memory where they can
    // (the table of 8-bit LUT indices takes its share of that memory)
    const int budget = 112 * 1024 - 1024 - (w->kind == MCTQ_PACK_LUT_U8 ? (int)kLut8TableBytes : 0);
    a.stages = std::min(kIMaxStages, std::max(kIMinStages, budget / (int)a.stage_bytes));
    a.tmem_cols = tmem_columns(a.nt);
    // s32 accumulator, signed or unsigned codes (LUT codes are int8)
    a.idesc = tc_idesc(2u, w->is_signed || pack_is_lut(w->kind) ? 1u : 0u, x_signed ? 1u : 0u, a.nt);
    a.codes = reinterpret_cast<const uint8_t*>(w->codes);
    a.w_zp = w->zp;
    a.x_rowsum = x_rowsum;
    a.w_rowsum = x_zero_point != 0 ? w_rowsum : nullptr;
    a.factor = factor;
    a.bias = bias;
    a.y = y;
    a.N = (int32_t)N;
    a.K = (int32_t)K;
    a.per_channel = w->C != 1;
    a.x_zp = x_zero_point;
}

template <bool CONV, int CP = 0>
int igemm_run(IgemmArgs& a, const MctqPackedDesc* w, int y_dtype, int64_t M, cudaStream_t st) {
    // LUT weights rebuild as f32 (packed_linear_check): one instantiation per index width
    if (w->kind == MCTQ_PACK_LUT_I4) return launch_igemm<WFmt::LUT4, true, float, CONV, CP>(a, M, st);
    if (w->kind == MCTQ_PACK_LUT_U8) return launch_igemm<WFmt::LUT8, true, float, CONV, CP>(a, M, st);
    auto typed = [&](auto fmt_tag, auto signed_tag) {
        constexpr WFmt F = decltype(fmt_tag)::value;
        constexpr bool WS = decltype(signed_tag)::value;
        if (y_dtype == MCTQ_F32) return launch_igemm<F, WS, float, CONV, CP>(a, M, st);
        if (y_dtype == MCTQ_BF16) return launch_igemm<F, WS, __nv_bfloat16, CONV, CP>(a, M, st);
        return launch_igemm<F, WS, __half, CONV, CP>(a, M, st);
    };
    using I4 = std::integral_constant<WFmt, WFmt::I4>;
    using True = std::true_type;
    using False = std::false_type;
    if (pack_is_int4(w->kind)) return w->is_signed ? typed(I4{}, True{}) : typed(I4{}, False{});
    // int8 weights reach the tensor cores as stored: the signedness is in idesc
    return typed(std::integral_constant<WFmt, WFmt::I8>{}, False{});
}

// the LUT table of `K` int8 codes, by value in the launch arguments (entries K.. are 0: no index reaches them)
void igemm_set_lut(IgemmArgs& a, const int8_t* codes, int K) {
    uint8_t b[256] = {};
    memcpy(b, codes, (size_t)K);
    memcpy(a.lut, b, sizeof(b));
}

// mctq_packed_linear_i8 (lut null: affine kinds) and mctq_packed_linear_i8_lut (lut: the table, LUT kinds)
int linear_i8(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x_codes, int x_signed,
              int32_t x_zero_point, int64_t M, const int32_t* x_rowsum, const int32_t* w_rowsum, const float* factor,
              const void* bias, int y_dtype, void* y, int64_t ldy, const int8_t* lut, void* stream) {
    if (const int rc = packed_linear_check(w, out_features, in_features, x_codes, y_dtype, M, y)) return rc;
    const bool int4 = pack_is_int4(w->kind);
    if (in_features % (int4 ? 32 : 16) != 0 || M >= (1LL << 31) || ldy < out_features) return MCTQ_E_BADARG;
    if (const int rc = igemm_check(w, lut || w->is_signed, in_features, x_codes, x_signed, x_zero_point, w_rowsum, factor))
        return rc;
    if (M == 0) return 0;

    IgemmArgs a;
    igemm_prepare(a, w, out_features, in_features, M, x_signed, x_zero_point, lut ? nullptr : x_rowsum, w_rowsum, factor,
                  bias, y);
    if (lut) igemm_set_lut(a, lut, w->K);
    a.ldy = ldy;
    EncodeTiled fn;
    int rc = encode_fn(&fn);
    if (!rc) rc = encode_codes(fn, &a.tm_x, x_codes, in_features, M, (uint32_t)a.nt);
    if (!rc && w->kind == MCTQ_PACK_AFFINE_I8) rc = encode_codes(fn, &a.tm_w, w->codes, in_features, out_features, kTcRows);
    if (rc) return rc;
    return igemm_run<false>(a, w, y_dtype, M, (cudaStream_t)stream);
}

// mctq_packed_conv2d_i8 and mctq_packed_conv2d_i8_lut, as linear_i8; narrow: the narrow gather of Cp = g->Cin = 4 / 8
int conv2d_i8(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cout, const void* x_codes, int x_signed,
              int32_t x_zero_point, const int32_t* x_rowsum, const int32_t* w_rowsum, const float* factor, const void* bias,
              int y_dtype, void* y, int y_nchw, const int8_t* lut, void* stream, bool narrow = false) {
    if (!g) return MCTQ_E_BADARG;
    if (g->N < 0 || g->H < 1 || g->W < 1 || g->Cin < 1 || g->Ho < 1 || g->Wo < 1 || g->kh < 1 || g->kw < 1 || g->sh < 1 ||
        g->sw < 1 || g->dh < 1 || g->dw < 1 || g->pt < 0 || g->pb < 0 || g->pl < 0 || g->pr < 0 || (y_nchw != 0 && y_nchw != 1))
        return MCTQ_E_BADARG;
    const bool int4 = pack_is_int4(w->kind);
    const int64_t step = int4 ? 32 : 16;                       // narrow: kh * kw * Cp and a row tail up to the granule
    const int64_t K = narrow ? ((int64_t)g->Cin * g->kh * g->kw + step - 1) / step * step : (int64_t)g->Cin * g->kh * g->kw;
    const int64_t M = (int64_t)g->N * g->Ho * g->Wo;
    if (const int rc = packed_linear_check(w, Cout, K, x_codes, y_dtype, M, y)) return rc;
    if ((!narrow && g->Cin % 16 != 0) || (int4 && K % 32 != 0) || M >= (1LL << 31)) return MCTQ_E_BADARG;
    if (const int rc = igemm_check(w, lut || w->is_signed, K, x_codes, x_signed, x_zero_point, w_rowsum, factor)) return rc;
    if (M == 0) return 0;

    IgemmArgs a;
    igemm_prepare(a, w, Cout, K, M, x_signed, x_zero_point, lut ? nullptr : x_rowsum, w_rowsum, factor, bias, y);
    if (lut) igemm_set_lut(a, lut, w->K);
    a.ldy = Cout;
    a.x_nhwc = reinterpret_cast<const uint8_t*>(x_codes);
    a.g = *g;
    a.div_howo = make_fastdiv((uint32_t)(g->Ho * g->Wo));
    a.div_wo = make_fastdiv((uint32_t)g->Wo);
    a.div_cin = make_fastdiv((uint32_t)g->Cin);
    a.div_kw = make_fastdiv((uint32_t)g->kw);
    a.y_nchw = y_nchw;
    a.zx_splat = ((uint32_t)x_zero_point & 0xFFu) * 0x01010101u;
    if (w->kind == MCTQ_PACK_AFFINE_I8) {
        EncodeTiled fn;
        int rc = encode_fn(&fn);
        if (!rc) rc = encode_codes(fn, &a.tm_w, w->codes, K, Cout, kTcRows);
        if (rc) return rc;
    }
    if (narrow) {
        return g->Cin == 4 ? igemm_run<true, 4>(a, w, y_dtype, M, (cudaStream_t)stream)
                           : igemm_run<true, 8>(a, w, y_dtype, M, (cudaStream_t)stream);
    }
    return igemm_run<true>(a, w, y_dtype, M, (cudaStream_t)stream);
}

}  // namespace

extern "C" {

int64_t mctq_packed_linear_i8_max_k(int w_signed, int x_signed) { return igemm_max_k(w_signed != 0, x_signed != 0); }

int mctq_packed_linear_i8(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x_codes,
                          int x_signed, int32_t x_zero_point, int64_t M, const int32_t* x_rowsum, const int32_t* w_rowsum,
                          const float* factor, const void* bias, int y_dtype, void* y, int64_t ldy, void* stream) {
    MCTQ_NVTX("mctq_packed_linear_i8");
    if (!w || pack_is_lut(w->kind)) return MCTQ_E_BADARG;
    return linear_i8(w, out_features, in_features, x_codes, x_signed, x_zero_point, M, x_rowsum, w_rowsum, factor, bias,
                     y_dtype, y, ldy, nullptr, stream);
}

int mctq_packed_linear_i8_lut(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x_codes,
                              int x_signed, int32_t x_zero_point, int64_t M, const int32_t* x_rowsum, const int32_t* w_rowsum,
                              const float* factor, const void* bias, int y_dtype, void* y, int64_t ldy,
                              const int8_t* lut_codes_host, void* stream) {
    MCTQ_NVTX("mctq_packed_linear_i8_lut");
    if (!w || !pack_is_lut(w->kind) || !lut_codes_host) return MCTQ_E_BADARG;
    return linear_i8(w, out_features, in_features, x_codes, x_signed, x_zero_point, M, x_rowsum, w_rowsum, factor, bias,
                     y_dtype, y, ldy, lut_codes_host, stream);
}

int mctq_packed_linear_i8_padded(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, int64_t ldc,
                                 const void* x_codes, int x_signed, int32_t x_zero_point, int64_t M, const int32_t* x_rowsum,
                                 const int32_t* w_rowsum, const float* factor, const void* bias, int y_dtype, void* y,
                                 int64_t ldy, const int8_t* lut_codes_host, void* stream) {
    MCTQ_NVTX("mctq_packed_linear_i8_padded");
    if (!w || pack_is_lut(w->kind) != (lut_codes_host != nullptr)) return MCTQ_E_BADARG;
    if (in_features < 1 || ldc < in_features) return MCTQ_E_BADARG;
    // the GEMM of mctq_packed_linear_i8 over rows of ldc columns (its checks: ldc % 16 / 32, the int32 bound on ldc)
    return linear_i8(w, out_features, ldc, x_codes, x_signed, x_zero_point, M, x_rowsum, w_rowsum, factor, bias, y_dtype, y,
                     ldy, lut_codes_host, stream);
}

int mctq_packed_conv2d_i8_padded(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cp, int64_t Cout,
                                 const void* x_codes, int x_signed, int32_t x_zero_point, const int32_t* x_rowsum,
                                 const int32_t* w_rowsum, const float* factor, const void* bias, int y_dtype, void* y,
                                 int y_nchw, const int8_t* lut_codes_host, void* stream) {
    MCTQ_NVTX("mctq_packed_conv2d_i8_padded");
    if (!w || !g || pack_is_lut(w->kind) != (lut_codes_host != nullptr)) return MCTQ_E_BADARG;
    if (g->Cin < 1 || Cp < g->Cin || Cp > (1 << 20) || (Cp != 4 && Cp != 8 && Cp % 16 != 0)) return MCTQ_E_BADARG;
    MctqConv2dGeom gp = *g;                                    // the kernel sees Cin := Cp
    gp.Cin = (int32_t)Cp;
    return conv2d_i8(w, &gp, Cout, x_codes, x_signed, x_zero_point, x_rowsum, w_rowsum, factor, bias, y_dtype, y, y_nchw,
                     lut_codes_host, stream, Cp < 16);
}

int mctq_packed_conv2d_i8(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cout, const void* x_codes, int x_signed,
                          int32_t x_zero_point, const int32_t* x_rowsum, const int32_t* w_rowsum, const float* factor,
                          const void* bias, int y_dtype, void* y, int y_nchw, void* stream) {
    MCTQ_NVTX("mctq_packed_conv2d_i8");
    if (!w || pack_is_lut(w->kind)) return MCTQ_E_BADARG;
    return conv2d_i8(w, g, Cout, x_codes, x_signed, x_zero_point, x_rowsum, w_rowsum, factor, bias, y_dtype, y, y_nchw,
                     nullptr, stream);
}

int mctq_packed_conv2d_i8_lut(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cout, const void* x_codes,
                              int x_signed, int32_t x_zero_point, const int32_t* x_rowsum, const int32_t* w_rowsum,
                              const float* factor, const void* bias, int y_dtype, void* y, int y_nchw,
                              const int8_t* lut_codes_host, void* stream) {
    MCTQ_NVTX("mctq_packed_conv2d_i8_lut");
    if (!w || !pack_is_lut(w->kind) || !lut_codes_host) return MCTQ_E_BADARG;
    return conv2d_i8(w, g, Cout, x_codes, x_signed, x_zero_point, x_rowsum, w_rowsum, factor, bias, y_dtype, y, y_nchw,
                     lut_codes_host, stream);
}

}  // extern "C"
