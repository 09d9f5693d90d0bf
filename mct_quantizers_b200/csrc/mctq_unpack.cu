// mctq_unpack.cu -- rebuild weights from packed codes (affine int8 / int4 codes, LUT indices) for many tensors per launch:
// the consumer side of the code wire format for packed models (pytorch/packed_weights.py).
//
// The result is bit-identical to the fake-quant kernels' output for the weight the codes were taken from:
//   affine: y = from_f32<T>((q - zp_c) * s_c)          T = f32 / bf16 / f16, one f32 rounding then one rounding to T
//   LUT:    y = q_idx * thr_c  (f32),  q_k = lut_k / 2^(bw - signed) formed on the host in f32
// Launch pattern of fq_lut_multi_kernel (mctq_lutp.cu): the per-tensor argument blocks are __grid_constant__ kernel
// parameters, the grid is 2-D (y = tensor, x = tile), every launch is specialised for one variant (kind, output dtype,
// channel mode, vector width) and the host plan groups the tensors by variant, <= 64 tensors per launch.
#include <algorithm>
#include <vector>

#include "mctq_common.cuh"

namespace mctq {

struct UnpackArgs {
    const uint8_t* codes;
    void* y;
    const float* scale;          // affine: scale[C]; LUT: thr[C]
    const int32_t* zp;           // affine: zp[C]
    const float* quot;           // LUT: q_k, K entries
    int64_t n;
    uint32_t C, inner;
    FastDiv div_inner, div_C;
    int32_t is_signed, K;
};

constexpr int kUnpackMaxDesc = 64;
template <int CAP>
struct UnpackParamsT {
    int32_t n_desc, kind, dtype, mode, v, pad[3];
    int32_t tiles[CAP + 4];      // tiles[k] = tiles of tensor k; tiles[CAP] = the largest of them (grid x)
    UnpackArgs e[CAP];
};
using UnpackParams = UnpackParamsT<kUnpackMaxDesc>;
static_assert(sizeof(UnpackParams) <= 32764, "kernel parameter space");

constexpr int kUnpackUnroll = 4;

template <int KIND, typename T, int MODE, int V, int CAP>
__global__ void __launch_bounds__(kThreads) unpack_multi_kernel(const __grid_constant__ UnpackParamsT<CAP> p) {
    constexpr bool LUT = pack_is_lut(KIND);
    constexpr int CODE = pack_code_mode(KIND);
    constexpr int NQ = pack_max_k(KIND);
    constexpr int64_t TILE = (int64_t)kThreads * kUnpackUnroll * V;
    __shared__ float sm_q[LUT ? NQ : 1];
    const uint32_t k = blockIdx.y;
    if ((int32_t)blockIdx.x >= p.tiles[k]) return;
    const UnpackArgs& a = p.e[k];
    pdl_wait();
    pdl_launch_dependents();
    if constexpr (LUT) {
        if (threadIdx.x < NQ) sm_q[threadIdx.x] = (int32_t)threadIdx.x < a.K ? __ldg(a.quot + threadIdx.x) : 0.0f;
        __syncthreads();
        codes_tile<CODE, MODE, V, kUnpackUnroll>(a.codes, reinterpret_cast<float*>(a.y), (int64_t)blockIdx.x * TILE, a.n, 0, a.C,
                                                 a.inner, 0, a.div_inner, a.div_C, LutCodeOp{a.scale, sm_q});
    } else {
        codes_tile<CODE, MODE, V, kUnpackUnroll>(a.codes, reinterpret_cast<T*>(a.y), (int64_t)blockIdx.x * TILE, a.n, a.is_signed,
                                                 a.C, a.inner, 0, a.div_inner, a.div_C, AffineCodeOp{a.scale, a.zp});
    }
}

}  // namespace mctq

using namespace mctq;

namespace {

constexpr uint32_t kUnpackMagic = 0x4d51554eu;   // 'MQUN'
struct UnpackHeader {        // 64 bytes
    uint32_t magic;
    int32_t n_desc, n_chunks, reserved0;
    int64_t total_tiles;
    int32_t reserved[10];
};
static_assert(sizeof(UnpackHeader) == 64, "unpack header layout");

size_t unpack_bytes(int n_chunks) { return sizeof(UnpackHeader) + (size_t)n_chunks * sizeof(UnpackParams); }

template <int KIND, typename T, int MODE, int V, int CAP>
int launch_unpack_variant(const UnpackParams& c, cudaStream_t st) {
    static thread_local UnpackParamsT<CAP> p;                // up to 7 KB: not on the stack
    p.n_desc = c.n_desc; p.kind = c.kind; p.dtype = c.dtype; p.mode = c.mode; p.v = c.v;
    memcpy(p.tiles, c.tiles, (size_t)c.n_desc * sizeof(int32_t));
    memcpy(p.e, c.e, (size_t)c.n_desc * sizeof(UnpackArgs));
    // ranges "unknown": the successor of this launch takes the late dependent-launch order
    return launch_streaming(unpack_multi_kernel<KIND, T, MODE, V, CAP>, dim3((unsigned)c.tiles[kUnpackMaxDesc], (unsigned)c.n_desc),
                            0, st, p);
}

// exactly the (mode, vector width) pairs unpack_make_args selects
template <int KIND, typename T, int CAP>
int launch_unpack_typed(const UnpackParams& c, cudaStream_t st) {
    constexpr int V0 = sizeof(T) == 2 ? 8 : 4;                                              // per tensor
    constexpr bool WIDE1 = sizeof(T) == 2 || pack_is_int4(KIND);                             // per channel
    if (c.mode == 0 && c.v == V0) return launch_unpack_variant<KIND, T, 0, V0, CAP>(c, st);
    if (c.mode == 1 && c.v == 4) return launch_unpack_variant<KIND, T, 1, 4, CAP>(c, st);
    if constexpr (WIDE1) if (c.mode == 1 && c.v == 8) return launch_unpack_variant<KIND, T, 1, 8, CAP>(c, st);
    if (c.mode == 2 && c.v == 4) return launch_unpack_variant<KIND, T, 2, 4, CAP>(c, st);
    return MCTQ_E_BADARG;
}

template <int CAP>
int launch_unpack_chunk(const UnpackParams& c, cudaStream_t st) {
    return dispatch_packed(c.kind, c.dtype, [&](auto kind, auto type) {
        return launch_unpack_typed<decltype(kind)::value, typename decltype(type)::type, CAP>(c, st);
    });
}

// argument block and variant of one descriptor; 0 or MCTQ_E_*.  *skip = 1 for an empty tensor (nothing to launch).
int unpack_make_args(const MctqPackedDesc& d, UnpackArgs* a, int* mode, int* v, int* skip) {
    *skip = 0;
    if (const int rc = pack_check_kind(d.kind, d.y_dtype)) return rc;
    if (d.n < 0 || d.C < 1 || d.inner < 1 || d.C >= (1LL << 31) || d.inner >= (1LL << 31)) return MCTQ_E_BADARG;
    if (d.n % (d.C * d.inner) != 0) return MCTQ_E_BADARG;                      // [outer][C][inner]
    if (d.n == 0) { *skip = 1; return 0; }
    if (!d.codes || !d.y || !d.scale || !aligned16(d.codes) || !aligned16(d.y)) return MCTQ_E_BADARG;
    if (const int rc = pack_check_params(d)) return rc;
    const bool lut = pack_is_lut(d.kind);
    memset(a, 0, sizeof(*a));
    a->codes = reinterpret_cast<const uint8_t*>(d.codes);
    a->y = d.y;
    a->scale = d.scale;
    a->zp = lut ? nullptr : d.zp;
    a->quot = lut ? d.lut_quotients : nullptr;
    a->n = d.n;
    a->C = (uint32_t)d.C;
    a->inner = (uint32_t)(d.C == 1 ? 1 : d.inner);
    a->div_inner = make_fastdiv(a->inner);
    a->div_C = make_fastdiv(a->C);
    a->is_signed = lut ? 0 : (d.is_signed ? 1 : 0);
    a->K = lut ? d.K : 0;
    *mode = d.C == 1 ? 0 : (d.inner % 4 == 0 ? 1 : 2);
    // 8 codes per vector where the whole vector lies in one channel and (f32) y takes a 32-byte store: always for 2-byte
    // outputs (16-byte instead of 8-byte stores); for f32 where dequant_affine measured it faster, packed nibbles per channel
    const bool fits8 = *mode != 2 && (*mode == 0 || d.inner % 8 == 0) && (d.y_dtype != MCTQ_F32 || aligned32(d.y));
    *v = fits8 && (d.y_dtype != MCTQ_F32 || (*mode == 1 && pack_is_int4(d.kind))) ? 8 : 4;
    return 0;
}

inline int variant_key(int kind, int dtype, int mode, int v) { return (((kind - 1) * 3 + dtype) * 3 + mode) * 2 + (v == 8 ? 1 : 0); }
constexpr int kUnpackVariants = 4 * 3 * 3 * 2;

// a compiled plan on the host: the header and the chunks of the blob mctq_unpack_plan writes
struct UnpackPlanHost {
    UnpackHeader h = {};
    std::vector<UnpackParams> chunks;
};

// validates every descriptor and groups the tensors by kernel variant (one chunk = one launch, <= 64 tensors whose tile counts
// are within a factor of 16: the grid is [largest tile count] x [tensors] and CTAs past a tensor's last tile exit at once);
// 0 or MCTQ_E_*
int unpack_compile(const MctqPackedDesc* descs, int n_desc, UnpackPlanHost& plan) {
    if (!descs || n_desc < 1) return MCTQ_E_BADARG;
    std::vector<UnpackArgs> args((size_t)n_desc);
    std::vector<int> key((size_t)n_desc, -1), vv((size_t)n_desc), md((size_t)n_desc);
    for (int k = 0; k < n_desc; ++k) {
        int skip = 0;
        const int rc = unpack_make_args(descs[k], &args[k], &md[k], &vv[k], &skip);
        if (rc) return rc;
        if (!skip) key[k] = variant_key(descs[k].kind, descs[k].y_dtype, md[k], vv[k]);
    }
    int64_t total = 0;
    for (int var = 0; var < kUnpackVariants; ++var) {
        std::vector<std::pair<int64_t, int>> order;               // tensors of this variant, largest first
        for (int k = 0; k < n_desc; ++k) {
            if (key[k] != var) continue;
            const int64_t per_tile = (int64_t)kThreads * kUnpackUnroll * vv[k];
            const int64_t tiles = (descs[k].n + per_tile - 1) / per_tile;
            if (tiles > 0x7fffffffLL) return MCTQ_E_BADARG;
            order.push_back({-tiles, k});
        }
        std::stable_sort(order.begin(), order.end());
        int in_chunk = 0;
        int64_t first_tiles = 0;
        for (const auto& it : order) {
            const int64_t tiles = -it.first;
            const int k = it.second;
            if (in_chunk == kUnpackMaxDesc || (in_chunk && tiles * 16 < first_tiles)) in_chunk = 0;
            if (in_chunk == 0) {
                first_tiles = tiles;
                UnpackParams& c = plan.chunks.emplace_back();         // zero-filled
                c.kind = descs[k].kind; c.dtype = descs[k].y_dtype; c.mode = md[k]; c.v = vv[k];
                c.tiles[kUnpackMaxDesc] = (int32_t)tiles;
            }
            UnpackParams& c = plan.chunks.back();
            c.e[in_chunk] = args[k];
            c.tiles[in_chunk] = (int32_t)tiles;
            c.n_desc = ++in_chunk;
            total += tiles;
        }
    }
    plan.h.magic = kUnpackMagic;
    plan.h.n_desc = n_desc;
    plan.h.n_chunks = (int32_t)plan.chunks.size();
    plan.h.total_tiles = total;
    return 0;
}

}  // namespace

extern "C" {

size_t mctq_unpack_plan_bytes(const MctqPackedDesc* descs, int n_desc) {
    UnpackPlanHost plan;
    return unpack_compile(descs, n_desc, plan) ? 0 : unpack_bytes(plan.h.n_chunks);
}

int64_t mctq_unpack_plan(const MctqPackedDesc* descs, int n_desc, void* plan_host_out, size_t plan_bytes) {
    UnpackPlanHost plan;
    if (const int rc = unpack_compile(descs, n_desc, plan)) return rc;
    if (!plan_host_out || plan_bytes < unpack_bytes(plan.h.n_chunks)) return MCTQ_E_BADARG;
    uint8_t* out = reinterpret_cast<uint8_t*>(plan_host_out);
    memcpy(out, &plan.h, sizeof(UnpackHeader));
    if (!plan.chunks.empty()) memcpy(out + sizeof(UnpackHeader), plan.chunks.data(), plan.chunks.size() * sizeof(UnpackParams));
    return plan.h.total_tiles;
}

int mctq_unpack_multi(const void* plan_host, void* stream) {
    MCTQ_NVTX("mctq_unpack_multi");
    if (!plan_host) return MCTQ_E_BADARG;
    const UnpackHeader* h = reinterpret_cast<const UnpackHeader*>(plan_host);
    if (h->magic != kUnpackMagic || h->n_desc < 1 || h->n_chunks < 0) return MCTQ_E_BADARG;
    const UnpackParams* chunks = reinterpret_cast<const UnpackParams*>(reinterpret_cast<const uint8_t*>(plan_host) + sizeof(UnpackHeader));
    for (int c = 0; c < h->n_chunks; ++c) {
        const UnpackParams& p = chunks[c];
        const int rc = p.n_desc <= 4 ? launch_unpack_chunk<4>(p, (cudaStream_t)stream) : launch_unpack_chunk<kUnpackMaxDesc>(p, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return 0;
}

}  // extern "C"
