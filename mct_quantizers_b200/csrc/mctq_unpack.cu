// mctq_unpack.cu -- rebuild weights from packed codes (affine int8 / int4 codes, LUT indices) for many tensors per launch:
// the consumer side of the code wire format for packed models (pytorch/packed_weights.py).
//
// The result is bit-identical to the fake-quant kernels' output for the weight the codes were taken from:
//   affine: y = from_f32<T>((q - zp_c) * s_c)          T = f32 / bf16 / f16, one f32 rounding then one rounding to T
//   LUT:    y = q_idx * thr_c  (f32),  q_k = lut_k / 2^(bw - signed) formed on the host in f32
// Launch pattern of fq_lut_multi_kernel (mctq_lutp.cu): the per-tensor argument blocks are __grid_constant__ kernel
// parameters, the grid is 2-D (y = tensor, x = tile), every launch is specialised for one variant (kind, output dtype,
// channel mode, vector width) and the host plan groups the tensors by variant, <= 64 tensors per launch.
#include "mctq_plan.cuh"

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

struct UnpackVariant {
    int32_t kind, dtype, mode, v, pad[3];
};
template <int CAP>
using UnpackParamsT = PlanChunk<UnpackVariant, UnpackArgs, CAP>;

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

using UnpackPlan = Plan<UnpackVariant, UnpackArgs, 0x4d51554eu>;   // 'MQUN'

template <int KIND, typename T, int MODE, int V, int CAP>
int launch_unpack_variant(const UnpackParamsT<CAP>& p, cudaStream_t st) {
    // ranges "unknown": the successor of this launch takes the late dependent-launch order
    return launch_streaming(unpack_multi_kernel<KIND, T, MODE, V, CAP>, dim3((unsigned)p.tiles[CAP], (unsigned)p.n_desc), 0, st, p);
}

// exactly the (mode, vector width) pairs unpack_describe selects
template <int KIND, typename T, int CAP>
int launch_unpack_typed(const UnpackParamsT<CAP>& c, cudaStream_t st) {
    constexpr int V0 = sizeof(T) == 2 ? 8 : 4;                                              // per tensor
    constexpr bool WIDE1 = sizeof(T) == 2 || pack_is_int4(KIND);                             // per channel
    const UnpackVariant& var = c.var;
    if (var.mode == 0 && var.v == V0) return launch_unpack_variant<KIND, T, 0, V0, CAP>(c, st);
    if (var.mode == 1 && var.v == 4) return launch_unpack_variant<KIND, T, 1, 4, CAP>(c, st);
    if constexpr (WIDE1) if (var.mode == 1 && var.v == 8) return launch_unpack_variant<KIND, T, 1, 8, CAP>(c, st);
    if (var.mode == 2 && var.v == 4) return launch_unpack_variant<KIND, T, 2, 4, CAP>(c, st);
    return MCTQ_E_BADARG;
}

template <int CAP>
int launch_unpack_chunk(const UnpackParamsT<CAP>& c, cudaStream_t st) {
    return dispatch_packed(c.var.kind, c.var.dtype, [&](auto kind, auto type) {
        return launch_unpack_typed<decltype(kind)::value, typename decltype(type)::type, CAP>(c, st);
    });
}

// argument block, variant and tiles of one descriptor; 0 or MCTQ_E_*.  An empty tensor is skipped (nothing to launch).
int unpack_describe(const MctqPackedDesc& d, UnpackPlan::Item& it) {
    if (const int rc = pack_check_kind(d.kind, d.y_dtype)) return rc;
    if (d.n < 0 || d.C < 1 || d.inner < 1 || d.C >= (1LL << 31) || d.inner >= (1LL << 31)) return MCTQ_E_BADARG;
    if (d.n % (d.C * d.inner) != 0) return MCTQ_E_BADARG;                      // [outer][C][inner]
    if (d.n == 0) { it.skip = true; return 0; }
    if (!d.codes || !d.y || !d.scale || !aligned16(d.codes) || !aligned16(d.y)) return MCTQ_E_BADARG;
    if (const int rc = pack_check_params(d)) return rc;
    const bool lut = pack_is_lut(d.kind);
    UnpackArgs* a = &it.args;
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
    const int mode = d.C == 1 ? 0 : (d.inner % 4 == 0 ? 1 : 2);
    // 8 codes per vector where the whole vector lies in one channel and (f32) y takes a 32-byte store: always for 2-byte
    // outputs (16-byte instead of 8-byte stores); for f32 where dequant_affine measured it faster, packed nibbles per channel
    const bool fits8 = mode != 2 && (mode == 0 || d.inner % 8 == 0) && (d.y_dtype != MCTQ_F32 || aligned32(d.y));
    const int v = fits8 && (d.y_dtype != MCTQ_F32 || (mode == 1 && pack_is_int4(d.kind))) ? 8 : 4;
    it.var = {d.kind, d.y_dtype, mode, v, {}};
    const int64_t per_tile = (int64_t)kThreads * kUnpackUnroll * v;
    it.tiles = (d.n + per_tile - 1) / per_tile;
    return 0;
}

}  // namespace

extern "C" {

size_t mctq_unpack_plan_bytes(const MctqPackedDesc* descs, int n_desc) {
    UnpackPlan plan;
    return plan.compile(descs, n_desc, unpack_describe) ? 0 : plan.bytes();
}

int64_t mctq_unpack_plan(const MctqPackedDesc* descs, int n_desc, void* plan_host_out, size_t plan_bytes) {
    UnpackPlan plan;
    if (const int rc = plan.compile(descs, n_desc, unpack_describe)) return rc;
    return plan.write(plan_host_out, plan_bytes);
}

int mctq_unpack_multi(const void* plan_host, void* stream) {
    MCTQ_NVTX("mctq_unpack_multi");
    return UnpackPlan::run<4>(plan_host, 0, [&](const auto& p, const PlanHeader&) { return launch_unpack_chunk(p, (cudaStream_t)stream); });
}

}  // extern "C"
