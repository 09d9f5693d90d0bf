/*
 * mctq.h -- C ABI of libmctq_sm100.so, the B200 (sm_100a) fake-quant path that replaces the arithmetic
 * underneath mct_quantizers' PyTorch inferable quantizers.
 *
 * The reference (sony/mct_quantizers 1.6.0) is pure Python and has no FFI of its own: its hot path is
 *   - torch.fake_quantize_per_tensor_affine / torch.fake_quantize_per_channel_affine, called from
 *       mct_quantizers/pytorch/quantizers/weights_inferable_quantizers/weights_symmetric_inferable_quantizer.py:139-151
 *       mct_quantizers/pytorch/quantizers/weights_inferable_quantizers/weights_uniform_inferable_quantizer.py:153-165
 *       mct_quantizers/pytorch/quantizers/activation_inferable_quantizers/activation_symmetric_inferable_quantizer.py:113-117
 *       mct_quantizers/pytorch/quantizers/activation_inferable_quantizers/activation_uniform_inferable_quantizer.py:124-128
 *   - lut_quantizer / int_quantization_with_threshold, mct_quantizers/pytorch/quantizer_utils.py:95-170, called from
 *       .../weights_lut_symmetric_inferable_quantizer.py:114-122 and .../activation_lut_pot_inferable_quantizer.py:86-91
 * Each entry point below names the reference call site(s) it stands in for.  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, a positive cudaError_t on a CUDA failure, or a negative
 *     MCTQ_E_* code on a bad argument; nothing throws, nothing allocates device memory, and the
 *     device-pointer entry points never synchronise: work is enqueued on `stream` (a cudaStream_t
 *     passed as void*; NULL = legacy default stream).
 *   - tensors are contiguous and are viewed as [outer][C][inner]; element i of the logical tensor has
 *     channel (i / inner) % C.  C == 1 is per-tensor quantisation.  `elem_offset` is the logical index
 *     of x[0], so a caller can hand in any flat slice of a tensor (batch / channel-block shards,
 *     host-staging chunks) without re-deriving parameters.
 *   - dtype tags: MCTQ_F32 / MCTQ_BF16 / MCTQ_F16 describe x (and y for the affine ops).
 *   - grouped multi-tensor plans (mctq_unpack_plan, mctq_lut_multi_plan) compile a HOST descriptor array into an opaque
 *     HOST blob that travels as kernel parameters, so there is no device-side copy of the plan.  Grouping rule: the
 *     tensors are sorted by kernel variant, and within a variant largest first (ties in descriptor order); a launch holds
 *     one variant and a new launch starts after 64 tensors, or at a tensor with fewer than 1/16 of the tiles of the
 *     launch's first (largest) tensor.  Each launch runs on a 2-D grid: one row of CTAs per tensor, as many CTAs per
 *     row as its largest tensor has tiles.
 *   - arithmetic contract (bit-exact with CPU torch 2.11, see DESIGN.md):
 *       affine:  inv = 1.0f / s;  q = clamp(rint(x * inv) + zp, qmin, qmax);  y = (q - zp) * s
 *       lut:     t = clip((x / (thr + eps)) * 2^(bw - signed), lo, hi);  idx = first argmin_k |t - lut_k|;
 *                y = (lut[idx] / 2^(bw - signed)) * thr            (y is always f32)
 *     valid for finite inputs, |qmin - zp|, |qmax - zp| < 2^21 (else an rint-based slower variant is
 *     selected automatically) and NaN -> qmin / LUT index 0.
 */
#ifndef MCTQ_H_
#define MCTQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCTQ_ABI_VERSION 1

/* dtype tags */
#define MCTQ_F32 0
#define MCTQ_BF16 1
#define MCTQ_F16 2

/* integer-code / LUT-index emission */
#define MCTQ_CODES_NONE 0
#define MCTQ_CODES_INT8 1 /* one byte per element: (uint8_t)(q & 0xff) -- int8 when qmin < 0, uint8 otherwise */
#define MCTQ_CODES_INT4 2 /* two elements per byte, element 2j in the low nibble; n is rounded up to even */

/* argument errors (negative so they cannot collide with cudaError_t) */
#define MCTQ_E_BADARG (-1)
#define MCTQ_E_DTYPE (-2)
#define MCTQ_E_RANGE (-3)   /* qmin > qmax, or codes requested for a range that does not fit the code width */
#define MCTQ_E_LUT (-4)     /* malformed LUT table blob */
#define MCTQ_E_NODEVICE (-5)

int mctq_abi_version(void);
/* compile-time facts a caller can assert on: "sm_100a", tile geometry, ... (static string, never freed) */
const char* mctq_build_info(void);

/* ------------------------------------------------------------------------------------------------------
 * Affine fake-quant, device pointers.
 * Replaces: torch.fake_quantize_per_channel_affine(x, scales, zero_points, axis, qmin, qmax)
 *             (weights_symmetric_inferable_quantizer.py:139-144, weights_uniform_inferable_quantizer.py:153-158)
 *           torch.fake_quantize_per_tensor_affine(x, scales[1], zero_points[1], qmin, qmax)   [tensor qparams]
 *             (weights_symmetric_inferable_quantizer.py:147-151, weights_uniform_inferable_quantizer.py:160-165)
 * x, y       device, n elements of x_dtype; y may be NULL when only codes are wanted
 * codes      device or NULL; layout per code_mode
 * scale, zp  device arrays of C entries (read on the device: no host sync, unlike the reference's
 *            per-channel path which does two .item() round trips per call).  ATen rejects per-channel zero points
 *            outside [qmin, qmax]; this entry point cannot look (no sync) and only needs |q - zp[c]| < 2^22 for every
 *            q in [qmin, qmax] when qmax - qmin < 2^21 (the fast-rounding path); the Python quantizers check the range on
 *            the host at construction time and raise ATen's error.
 */
int mctq_fq_affine(const void* x, void* y, void* codes, int64_t n, int x_dtype,
                   const float* scale, const int32_t* zp, int64_t C, int64_t inner, int64_t elem_offset,
                   int32_t qmin, int32_t qmax, int code_mode, void* stream);

/* Per-tensor affine fake-quant with scalar parameters passed by value.
 * Replaces: torch.fake_quantize_per_tensor_affine(x, scale=float, zero_point=int, qmin, qmax)
 *             (activation_symmetric_inferable_quantizer.py:113-117, activation_uniform_inferable_quantizer.py:124-128)
 * `scale` is the Python float already narrowed to f32 (what ATen does internally). */
int mctq_fq_affine_scalar(const void* x, void* y, void* codes, int64_t n, int x_dtype,
                          float scale, int32_t zp, int32_t qmin, int32_t qmax, int code_mode, void* stream);

/* Prepared per-channel parameters (the fast path for per-channel weights): mctq_affine_prepare turns scale[C] / zp[C]
 * into a device blob holding, per channel, the record {1/s, s, zp, (float)zp} plus the same values as three arrays; the
 * kernels launched by mctq_fq_affine_prepared stage the channel window of every tile from that blob with 1-D TMA bulk
 * copies (cp.async.bulk + mbarrier) instead of per-thread load / divide / store loops.  Same reference call sites and
 * arithmetic as mctq_fq_affine (1/s is the same IEEE f32 reciprocal, computed once).  Neither call synchronises.
 *   prepared_dev   DEVICE buffer, 16-byte aligned, >= mctq_affine_prepared_bytes(C) bytes; valid for as long as
 *                  scale / zp do not change */
size_t mctq_affine_prepared_bytes(int64_t C);
int mctq_affine_prepare(const float* scale, const int32_t* zp, int64_t C, void* prepared_dev, size_t prepared_bytes,
                        void* stream);
int mctq_fq_affine_prepared(const void* x, void* y, void* codes, int64_t n, int x_dtype, const void* prepared_dev,
                            int64_t C, int64_t inner, int64_t elem_offset, int32_t qmin, int32_t qmax, int code_mode,
                            void* stream);

/* Per-tensor affine fake-quant fused with the elementwise producer of the activation (SURVEY 8f rank 3).
 * Replaces the pair  <producer>(x[, x2]) -> PytorchActivationQuantizationHolder.forward
 *   (mct_quantizers/pytorch/activation_quantization_holder.py:43-53 after a ReLU / ReLU6 / residual add of the exported
 *   model) with ONE kernel: the intermediate activation is never written to HBM.  Bit-identical to the eager
 *   composition (producer evaluated in f32 and rounded to x_dtype, then the recipe of mctq_fq_affine_scalar).
 * x2 is read only by the ADD flavours (same dtype and length as x). */
#define MCTQ_PRE_RELU 1      /* y = fq(max(x, 0))        */
#define MCTQ_PRE_RELU6 2     /* y = fq(min(max(x, 0), 6)) */
#define MCTQ_PRE_ADD 3       /* y = fq(x + x2)           */
#define MCTQ_PRE_ADD_RELU 4  /* y = fq(max(x + x2, 0))   */
int mctq_fq_affine_scalar_pre(const void* x, const void* x2, void* y, int64_t n, int x_dtype, int pre_op, float scale,
                              int32_t zp, int32_t qmin, int32_t qmax, void* stream);

/* Dequantise codes written by the functions above: y = (q - zp) * s  (f32 out; exact for |q - zp| < 2^22, i.e. for any
 * zero point inside the code range).  No reference call site: this is the consumer side of the code wire format
 * (SURVEY 8f rank 2). */
int mctq_dequant_affine(const void* codes, int code_mode, int is_signed, float* y, int64_t n,
                        const float* scale, const int32_t* zp, int64_t C, int64_t inner, int64_t elem_offset,
                        void* stream);

/* Rebuild weights from packed codes, many tensors per launch (packed models: mct_quantizers_b200/pytorch/packed_weights.py).
 * No reference call site: the result is bit-identical to what the weight quantizer returns for the float weight the codes were
 * taken from (mctq_fq_affine* with code_mode / mctq_fq_lut* with idx_mode), so a packed model computes the float model's
 * outputs.  Per tensor, elements are [outer][C][inner] in memory order and
 *   affine: y = (T)((float)(q - zp[c]) * scale[c])      T = y_dtype (one f32 rounding, then one rounding to T)
 *   LUT:    y = lut_quotients[idx] * thr[c]             f32 out; lut_quotients[k] = lut_k / 2^(bw - signed) in f32, idx is the
 *                                                       index into the ORIGINAL centroid list (what mctq_fq_lut* emit)
 * mctq_unpack_plan compiles the HOST descriptor array into a HOST plan blob of mctq_unpack_plan_bytes(descs, n_desc) bytes
 * (returns the total number of tiles, or < 0: MCTQ_E_BADARG for a malformed descriptor or a code / output buffer that is not
 * 16-byte aligned, MCTQ_E_DTYPE, MCTQ_E_LUT for K outside 1..256 (1..16 for MCTQ_PACK_LUT_I4)).  Tensors are grouped by the
 * plan grouping rule (Conventions above); the kernel variant is (kind, output dtype, channel mode, vector width).  Tensors
 * with n == 0 are accepted and skipped.  codes, y and the parameter arrays
 * (device memory) must stay valid while the plan is in use; mctq_unpack_multi enqueues the launches on `stream`. */
#define MCTQ_PACK_AFFINE_I8 1 /* one byte per element, int8 if is_signed else uint8 */
#define MCTQ_PACK_AFFINE_I4 2 /* two per byte, element 2j in the low nibble (the MCTQ_CODES_INT4 layout) */
#define MCTQ_PACK_LUT_U8 3    /* one LUT index per byte, K <= 256 */
#define MCTQ_PACK_LUT_I4 4    /* two LUT indices per byte, K <= 16 */
typedef struct MctqPackedDesc {
    const void* codes;
    void* y;
    int64_t n, C, inner;
    int32_t kind, is_signed, y_dtype, K;
    const float* scale;         /* affine: scale[C];   LUT: thr[C] */
    const int32_t* zp;          /* affine: zp[C];      LUT: NULL */
    const float* lut_quotients; /* LUT: K entries;     affine: NULL */
} MctqPackedDesc;
size_t mctq_unpack_plan_bytes(const MctqPackedDesc* descs_host, int n_desc);     /* 0: some tensor is not plannable */
int64_t mctq_unpack_plan(const MctqPackedDesc* descs_host, int n_desc, void* plan_host_out, size_t plan_bytes);
int mctq_unpack_multi(const void* plan_host, void* stream);

/* Fused packed linear: y[M][out] = x[M][in] @ W^T + bias, reading the packed codes of W directly (W is never built in memory).
 * Replaces the pair  mctq_unpack_multi(W) -> F.linear(x, W, bias)  of a packed nn.Linear wrapper's forward at small M, where
 * the product is bound by the bytes of W: the codes are read once instead of being expanded to a float W in HBM and read back.
 *   w          HOST descriptor of the packed weight, row-major [out][in]: n = out * in, C = 1 (per tensor) or C = out with
 *              inner = in (per output row); w->y is unused.  Any kind; codes at any alignment (any `in`, int4 rows may start
 *              in a high nibble)
 *   x, y       device, M rows of x_dtype, contiguous; x_dtype must equal w->y_dtype (the rebuilt weight's dtype, f32 for LUT)
 *   bias       device, out entries of x_dtype, or NULL
 * W means exactly the weight mctq_unpack_multi rebuilds.  Accumulation is in f32 (a per-row scale or threshold may be applied
 * once per row for f32 outputs), y is rounded once to x_dtype, and the summation order is fixed: two calls on the same inputs
 * give the same bits.  Not bit-identical to a cuBLAS product.  Envelope of the per-row factoring: for f32 affine weights the
 * row sum is sum_k x_k * (q_k - zp_c), scaled afterwards, so the result is "W is exactly the rebuilt weight" (within the error
 * of f32 accumulation) only while every partial sum of x * (q - zp) stays below FLT_MAX; max|x| * max|q - zp| * in_features
 * < FLT_MAX suffices (|q - zp| <= 255: max|x| < 1.3e36 / in_features).  Beyond it the result may be +-inf or NaN where
 * x @ W^T is finite.  Nothing checks this (a host-side check would need a synchronisation).
 * M == 0 is a no-op.  Returns MCTQ_E_BADARG (shape, null or
 * parameter-layout errors), MCTQ_E_DTYPE, MCTQ_E_LUT (K outside 1..16 / 1..256) before any CUDA call. */
int mctq_packed_linear(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x, int x_dtype,
                       int64_t M, const void* bias, void* y, void* stream);

/* Batched packed linear: the product of mctq_packed_linear on the tensor cores (tcgen05.mma), for the row counts of batched
 * decode and short prefills (tens to hundreds of rows), where the CUDA-core kernel's time grows with M.  Same descriptor,
 * arguments and checks as mctq_packed_linear, plus
 *   lut_quotients_host  LUT kinds: a HOST copy of the w->K quotients of w->lut_quotients (affine kinds: ignored, may be NULL).
 *                       The kernel takes the quotients from it (by value); MCTQ_E_LUT when one is not exact in bf16.
 * Contract: every operand the tensor cores multiply is exact -- the bf16 / f16 rebuilt weight itself; for f32 weights
 * q - zp (needs |q - zp| <= 256, which packed weights satisfy) or the LUT quotient, with the per-row scale / threshold
 * applied once per row after the sum (the factoring and the envelope of mctq_packed_linear); for f32 x, three bf16 terms
 * x0 + x1 + x2 = x (exact for finite x; inf / NaN x enter as x0 alone, so a non-finite x gives the exact product's inf / NaN).
 * Products are accumulated in f32 by the tensor cores and rounded once to x_dtype after the scale and the bias.
 * Error bound (the tests enforce it): |y - y_exact| <= 2^-22 * (in_features / 16 + 8) * sum_k |x_k * W_jk| + u_T * |y_exact|
 * + 2^-126 * sum_k |W_jk| (+ the output dtype's subnormal grain), u_T the unit roundoff of x_dtype.  The first term covers
 * the f32 accumulation of the tensor cores (16 products per step, alignment that may truncate: a few units of 2^-24 per step)
 * and the epilogue roundings; the third the f32 x below the normal range, whose low split terms bf16 cannot hold.  On data
 * whose products and partial sums are exact in f32 the result is exact (the tests check this bit for bit).
 * Deterministic: the split of the row length over the CTAs of a cluster and the order of the partial sums are fixed by the
 * shape, so two calls on the same inputs give the same bits.  M == 0 is a no-op.  Returns MCTQ_E_BADARG, MCTQ_E_DTYPE,
 * MCTQ_E_LUT before any CUDA call. */
int mctq_packed_linear_batched(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x, int x_dtype,
                               int64_t M, const void* bias, void* y, const float* lut_quotients_host, void* stream);

/* Integer linear mode (packed nn.Linear wrappers whose input comes from a per-tensor 8-bit affine activation quantizer Q).
 * Both operands of the product are integer codes: x = sx * (qx - zx), W = sw[o] * (qw - zw[o]).
 *
 * mctq_quantize_rows_i8: qx [M][K] (row-major, one byte per element: int8 if qmin < 0 else uint8) of x [M][K] (x_dtype,
 * row-major), by the recipe of mctq_fq_affine_scalar with code_mode MCTQ_CODES_INT8 -- the same codes bit for bit, NaN -> qmin,
 * +-inf clamped -- and, when rowsum is not NULL, Sx[n] = sum_k qx[n,k] (int32).  scale is Q's scale narrowed to f32.
 * MCTQ_E_BADARG (null x / codes, M < 0, K < 1), MCTQ_E_DTYPE, MCTQ_E_RANGE (qmin > qmax or a range that does not fit 8-bit
 * codes) before any CUDA call; M == 0 is a no-op.
 *
 * mctq_packed_linear_i8: y[n, o] for n < M, o < out_features, rows of y ldy elements apart (ldy >= out_features; nothing else
 * of y is written), computed as
 *   acc = sum_k qx[n,k] * qw[o,k]                                  int32, exact (tcgen05.mma kind::i8)
 *   c   = acc - zw[o] * Sx[n] - zx * Sw[o] + K * zx * zw[o]       int64, exact;  Sx / Sw: row sums of the codes
 *   y   = T(fl(fl((float)c * f[o]) + bias[o]))                     T = y_dtype; f[o] = fl32(sx * sw[o]) supplied by the caller
 *   w          HOST descriptor of an MCTQ_PACK_AFFINE_I8 / _I4 weight [out][in], per tensor or per output row (as for
 *              mctq_packed_linear); w->y_dtype == y_dtype; codes 16-byte aligned; w->scale is not read (f replaces it)
 *   x_codes    device qx [M][in_features], 16-byte aligned; x_signed: int8 (1) or uint8 (0) codes; x_zero_point = zx
 *   x_rowsum   device Sx [M], or NULL when every weight zero point is 0 (the term is then skipped)
 *   w_rowsum   device Sw [out_features] (int32), needed when zx != 0
 *   factor     device f [C] (C = w->C); bias: device [out_features] of y_dtype, or NULL
 * Every output bit is fixed by the formula: the result does not depend on the split of the row length or the tiling, and
 * two calls give the same bits.  Returns, before any CUDA call: MCTQ_E_BADARG for a LUT kind, a null pointer, a shape or
 * layout error, in_features not a multiple of 16 (32 for int4 weights), ldy < out_features or unaligned codes;
 * MCTQ_E_DTYPE; MCTQ_E_RANGE for a zx outside the x codes' range or in_features above
 * mctq_packed_linear_i8_max_k(w->is_signed, x_signed) (the largest K whose int32 sum cannot overflow: 33025 for uint8 x
 * uint8, 65793 for one signed operand, 131071 for int8 x int8).  M == 0 is a no-op. */
int mctq_quantize_rows_i8(const void* x, int x_dtype, int64_t M, int64_t K, float scale, int32_t zp, int32_t qmin,
                          int32_t qmax, void* codes, int32_t* rowsum, void* stream);
int64_t mctq_packed_linear_i8_max_k(int w_signed, int x_signed);
int mctq_packed_linear_i8(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x_codes,
                          int x_signed, int32_t x_zero_point, int64_t M, const int32_t* x_rowsum, const int32_t* w_rowsum,
                          const float* factor, const void* bias, int y_dtype, void* y, int64_t ldy, void* stream);

/* Integer convolution mode (packed nn.Conv2d wrappers, groups 1, zero padding, fed by the same quantizer Q as above).
 *
 * mctq_quantize_nhwc_i8: qx [N][H*W][C] (NHWC, one byte per element, int8 if qmin < 0 else uint8) of an NCHW-contiguous
 * x [N][C][H][W] (x_dtype), codes bit for bit those of mctq_quantize_rows_i8 / mctq_fq_affine_scalar, and, when P is not
 * NULL, P[(b*H + h)*W + w] = sum_c qx (int32).  A channels_last x needs no transpose: mctq_quantize_rows_i8 with M = N*H*W
 * rows of K = C codes writes the same codes, and its row sums are P.  MCTQ_E_BADARG (null x / codes, N < 0, C / H / W < 1),
 * MCTQ_E_DTYPE, MCTQ_E_RANGE as mctq_quantize_rows_i8, before any CUDA call; N == 0 is a no-op.
 *
 * mctq_packed_conv2d_i8: y = conv2d(x, W) in the integer arithmetic of mctq_packed_linear_i8, with
 *   qx[b,c,h,w] = Q's codes of x;  zx for (h, w) outside the image (zero padding of Q(x) is exactly code zx)
 *   row n = (b, ho, wo), column k = (r, s, c),  K = Cin*kh*kw,  M = N*Ho*Wo
 *   X[n,k] = qx[b, c, ho*sh - pt + r*dh, wo*sw - pl + s*dw]
 *   acc    = sum_k X[n,k] * qw[o,k]                               int32, exact (tcgen05.mma kind::i8)
 *   c      = acc - zw[o] * Sx[n] - zx * Sw[o] + K * zx * zw[o]    int64, exact;  Sx[n] = sum_k X[n,k] (padding counts as zx)
 *   y[b,o,ho,wo] = T(fl(fl((float)c * f[o]) + bias[o]))          T = y_dtype; f[o] = fl32(sx * sw[o])
 * Padded taps hold zx and so contribute exactly 0, as in the float model; the sum is exact, so the output does not depend on
 * the order of k, the tiling or the split of K.
 *   w          HOST descriptor of an MCTQ_PACK_AFFINE_I8 / _I4 weight [Cout][K] in (r, s, c) order (the memory order of a
 *              channels_last [Cout, Cin, kh, kw] weight), per tensor or per output channel; codes 16-byte aligned
 *   g          the geometry; Ho / Wo are the caller's (taps outside the image are never read, whatever they are)
 *   x_codes    device NHWC codes [N][H][W][Cin], 16-byte aligned; x_signed, x_zero_point as for mctq_packed_linear_i8
 *   x_rowsum   device Sx [M], or NULL when every weight zero point is 0
 *   w_rowsum, factor, bias   as for mctq_packed_linear_i8 (Cout entries)
 *   y_nchw     0: y is [M][Cout] row-major (NHWC / channels_last);  1: y is NCHW, y[(b*Cout + o)*Ho*Wo + ho*Wo + wo]
 * Returns, before any CUDA call: MCTQ_E_BADARG for a LUT kind, a null pointer, a non-positive extent, stride or dilation, a
 * negative pad, Cin not a multiple of 16, K not a multiple of 32 for int4 weights, unaligned codes, M >= 2^31, or zx != 0
 * without w_rowsum; MCTQ_E_DTYPE; MCTQ_E_RANGE for a zx outside the x codes' range or K above
 * mctq_packed_linear_i8_max_k(w->is_signed, x_signed).  M == 0 is a no-op. */
typedef struct MctqConv2dGeom {
    int32_t N, H, W, Cin;           /* input [N][H][W][Cin] */
    int32_t Ho, Wo;                 /* output extent */
    int32_t kh, kw;
    int32_t sh, sw, dh, dw;         /* stride, dilation */
    int32_t pt, pb, pl, pr;         /* zero padding per side */
} MctqConv2dGeom;
int mctq_quantize_nhwc_i8(const void* x, int x_dtype, int64_t N, int64_t C, int64_t H, int64_t W, float scale, int32_t zp,
                          int32_t qmin, int32_t qmax, void* codes, int32_t* P, void* stream);
int mctq_packed_conv2d_i8(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cout, const void* x_codes, int x_signed,
                          int32_t x_zero_point, const int32_t* x_rowsum, const int32_t* w_rowsum, const float* factor,
                          const void* bias, int y_dtype, void* y, int y_nchw, void* stream);

/* Integer linear and convolution modes for LUT weights.  A LUT weight rebuilds as W[o,k] = fl32(q[idx[o,k]] * thr[o]) with
 * q_k = lut_k / 2^(bw-1) and integer centroids lut_k in [-128, 127]: an int8 code lut_k times sw[o] = fl32(thr[o]) * 2^-(bw-1)
 * (exact in f32 for the weights the wrappers switch), an affine weight with zero point 0.  The formula of
 * mctq_packed_linear_i8 / mctq_packed_conv2d_i8 then reads
 *   qw[o,k] = lut[idx[o,k]]   int8;   zw = 0;   Sw[o] = sum_k qw[o,k];   f[o] = fl32(sx * sw[o])
 *   acc = sum_k qx[n,k] * lut[idx[o,k]]                              int32, exact (tcgen05.mma kind::i8)
 *   c   = acc - zx * Sw[o]                                           int64, exact
 *   y   = T(fl(fl((float)c * f[o]) + bias[o]))                       T = f32 (LUT weights rebuild as f32)
 * Every output bit is fixed by the formula; it does not depend on the tiling, the split of K or the conv's order of k.
 * The arguments are those of mctq_packed_linear_i8 / mctq_packed_conv2d_i8, with:
 *   w              HOST descriptor of an MCTQ_PACK_LUT_I4 / _U8 weight (indices, K = w->K table entries, f32, its
 *                  quotients present but not read; w->scale is not read, f replaces it)
 *   x_rowsum       unused (zw = 0)
 *   lut_codes_host HOST array of w->K int8 centroid codes lut[0 .. K-1]; it travels by value in the kernel arguments, so a
 *                  call (and a CUDA-graph capture of it) needs no device copy of the table and no synchronisation
 * The index → code lookup happens in the GEMM's weight producers: 4-bit indices by byte permutations of the 16-byte table
 * held in registers, 8-bit indices through a shared-memory table.  Returns, before any CUDA call: MCTQ_E_BADARG for an
 * affine kind, a null table and the other argument errors of the affine entry points (in_features / K a multiple of 32 for
 * 4-bit and of 16 for 8-bit indices); MCTQ_E_DTYPE; MCTQ_E_LUT for K outside 1..16 (4-bit) / 1..256 (8-bit);
 * MCTQ_E_RANGE for a zx outside the x codes' range or a row length above mctq_packed_linear_i8_max_k(1, x_signed). */
int mctq_packed_linear_i8_lut(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, const void* x_codes,
                              int x_signed, int32_t x_zero_point, int64_t M, const int32_t* x_rowsum, const int32_t* w_rowsum,
                              const float* factor, const void* bias, int y_dtype, void* y, int64_t ldy,
                              const int8_t* lut_codes_host, void* stream);
int mctq_packed_conv2d_i8_lut(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cout, const void* x_codes,
                              int x_signed, int32_t x_zero_point, const int32_t* x_rowsum, const int32_t* w_rowsum,
                              const float* factor, const void* bias, int y_dtype, void* y, int y_nchw,
                              const int8_t* lut_codes_host, void* stream);

/* Integer convolution mode for depthwise Conv2d (groups == Cin, any channel multiplier; DESIGN.md §7e).  The formula of
 * mctq_packed_conv2d_i8 with one input channel per group, in its centred form:
 *   m = Cout / Cin (channel multiplier); output channel o reads input channel c(o) = o / m;  K = kh * kw
 *   qx[b,c,h,w]  = Q's codes of x: the recipe of mctq_quantize_rows_i8, bit for bit the codes mctq_fq_affine_scalar emits
 *                  (NaN -> qmin, +-inf clamped);  zx outside the image
 *   c[b,o,ho,wo] = sum_{r,s} (qx[b, c(o), ho*sh - pt + r*dh, wo*sw - pl + s*dw] - zx) * (qw[o,r,s] - zw[o])
 *                  int32, exact for K <= 33025 (each factor has magnitude <= 255); padded taps contribute exactly 0
 *   y[b,o,ho,wo] = T(fl(fl((float)c * f[o]) + bias[o])),  f[o] = fl32(sx_f32 * sw[o]),  T = the rebuilt weight's dtype
 *   LUT weights: qw = lut[idx] (int8), zw = 0, sw = thr * 2^-(bw-1), T = f32 (as for mctq_packed_conv2d_i8_lut)
 * c is the integer acc - zw Sx - zx Sw + K zx zw of mctq_packed_conv2d_i8, so the output does not depend on the order of
 * the taps or the tiling.  The kernel reads the float x once and computes Q's codes in registers: no code tensor, no Sx.
 *   w          HOST descriptor of an MCTQ_PACK_AFFINE_I8 / _I4 / LUT_I4 / LUT_U8 weight [Cout][kh*kw] (the memory order of a
 *              contiguous or channels_last [Cout, 1, kh, kw] weight), per tensor or per output channel (inner = kh*kw);
 *              w->y_dtype == x_dtype; w->scale is not read (factor replaces it); codes at any alignment
 *   g          the geometry (g->Cin = C, x's channels); Ho / Wo are the caller's (taps outside the image are never read)
 *   x          device x [N][C][H][W] (x_nhwc = 0, NCHW-contiguous) or [N][H][W][C] (x_nhwc = 1, channels_last), x_dtype;
 *              y [N][Cout][Ho][Wo] in the same layout and dtype
 *   x_scale, x_zero_point, x_qmin, x_qmax   Q (scale narrowed to f32), as for mctq_quantize_rows_i8
 *   factor     device f [1 or Cout];  bias: device [Cout] of x_dtype, or NULL
 *   lut_codes_host   LUT kinds: HOST array of w->K int8 centroid codes (by value in the kernel arguments); NULL otherwise
 * No host-device copy and no synchronisation: CUDA-graph capture works.  Returns, before any CUDA call: MCTQ_E_BADARG for
 * a null pointer, a non-positive extent, stride or dilation, a negative pad, x_nhwc not 0 / 1, Cout not a multiple of Cin,
 * w->n != Cout*kh*kw, a bad parameter layout, or a table present / absent against the kind; MCTQ_E_DTYPE; MCTQ_E_RANGE for
 * a range that does not fit 8-bit codes, zx outside it, kh*kw > 33025, or a dilated window too wide for shared memory even
 * for one output of one channel; MCTQ_E_LUT.  N == 0 is a no-op. */
int mctq_packed_dwconv2d_i8(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cout, const void* x, int x_dtype,
                            int x_nhwc, float x_scale, int32_t x_zero_point, int32_t x_qmin, int32_t x_qmax,
                            const float* factor, const void* bias, void* y, const int8_t* lut_codes_host, void* stream);

/* The tile plan mctq_packed_dwconv2d_i8 launches for a geometry (host only, no CUDA call).  A work unit is S slots (NCHW:
 * consecutive (b, c) planes; NHWC: consecutive channels of one image) times a TH x TW tile of output pixels, staged from an
 * IH x IW window tile in smem_bytes of shared memory.  The planner starts from about 2048 outputs per unit and halves TH,
 * then S, then TW until the tile fits 200 KB.  Returns 0, MCTQ_E_BADARG for the launch's geometry rejections or a null
 * `out`, or MCTQ_E_RANGE for kh*kw > 33025 or a dilated window that does not fit even at S = TH = TW = 1 (20 + 4 kh kw +
 * 4 IH IW bytes, IH = (kh-1) dh + 1, IW = (kw-1) dw + 1): the launch returns the same.  `out` is written only on 0. */
typedef struct MctqDwPlan {
    int32_t S, TH, TW, IH, IW, smem_bytes;
} MctqDwPlan;
int mctq_packed_dwconv2d_i8_plan(const MctqConv2dGeom* g, int64_t Cout, int x_nhwc, MctqDwPlan* out);

/* Integer modes for row lengths and channel counts off the GEMM's granule (DESIGN.md §7f).  The padding contract: every
 * column the kernel sums beyond the real K belongs to one of two classes --
 *   channel pad  the x code is zx (in the image and, as before, for taps outside it); the column is counted in K, Sx and
 *                Sw; its weight code may be anything (a LUT table needs no zero centroid)
 *   row tail     the x code is 0 and the column is counted in none of K, Sx and Sw (the GEMM's "columns >= K are zero")
 * A channel pad contributes (zx - zx) * (qw - zw) = 0 to the centred sum, so c, and every output bit, is the formula of
 * mctq_packed_linear_i8 / mctq_packed_conv2d_i8 / their LUT forms over the real row.
 *
 * mctq_quantize_rows_i8_padded: mctq_quantize_rows_i8 writing qx [M][ldc] (ldc >= K, ldc % 4 == 0, codes 4-byte aligned),
 * columns [K, ldc) holding zp; Sx[n] includes them.  MCTQ_E_BADARG also for ldc < K or ldc % 4 != 0, MCTQ_E_RANGE for zp
 * outside [qmin, qmax].
 * mctq_quantize_nhwc_i8_padded: mctq_quantize_nhwc_i8 writing qx [N][H*W][Cp] (Cp = 4, 8 or a multiple of 16, Cp >= C, codes
 * 16-byte aligned), channels [C, Cp) holding zp; P includes them.  One pixel per thread, whole 4 / 8 / 16-byte stores.
 * MCTQ_E_BADARG also for a Cp outside that set, MCTQ_E_RANGE for zp outside [qmin, qmax].
 *
 * mctq_packed_linear_i8_padded: mctq_packed_linear_i8 (lut_codes_host NULL) or mctq_packed_linear_i8_lut (a table) over
 * x codes [M][ldc] whose columns [in_features, ldc) are channel pads: w is the [out][ldc] weight, Sw sums its ldc columns,
 * and the correction counts K = ldc.  MCTQ_E_BADARG also for in_features < 1, ldc < in_features, ldc not a multiple of 16
 * (32 for 4-bit codes) or a table present / absent against the kind; MCTQ_E_RANGE for ldc above the int32 bound.
 * mctq_packed_conv2d_i8_padded: mctq_packed_conv2d_i8 / _lut over NHWC codes [N][H][W][Cp] whose channels [g->Cin, Cp) are
 * channel pads (g->Cin is the real channel count).  Sx counts Cp * zx for a tap outside the image.
 *   Cp % 16 == 0   w is [Cout][kh*kw*Cp] in (r, s, c) order, c < Cp; K = kh*kw*Cp (a multiple of 32 for 4-bit codes)
 *   Cp = 4 / 8     the narrow gather: w is [Cout][K] with K = kh*kw*Cp rounded up to 16 (32 for 4-bit codes); its first
 *                  kh*kw*Cp columns are (r, s, c) with c < Cp, the rest a row tail; the correction counts kh*kw*Cp
 * Sw[o] sums the counted columns.  MCTQ_E_BADARG also for Cp < g->Cin or Cp outside {4, 8, 16, 32, ...}; every other
 * return as for mctq_packed_conv2d_i8, the int32 bound applying to the kernel's row length K. */
int mctq_quantize_rows_i8_padded(const void* x, int x_dtype, int64_t M, int64_t K, int64_t ldc, float scale, int32_t zp,
                                 int32_t qmin, int32_t qmax, void* codes, int32_t* rowsum, void* stream);
int mctq_quantize_nhwc_i8_padded(const void* x, int x_dtype, int64_t N, int64_t C, int64_t H, int64_t W, int64_t Cp,
                                 float scale, int32_t zp, int32_t qmin, int32_t qmax, void* codes, int32_t* P, void* stream);
int mctq_packed_linear_i8_padded(const MctqPackedDesc* w, int64_t out_features, int64_t in_features, int64_t ldc,
                                 const void* x_codes, int x_signed, int32_t x_zero_point, int64_t M, const int32_t* x_rowsum,
                                 const int32_t* w_rowsum, const float* factor, const void* bias, int y_dtype, void* y,
                                 int64_t ldy, const int8_t* lut_codes_host, void* stream);
int mctq_packed_conv2d_i8_padded(const MctqPackedDesc* w, const MctqConv2dGeom* g, int64_t Cp, int64_t Cout,
                                 const void* x_codes, int x_signed, int32_t x_zero_point, const int32_t* x_rowsum,
                                 const int32_t* w_rowsum, const float* factor, const void* bias, int y_dtype, void* y,
                                 int y_nchw, const int8_t* lut_codes_host, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Whole-model weight quantisation: one launch over a table of tensors (SURVEY 8f rank 1).
 * Replaces the per-layer loop  for name, w, quantizer in self._weights_vars: quantizer(w)
 *   (mct_quantizers/pytorch/quantize_wrapper.py:228-240 and :260-270) for affine weight quantizers.
 * `descs` and `tile_starts` live in DEVICE memory (the caller uploads them once; weights do not move).
 * tile_starts has n_desc + 1 entries: tile_starts[k] = first tile of tensor k, in units of
 * mctq_multi_tile_elems(dtype) elements; mctq_multi_plan fills it on the host.
 */
typedef struct MctqTensorDesc {
    const void* x;
    void* y;
    void* codes; /* or NULL */
    const float* scale;
    const int32_t* zp;
    int64_t n;
    int64_t C;
    int64_t inner;
    int32_t qmin;
    int32_t qmax;
    int32_t dtype;
    int32_t code_mode;
} MctqTensorDesc;

int64_t mctq_multi_tile_elems(void);
/* host helper: fills tile_starts[0..n_desc] from descs[k].n (both HOST arrays); returns total tiles or <0 */
int64_t mctq_multi_plan(const MctqTensorDesc* descs_host, int n_desc, int32_t* tile_starts_host);
int mctq_fq_affine_multi(const MctqTensorDesc* descs_dev, const int32_t* tile_starts_dev, int n_desc,
                         int64_t total_tiles, void* stream);

/* Many per-tensor (scalar-parameter) sites in ONE launch: the activation holders of a model whose inputs already exist
 * (calibration / analysis passes, batched serving of independent tensors).
 * Replaces: a loop of PytorchActivationQuantizationHolder.forward calls, each one
 *           torch.fake_quantize_per_tensor_affine(x, scale: float, zero_point: int, quant_min, quant_max)
 *           (mct_quantizers/pytorch/activation_quantization_holder.py:43-53 ->
 *            activation_symmetric_inferable_quantizer.py:113-117 / activation_uniform_inferable_quantizer.py:124-128).
 * `sites` is a HOST array (it travels as kernel parameters, 64 sites per launch); x / y are device pointers, 16-byte
 * aligned, y has x's dtype; arithmetic identical to mctq_fq_affine_scalar.  Sites with n == 0 are skipped. */
typedef struct MctqSiteDesc {
    const void* x;
    void* y;
    int64_t n;
    int32_t dtype;
    float scale;
    int32_t zp;
    int32_t qmin;
    int32_t qmax;
    int32_t reserved;
} MctqSiteDesc;
int mctq_fq_affine_scalar_multi(const MctqSiteDesc* sites_host, int n_sites, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * LUT (nearest-centroid) fake-quant.
 * Replaces: lut_quantizer(...)  mct_quantizers/pytorch/quantizer_utils.py:95-139 (which calls
 *           int_quantization_with_threshold :142-170) as used by
 *           weights_lut_symmetric_inferable_quantizer.py:114-122, weights_lut_pot_inferable_quantizer.py:74-104,
 *           activation_lut_pot_inferable_quantizer.py:86-91.
 *
 * The centroid list is first compiled (on the host, once per quantizer) into a search table: sorted
 * unique centroids, the exact f32 decision threshold between each adjacent pair under torch.argmin's
 * first-minimum rule, and the original index of every sorted entry.  The table is a POD blob of
 * mctq_lut_table_bytes(K) bytes that the caller copies to the device; K (the length of the original
 * centroid list, <= 256) travels with it because the blob's geometry is a function of K alone.
 */
size_t mctq_lut_table_bytes(int K);
int mctq_lut_build_table(const float* lut_host, int K, int lut_values_bitwidth, int is_signed,
                         void* table_host_out, size_t table_bytes);

/* weights flavour: thr is a DEVICE f32 array [C]; d_c = thr_c + (float)eps (f32 add), no intermediate
 * rounding, f32 output.  idx (optional) receives the LUT index per element (MCTQ_CODES_INT8: one byte,
 * MCTQ_CODES_INT4: packed nibbles, K <= 16). */
int mctq_fq_lut(const void* x, float* y, void* idx, int64_t n, int x_dtype,
                const void* table_dev, int K, const float* thr, int64_t C, int64_t inner, int64_t elem_offset,
                float eps, int idx_mode, void* stream);

/* activation flavour: threshold and eps are Python floats in the reference, so the divisor is
 * d = (float)(thr + eps) computed in double by the caller and passed by value with thr_f32 = (float)thr;
 * for bf16/f16 inputs the reference's eager ops round the normalised value back to the input dtype
 * before the search (round_to_x_dtype = 1). */
#define MCTQ_LUT_DIVISOR_IS_MULTIPLIER 2   /* OR into round_to_x_dtype: `divisor` is r = (float)(1.0 / (thr + eps)) and the
                                            * normalisation is x * r -- what libtorch's CUDA kernel for `tensor / python_number`
                                            * computes, i.e. what the unmodified reference yields for CUDA tensors (it differs from
                                            * the CPU kernel's true division at rounding ties).  mctq_lut_prepare: scalar_mode = 2 */
int mctq_fq_lut_scalar(const void* x, float* y, void* idx, int64_t n, int x_dtype,
                       const void* table_dev, int K, float divisor, float thr_f32, int round_to_x_dtype,
                       int idx_mode, void* stream);

/* Prepared flavour (the fast path): per-channel decision tables in the x domain.
 * Normalise -> clip -> argmin is a monotone function of x for each channel, so the LUT entry is decided by which of the
 * K - 1 per-channel thresholds X[c][j] the element exceeds.  mctq_lut_prepare computes them exactly (bisection over f32
 * bit patterns through the reference arithmetic: IEEE division by thr + eps, optional rounding to the activation dtype,
 * first-minimum thresholds of the search table) together with the dequantised outputs (lut / 2^(bw - s)) * thr_c, once per
 * quantizer; mctq_fq_lut_prepared then runs without any division or search loop.  Same reference call sites as above.
 *   table_host        the HOST copy of the blob from mctq_lut_build_table
 *   thr_dev           DEVICE f32 [C] (weights flavour) or NULL with scalar_mode = 1 (divisor / thr_f32 by value, C = 1)
 *   round_dtype       0 none; 1 / 2: the normalised value is rounded to bf16 / f16 first (activation flavour)
 *   prepared_dev      DEVICE buffer of mctq_lut_prepared_bytes(K, bw, signed, C) bytes (0 = configuration unsupported)
 * Grids of more than 10 bits use a cell table coarser than the integer grid; mctq_lut_prepare returns MCTQ_E_RANGE when the
 * centroid list is too dense for it (two decision thresholds in one cell): use the generic entry points then.
 * mctq_lut_prepare is one-off setup and synchronises `stream` once.  mctq_fq_lut_prepared needs 16-byte aligned x / y and
 * returns MCTQ_E_RANGE when the channel window of a tile does not fit in shared memory (rows shorter than ~16
 * elements with large K): callers fall back to mctq_fq_lut. */
size_t mctq_lut_prepared_bytes(int K, int lut_values_bitwidth, int is_signed, int64_t C);
int mctq_lut_prepare(const void* table_host, int K, const float* thr_dev, int64_t C, float eps, int scalar_mode,
                     float divisor, float thr_f32, int round_dtype, void* prepared_dev, size_t prepared_bytes,
                     void* stream);
int mctq_fq_lut_prepared(const void* x, float* y, void* idx, int64_t n, int x_dtype, const void* prepared_dev, int K,
                         int lut_values_bitwidth, int is_signed, int64_t C, int64_t inner, int64_t elem_offset,
                         int idx_mode, void* stream);

/* Whole-model LUT weight quantization in ONE launch (the LUT counterpart of mctq_fq_affine_multi; replaces the per-layer
 * loop mct_quantizers/pytorch/quantize_wrapper.py:228-240 over weights_lut_symmetric_inferable_quantizer.py:89-128 /
 * weights_lut_pot_inferable_quantizer.py:74-104 calls).  Every tensor brings its own prepared blob (mctq_lut_prepare).
 * mctq_lut_multi_plan compiles the HOST descriptor array into an opaque plan blob of
 * mctq_lut_multi_plan_bytes(descs, n_desc) bytes in HOST memory (returns the number of CTAs of the launch, or < 0:
 * MCTQ_E_RANGE / MCTQ_E_BADARG mean "this tensor needs the single-tensor / generic entry point").  Tensors are grouped by
 * the plan grouping rule (Conventions above); the kernel variant is (dtype, channel mode, vector width, record kind), so a
 * model whose LUT weights share one layout and similar sizes is one launch per 64 tensors.
 * x, y and the prepared blobs must stay valid while the plan is in use. */
typedef struct MctqLutTensorDesc {
    const void* x;            /* device, dtype below, 16-byte aligned */
    float* y;                 /* device f32, 16-byte aligned */
    const void* prepared_dev; /* mctq_lut_prepare blob of this tensor's quantizer */
    int64_t n;
    int64_t C;
    int64_t inner;
    int32_t dtype;
    int32_t K;
    int32_t lut_values_bitwidth;
    int32_t is_signed;
} MctqLutTensorDesc;
size_t mctq_lut_multi_plan_bytes(const MctqLutTensorDesc* descs_host, int n_desc);   /* 0: some tensor is not plannable */
int64_t mctq_lut_multi_plan(const MctqLutTensorDesc* descs_host, int n_desc, void* plan_host_out, size_t plan_bytes);
int mctq_fq_lut_prepared_multi(const void* plan_host, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Host-buffer entry points: the same operators for tensors that live in HOST memory (pinned memory
 * overlaps; pageable memory works but serialises).  The data is streamed through `staging_dev`
 * (device scratch owned by the caller, >= mctq_host_staging_min_bytes() = 304 MiB) in chunks on three internal streams:
 * H2D copy, kernel and D2H copy of neighbouring chunks overlap.  Parameters are HOST arrays (copied
 * before the call returns; at most 384 Ki channels).  By default these calls return after y_host is
 * complete (they synchronise their internal streams only).
 * They are what a CPU-tensor call of a quantizer maps to: the product has no CPU arithmetic path.
 *
 * Deferred mode (mctq_host_set_deferred(device, 1)): the calls return as soon as their copies and kernels
 * are enqueued, so the three-stage pipeline keeps running across the tensors of a model instead of
 * filling and draining once per tensor; x_host must stay valid and y_host is complete only after
 * mctq_host_wait(device) (or after deferred mode is switched off, which waits as well).
 */
size_t mctq_host_staging_min_bytes(void);
int mctq_fq_affine_host(const void* x_host, void* y_host, int64_t n, int x_dtype,
                        const float* scale_host, const int32_t* zp_host, int64_t C, int64_t inner,
                        int32_t qmin, int32_t qmax, void* staging_dev, size_t staging_bytes, int device);
int mctq_host_set_deferred(int device, int on);
int mctq_host_wait(int device);
int mctq_fq_lut_host(const void* x_host, float* y_host, int64_t n, int x_dtype,
                     const void* table_host, int K, const float* thr_host, int64_t C, int64_t inner,
                     float eps, int scalar_mode, float divisor, float thr_f32, int round_to_x_dtype,
                     void* staging_dev, size_t staging_bytes, int device);

/* ------------------------------------------------------------------------------------------------------
 * Introspection / test hooks (no reference counterpart).
 */
/* launches of this library's kernels since load (what bench.py reports as gpu_launches) */
int64_t mctq_launch_count(void);
/* process-wide switches.  key 3 = programmatic dependent launch: 0 off, 1 wait-then-load (default),
 *   2 = load-then-wait for launches whose input is not an output of a launch of this library still in flight on the stream,
 *   3 = additionally no wait at all (until a CTA's last instruction) for launches whose buffers are disjoint from those of
 *   every launch still in flight (at most three launches in flight together, then a waiting one) -- 2 and 3 are only
 *   legal while the stream carries NO work of other libraries (their kernels may release dependents before their stores
 *   are visible; the allocator may recycle their buffers); opt-in, see
 *   mct_quantizers_b200.private_stream(); changing the key makes the next launch on every stream a waiting one,
 * key 9 = NVTX ranges (nvtx3, header-only) around every compute entry point, named after the entry point (default 0;
 *   `ncu --nvtx` and timeline tools then attribute kernels to the call of the reference's API they belong to);
 * every other key is rejected with MCTQ_E_BADARG.  Returns the previous value or <0 */
int mctq_set_tuning(int key, int value);
/* device self-test of the 5-op correctly-rounded division used by the LUT kernels against __fdiv_rn
 * on n_pairs pseudo-random (x, d) pairs; *mismatches_dev (device int64) receives the number that differ */
int mctq_selftest_division(int64_t n_pairs, uint64_t seed, int64_t* mismatches_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MCTQ_H_ */
