"""torch.library operators of the `mctq` namespace: the boundary between the quantizer objects and the
sm_100a kernels.

    torch.ops.mctq.fq_affine_scalar   <- torch.fake_quantize_per_tensor_affine(x, float, int, qmin, qmax)
    torch.ops.mctq.fq_affine_tensor   <- torch.fake_quantize_per_tensor_affine(x, Tensor[1], Tensor[1], qmin, qmax)
    torch.ops.mctq.fq_affine_channel  <- torch.fake_quantize_per_channel_affine(x, scale, zp, axis, qmin, qmax)
    torch.ops.mctq.fq_lut_tensor      <- lut_quantizer(..., threshold=Tensor, per_channel, channel_axis, input_rank)
    torch.ops.mctq.fq_lut_scalar      <- lut_quantizer(..., threshold=float)            (activations)
    torch.ops.mctq.quantize_affine_*  -> integer codes (+ optional fake-quant values); mctq.dequantize_affine
    torch.ops.mctq.lut_indices        -> LUT indices;                                    mctq.dequantize_lut
    torch.ops.mctq.packed_linear      <- F.linear(x, <weight rebuilt from packed codes>, bias)   (small row counts)
    torch.ops.mctq.packed_linear_batched   the same product on the tensor cores                  (batched row counts)
    torch.ops.mctq.quantize_rows_i8   -> 8-bit codes of x (fq_affine_scalar's codes) and their row sums
    torch.ops.mctq.packed_linear_i8   <- the integer product of those codes and packed int8 / int4 weight codes
    torch.ops.mctq.quantize_nhwc_i8   -> NHWC 8-bit codes of an NCHW x and their per-pixel channel sums
    torch.ops.mctq.packed_conv2d_i8   <- the integer convolution of NHWC codes and packed weight codes (implicit GEMM)
    torch.ops.mctq.packed_linear_i8_lut / packed_conv2d_i8_lut   the same with LUT weights: indices looked up as int8 codes
    torch.ops.mctq.packed_dwconv2d_i8 <- the integer depthwise convolution of Q's codes of x (computed in the kernel)

(reference call sites: see include/mctq.h).  Each op has a CUDA implementation (device pointers + the
caller's current stream into the C ABI, no synchronisation), a CPU-tensor implementation that streams the
host buffer through the GPU (mctq_fq_*_host), and a fake/meta implementation so that fx tracing,
torch.compile and shape propagation work.  There is no eager / CPU arithmetic fallback anywhere.
"""
import ctypes
import functools

import numpy as np
import torch

from mct_quantizers_b200 import _native
from mct_quantizers_b200._native import MctqError, c_vp

_DT = {torch.float32: _native.F32, torch.bfloat16: _native.BF16, torch.float16: _native.F16}

_LIB = torch.library.Library("mctq", "DEF")
_LIB.define("fq_affine_scalar(Tensor x, float scale, int zero_point, int quant_min, int quant_max) -> Tensor")
_LIB.define("fq_affine_scalar_pre(Tensor x, Tensor? other, int pre_op, float scale, int zero_point, int quant_min, int quant_max) -> Tensor")
_LIB.define("fq_affine_tensor(Tensor x, Tensor scale, Tensor zero_point, int quant_min, int quant_max) -> Tensor")
_LIB.define("fq_affine_channel(Tensor x, Tensor scale, Tensor zero_point, int axis, int quant_min, int quant_max) -> Tensor")
_LIB.define("fq_lut_tensor(Tensor x, Tensor table, int K, Tensor threshold, bool per_channel, int axis, float eps) -> Tensor")
_LIB.define("fq_lut_scalar(Tensor x, Tensor table, int K, float divisor, float threshold, bool round_to_input_dtype, bool multiply=False) -> Tensor")
_LIB.define("quantize_affine_channel(Tensor x, Tensor scale, Tensor zero_point, int axis, int quant_min, int quant_max, "
            "int code_mode, bool want_values) -> (Tensor, Tensor)")
_LIB.define("dequantize_affine(Tensor codes, int code_mode, bool is_signed, int[] shape, Tensor scale, Tensor zero_point, "
            "int axis) -> Tensor")
_LIB.define("lut_indices(Tensor x, Tensor table, int K, Tensor threshold, bool per_channel, int axis, float eps, "
            "int idx_mode) -> Tensor")
_LIB.define("dequantize_lut(Tensor idx, int idx_mode, int[] shape, Tensor lut, int lut_values_bitwidth, bool is_signed, "
            "Tensor threshold, bool per_channel, int axis) -> Tensor")
_LIB.define("packed_linear(Tensor x, Tensor codes, int kind, bool is_signed, int out_features, Tensor scale, "
            "Tensor? zero_point, Tensor? lut_quotients, Tensor? bias) -> Tensor")
_LIB.define("packed_linear_batched(Tensor x, Tensor codes, int kind, bool is_signed, int out_features, Tensor scale, "
            "Tensor? zero_point, Tensor? lut_quotients, Tensor? bias) -> Tensor")
_LIB.define("quantize_rows_i8(Tensor x, float scale, int zero_point, int quant_min, int quant_max, bool want_rowsum) "
            "-> (Tensor, Tensor)")
_LIB.define("packed_linear_i8(Tensor x_codes, int x_zero_point, Tensor? x_rowsum, Tensor codes, int kind, bool is_signed, "
            "int out_features, Tensor zero_point, Tensor w_rowsum, Tensor factor, Tensor? bias, ScalarType dtype) -> Tensor")
_LIB.define("quantize_nhwc_i8(Tensor x, float scale, int zero_point, int quant_min, int quant_max, bool want_sums) "
            "-> (Tensor, Tensor)")
_LIB.define("packed_conv2d_i8(Tensor x_codes, int x_zero_point, Tensor? x_rowsum, Tensor codes, int kind, bool is_signed, "
            "int out_channels, int[] kernel_size, int[] stride, int[] dilation, int[] padding, Tensor zero_point, "
            "Tensor w_rowsum, Tensor factor, Tensor? bias, ScalarType dtype, bool channels_last) -> Tensor")
_LIB.define("packed_linear_i8_lut(Tensor x_codes, int x_zero_point, Tensor codes, int kind, int out_features, "
            "int[] lut_values, Tensor w_rowsum, Tensor factor, Tensor? bias) -> Tensor")
_LIB.define("packed_conv2d_i8_lut(Tensor x_codes, int x_zero_point, Tensor codes, int kind, int out_channels, "
            "int[] kernel_size, int[] stride, int[] dilation, int[] padding, int[] lut_values, Tensor w_rowsum, "
            "Tensor factor, Tensor? bias, bool channels_last) -> Tensor")
_LIB.define("quantize_rows_i8_padded(Tensor x, int ldc, float scale, int zero_point, int quant_min, int quant_max, "
            "bool want_rowsum) -> (Tensor, Tensor)")
_LIB.define("quantize_nhwc_i8_padded(Tensor x, int channel_pitch, float scale, int zero_point, int quant_min, int quant_max, "
            "bool want_sums) -> (Tensor, Tensor)")
_LIB.define("packed_linear_i8_padded(Tensor x_codes, int in_features, int x_zero_point, Tensor? x_rowsum, Tensor codes, "
            "int kind, bool is_signed, int out_features, Tensor? zero_point, Tensor w_rowsum, Tensor factor, Tensor? bias, "
            "ScalarType dtype, int[]? lut_values) -> Tensor")
_LIB.define("packed_conv2d_i8_padded(Tensor x_codes, int in_channels, int x_zero_point, Tensor? x_rowsum, Tensor codes, "
            "int kind, bool is_signed, int out_channels, int[] kernel_size, int[] stride, int[] dilation, int[] padding, "
            "Tensor? zero_point, Tensor w_rowsum, Tensor factor, Tensor? bias, ScalarType dtype, bool channels_last, "
            "int[]? lut_values) -> Tensor")
_LIB.define("packed_dwconv2d_i8(Tensor x, float x_scale, int x_zero_point, int x_qmin, int x_qmax, Tensor codes, int kind, "
            "bool is_signed, int out_channels, int[] kernel_size, int[] stride, int[] dilation, int[] padding, "
            "Tensor? zero_point, Tensor factor, Tensor? lut_values, Tensor? bias, bool channels_last) -> Tensor")


# --------------------------------------------------------------------------------------------- helpers
def _dtype_tag(x):
    try:
        return _DT[x.dtype]
    except KeyError:
        raise NotImplementedError(f'"mctq_fake_quantize" not implemented for \'{x.dtype}\' '
                                  f'(float32, bfloat16 and float16 are supported)') from None


def _ptr(t):
    return t.data_ptr() if t is not None else None      # ctypes converts ints for c_void_p parameters


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_get_device = getattr(torch._C, "_cuda_getDevice", None)
_set_device = getattr(torch._C, "_cuda_setDevice", None)
if _raw_stream is None:                      # private fast paths missing in this torch build: public equivalents
    def _raw_stream(index):
        return torch.cuda.current_stream(index).cuda_stream
if _get_device is None:
    _get_device = torch.cuda.current_device
if _set_device is None:
    _set_device = torch.cuda.set_device


def _stream(device):
    """cudaStream_t (as int) of the current stream of `device`."""
    if _raw_stream is not None and device.index is not None:
        return _raw_stream(device.index)
    return torch.cuda.current_stream(device).cuda_stream


_PLAIN_TENSOR_TYPES = (torch.Tensor, torch.nn.Parameter)


def direct_ok(x):
    """True when the quantizers may call the launch functions below directly instead of going through the
    torch.ops dispatcher (saves ~10 us per call): a plain CUDA tensor, and nobody is tracing / compiling / exporting
    (tracers must see the custom operator)."""
    return (type(x) in _PLAIN_TENSOR_TYPES and x.is_cuda and not torch.jit.is_tracing()
            and not torch.compiler.is_compiling())


class _on_device:
    """Make `device` current for the duration of a launch (kernels launch on the current device)."""
    __slots__ = ("idx", "prev")

    def __init__(self, device):
        self.idx = device.index if device.index is not None else torch.cuda.current_device()

    def __enter__(self):
        self.prev = _get_device() if _get_device is not None else torch.cuda.current_device()
        if self.prev != self.idx:
            torch.cuda.set_device(self.idx)
        return self

    def __exit__(self, *exc):
        if self.prev != self.idx:
            torch.cuda.set_device(self.prev)


def _is_dense_permutation(x):
    """True when x's elements occupy one gap-free block of memory in some permutation of its dims."""
    dims = sorted((d for d in range(x.dim()) if x.shape[d] > 1), key=lambda d: x.stride(d))
    expect = 1
    for d in dims:
        if x.stride(d) != expect:
            return False
        expect *= x.shape[d]
    return True


def _dense(x):
    """x itself when its memory is one dense block (any permutation of strides), else a contiguous copy."""
    if x.is_contiguous() or x.numel() == 0:
        return x
    if _is_dense_permutation(x):
        return x
    return x.contiguous()


def _channel_layout(x, axis):
    """(x_dense, C, inner): the [outer][C][inner] view in MEMORY order.  For a permuted-but-dense tensor
    (e.g. channels_last) the channel axis keeps its meaning; only `inner` changes."""
    nd = x.dim()
    if not -nd <= axis < nd:
        raise IndexError(f"Dimension out of range (expected to be in range of [{-nd}, {nd - 1}], but got {axis})")
    axis %= nd
    x = _dense(x)
    C = x.shape[axis]
    if x.is_contiguous():
        inner = 1
        for s in x.shape[axis + 1:]:
            inner *= int(s)
        return x, int(C), inner
    # dense, permuted: dims that sit "inside" the channel axis in memory are those with a smaller stride
    # -- valid only if they tile the channel stride exactly
    strides, shape = x.stride(), x.shape
    inner = 1
    for d in range(nd):
        if d != axis and shape[d] > 1 and strides[d] < strides[axis]:
            inner *= int(shape[d])
    if C > 1 and strides[axis] != inner:
        x = x.contiguous()
        return _channel_layout(x, axis)
    return x, int(C), inner


def _check_range(qmin, qmax):
    if qmin > qmax:
        raise RuntimeError("`quant_min` should be less than or equal to `quant_max`.")


def _check_channel_params(x, scale, zp, axis):
    if scale.dtype != torch.float32:
        raise RuntimeError(f"Scale must be Float, found {scale.dtype}")
    if zp.dtype != torch.int32:
        raise RuntimeError(f"Zero-point must be Int32, found {zp.dtype}")
    if scale.dim() != 1 or zp.dim() != 1:
        raise RuntimeError("scale and zero-point need to be 1-D tensors")
    nd = x.dim()
    if not -nd <= axis < nd:
        raise RuntimeError("`axis` must be between 0 and number of dimensions of input")
    if scale.numel() != x.shape[axis] or zp.numel() != x.shape[axis]:
        raise RuntimeError("dimensions of scale and zero-point are not consistent with input tensor")


def _ver(t):
    """Version counter of a parameter tensor for cache keys; inference tensors have none (and cannot be edited in place
    outside inference mode), so they get a constant."""
    return -1 if t.is_inference() else t._version


_PARAM_COPIES = {}        # (data_ptr, version, numel, dtype, src device, dst device) -> (source kept alive, copy)


def _param_on(t, device):
    """`t` on `device`.  Cross-device copies are cached: a fresh copy per call would also defeat the prepared-parameter
    caches below (their keys hold the copy's data_ptr) and re-prepare on every call."""
    if t.device == device:
        return t
    key = (t.data_ptr(), _ver(t), t.numel(), t.dtype, str(t.device), str(device))
    hit = _PARAM_COPIES.get(key)
    if hit is None:
        if len(_PARAM_COPIES) >= 1024:
            _PARAM_COPIES.clear()
        hit = (t, t.to(device, non_blocking=True))
        _PARAM_COPIES[key] = hit
    return hit[1]


_staging = {}


def _staging_buffer(device_index):
    buf = _staging.get(device_index)
    nbytes = _native.load().mctq_host_staging_min_bytes()        # three staging slots + the parameter area (304 MiB)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(nbytes, dtype=torch.uint8, device=torch.device("cuda", device_index))
        _staging[device_index] = buf
    return buf


def _require_cuda_for_host_path():
    if not torch.cuda.is_available():
        raise MctqError("mct_quantizers_b200 received a CPU tensor but no CUDA device is available: the package "
                        "has no CPU arithmetic path (host tensors are streamed through the GPU)")
    return torch.cuda.current_device()


def _host_array(t, dtype):
    return np.ascontiguousarray(t.detach().cpu().numpy().astype(dtype, copy=False).reshape(-1))


# --------------------------------------------------------------------------------------------- CUDA impls
def affine_scalar_direct(x, scale_f32, zero_point, quant_min, quant_max):
    """Lean launch (no dispatcher, no re-validation): `scale_f32` is already narrowed to f32, the range was validated
    when the quantizer was built."""
    tag = _DT.get(x.dtype)
    if tag is None:
        _dtype_tag(x)
    xd = x if x.is_contiguous() else _dense(x)
    y = torch.empty_like(xd)
    n = xd.numel()
    if n:
        lib = _native._lib or _native.load()
        dev = xd.device
        prev = _get_device()
        if prev != dev.index:
            _set_device(dev.index)
        fast = _native.fast                     # CPython front door (METH_FASTCALL) when built; ctypes otherwise -- same entry point
        rc = (fast.fq_affine_scalar if fast is not None else lib.mctq_fq_affine_scalar)(
            xd.data_ptr(), y.data_ptr(), None, n, tag, scale_f32, zero_point, quant_min, quant_max, 0, _raw_stream(dev.index))
        if prev != dev.index:
            _set_device(prev)
        if rc:
            _native.check(rc, "mctq_fq_affine_scalar")
    return y


def _affine_scalar_cuda(x, scale, zero_point, quant_min, quant_max):
    _dtype_tag(x)
    _check_range(quant_min, quant_max)
    if not quant_min <= zero_point <= quant_max:
        raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
    return affine_scalar_direct(x, float(np.float32(scale)), int(zero_point), int(quant_min), int(quant_max))


def affine_scalar_pre_direct(x, other, pre_op, scale_f32, zero_point, quant_min, quant_max):
    """Producer (relu / relu6 / add / add+relu) and per-tensor fake-quant in ONE kernel: mctq_fq_affine_scalar_pre.
    Lean launch; arguments are already validated."""
    tag = _DT.get(x.dtype)
    if tag is None:
        _dtype_tag(x)
    xd = x if x.is_contiguous() else _dense(x)
    od = None
    if pre_op in (_native.PRE_ADD, _native.PRE_ADD_RELU):
        if other is None or other.shape != x.shape or other.dtype != x.dtype or other.device != x.device:
            raise RuntimeError("fused add needs a second tensor of the same shape, dtype and device (no broadcasting)")
        od = other if other.stride() == xd.stride() and _is_dense_permutation(other) else None
        if od is None:
            od = other.contiguous()
            if not xd.is_contiguous():
                xd = xd.contiguous()
    y = torch.empty_like(xd)
    n = xd.numel()
    if n:
        lib = _native._lib or _native.load()
        index = xd.device.index
        prev = _get_device()
        if prev != index:
            _set_device(index)
        fast = _native.fast
        rc = (fast.fq_affine_scalar_pre if fast is not None else lib.mctq_fq_affine_scalar_pre)(
            xd.data_ptr(), od.data_ptr() if od is not None else None, y.data_ptr(), n, tag, pre_op, scale_f32, zero_point,
            quant_min, quant_max, _raw_stream(index))
        if prev != index:
            _set_device(prev)
        if rc:
            _native.check(rc, "mctq_fq_affine_scalar_pre")
    return y


def _affine_scalar_pre_cuda(x, other, pre_op, scale, zero_point, quant_min, quant_max):
    _dtype_tag(x)
    _check_range(quant_min, quant_max)
    if not quant_min <= zero_point <= quant_max:
        raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
    if pre_op not in (_native.PRE_RELU, _native.PRE_RELU6, _native.PRE_ADD, _native.PRE_ADD_RELU):
        raise RuntimeError("pre_op must be 1 (relu), 2 (relu6), 3 (add) or 4 (add + relu)")
    if pre_op in (_native.PRE_ADD, _native.PRE_ADD_RELU) and (other is None or other.shape != x.shape or other.dtype != x.dtype
                                                              or other.device != x.device):
        # broadcasting / type-promoting add: the eager add, then the (relu-)fused fake-quant
        if other is None:
            raise RuntimeError("pre_op add needs `other`")
        t = torch.add(x, other)
        if pre_op == _native.PRE_ADD:
            return _affine_scalar_cuda(t, scale, zero_point, quant_min, quant_max)
        x, other, pre_op = t, None, _native.PRE_RELU
    return affine_scalar_pre_direct(x, other, int(pre_op), float(np.float32(scale)), int(zero_point), int(quant_min), int(quant_max))


# ---- prepared per-channel parameters: {1/s, s, zp} records the kernels stage with TMA bulk copies (mctq_affine_prepare)
_AFFINE_PREPARED = {}     # (scale ptr, zp ptr, versions, C, device) -> (scale, zp kept alive so the key stays unique, blob)


def clear_affine_caches():
    _AFFINE_PREPARED.clear()


def _affine_prepared(lib, scale, zero_point, index):
    """Device blob of prepared parameters for (scale, zero_point), built once per parameter pair; None while a CUDA
    graph is being captured and the blob does not exist yet (the raw-parameter entry point is used instead)."""
    key = (scale.data_ptr(), zero_point.data_ptr(), _ver(scale), _ver(zero_point), scale.numel(), index)
    ent = _AFFINE_PREPARED.get(key)
    if ent is None:
        if torch.cuda.is_current_stream_capturing():
            return None
        if len(_AFFINE_PREPARED) >= 4096:
            _AFFINE_PREPARED.clear()
        C = scale.numel()
        blob = torch.empty(lib.mctq_affine_prepared_bytes(C), dtype=torch.uint8, device=scale.device)
        stream = _raw_stream(index)
        rc = lib.mctq_affine_prepare(scale.data_ptr(), zero_point.data_ptr(), C, blob.data_ptr(), blob.numel(), stream)
        if rc:
            _native.check(rc, "mctq_affine_prepare")
        torch.cuda.current_stream(scale.device).synchronize()     # one-off: the blob may be used from any stream afterwards
        ent = (scale, zero_point, blob)
        _AFFINE_PREPARED[key] = ent
    return ent[2]


def _launch_affine_params(lib, x_ptr, y_ptr, codes_ptr, n, tag, scale, zero_point, C, inner, quant_min, quant_max, code_mode, index):
    """mctq_fq_affine_prepared for per-channel parameters (C > 1), mctq_fq_affine otherwise.  The caller has made
    `index` the current device."""
    fast = _native.fast
    if C > 1 and scale.is_contiguous() and zero_point.is_contiguous():
        blob = _affine_prepared(lib, scale, zero_point, index)
        if blob is not None:
            return (fast.fq_affine_prepared if fast is not None else lib.mctq_fq_affine_prepared)(
                x_ptr, y_ptr, codes_ptr, n, tag, blob.data_ptr(), C, inner, 0, quant_min, quant_max, code_mode,
                _raw_stream(index)), "mctq_fq_affine_prepared"
    return (fast.fq_affine if fast is not None else lib.mctq_fq_affine)(
        x_ptr, y_ptr, codes_ptr, n, tag, scale.data_ptr(), zero_point.data_ptr(), C, inner, 0, quant_min, quant_max, code_mode,
        _raw_stream(index)), "mctq_fq_affine"


def affine_params_direct(x, scale, zero_point, C, inner, quant_min, quant_max):
    """Lean launch of mctq_fq_affine for parameter TENSORS already on x's device and already validated
    (x: plain CUDA tensor; the (C, inner) view refers to x's memory order)."""
    tag = _DT.get(x.dtype)
    if tag is None:
        _dtype_tag(x)
    y = torch.empty_like(x)
    n = x.numel()
    if n:
        lib = _native._lib or _native.load()
        index = x.device.index
        prev = _get_device()
        if prev != index:
            _set_device(index)
        rc, what = _launch_affine_params(lib, x.data_ptr(), y.data_ptr(), None, n, tag, scale, zero_point, C, inner,
                                         quant_min, quant_max, 0, index)
        if prev != index:
            _set_device(prev)
        if rc:
            _native.check(rc, what)
    return y


def contiguous_layout(shape, axis):
    """(C, inner) of a contiguous tensor of `shape` quantized along `axis`."""
    inner = 1
    for d in shape[axis + 1:]:
        inner *= d
    return shape[axis], inner


def affine_codes(xd, scale, zero_point, C, inner, quant_min, quant_max, code_mode):
    """Integer codes of a dense CUDA tensor (no values) over its [outer][C][inner] memory-order view: int8 / uint8 [n] for
    CODES_INT8, packed nibbles uint8 [(n + 1) // 2] for CODES_INT4.  Same kernels and arithmetic as the fake-quant ops."""
    _check_range(quant_min, quant_max)
    n = xd.numel()
    if code_mode == _native.CODES_INT8:
        codes = torch.empty(n, dtype=torch.int8 if quant_min < 0 else torch.uint8, device=xd.device)
    else:
        codes = torch.empty(_native.packed_code_bytes(_native.PACK_AFFINE_I4, n), dtype=torch.uint8, device=xd.device)
    if n:
        lib = _native.load()
        s, z = _param_on(scale, xd.device), _param_on(zero_point, xd.device)
        with _on_device(xd.device) as cur:
            rc, what = _launch_affine_params(lib, xd.data_ptr(), None, codes.data_ptr(), n, _dtype_tag(xd), s, z, C, inner,
                                             int(quant_min), int(quant_max), int(code_mode), cur.idx)
        _native.check(rc, what)
    return codes


def _affine_tensor_cuda(x, scale, zero_point, quant_min, quant_max):
    tag = _dtype_tag(x)
    _check_range(quant_min, quant_max)
    if scale.numel() != 1 or zero_point.numel() != 1:
        raise RuntimeError(f"a Tensor with {max(scale.numel(), zero_point.numel())} elements cannot be converted to Scalar")
    if scale.dtype != torch.float32 or zero_point.dtype != torch.int32:
        raise RuntimeError("scale must be Float and zero_point Int32")
    xd = _dense(x)
    y = torch.empty_like(xd)
    if xd.numel():
        lib = _native.load()
        s, z = _param_on(scale, xd.device), _param_on(zero_point, xd.device)
        with _on_device(xd.device):
            rc = lib.mctq_fq_affine(_ptr(xd), _ptr(y), None, xd.numel(), tag, _ptr(s), _ptr(z), 1, 1, 0,
                                    int(quant_min), int(quant_max), 0, _stream(xd.device))
        _native.check(rc, "mctq_fq_affine")
    return y


def _affine_channel_launch(x, scale, zero_point, axis, quant_min, quant_max, code_mode, want_values):
    tag = _dtype_tag(x)
    _check_range(quant_min, quant_max)
    _check_channel_params(x, scale, zero_point, axis)
    xd, C, inner = _channel_layout(x, axis)
    y = torch.empty_like(xd) if want_values else None
    codes = None
    n = xd.numel()
    if code_mode == _native.CODES_INT8:
        codes = torch.empty_like(xd, dtype=torch.int8 if quant_min < 0 else torch.uint8)
    elif code_mode == _native.CODES_INT4:
        codes = torch.empty(_native.packed_code_bytes(_native.PACK_AFFINE_I4, n), dtype=torch.uint8, device=xd.device)
    if n:
        lib = _native.load()
        s, z = _param_on(scale, xd.device), _param_on(zero_point, xd.device)
        with _on_device(xd.device) as cur:
            rc, what = _launch_affine_params(lib, _ptr(xd), _ptr(y), _ptr(codes), n, tag, s.contiguous(), z.contiguous(), C, inner,
                                             int(quant_min), int(quant_max), int(code_mode), cur.idx)
        _native.check(rc, what)
    return y, codes


def _affine_channel_cuda(x, scale, zero_point, axis, quant_min, quant_max):
    return _affine_channel_launch(x, scale, zero_point, axis, quant_min, quant_max, 0, True)[0]


def _quantize_affine_channel_cuda(x, scale, zero_point, axis, quant_min, quant_max, code_mode, want_values):
    if code_mode not in (_native.CODES_INT8, _native.CODES_INT4):
        raise RuntimeError("code_mode must be 1 (int8) or 2 (packed int4)")
    y, codes = _affine_channel_launch(x, scale, zero_point, axis, quant_min, quant_max, code_mode, want_values)
    if y is None:
        y = torch.empty(0, dtype=x.dtype, device=x.device)
    return codes, y


def _dequantize_affine_cuda(codes, code_mode, is_signed, shape, scale, zero_point, axis):
    n = 1
    for s in shape:
        n *= int(s)
    nd = len(shape)
    axis %= max(nd, 1)
    C = int(shape[axis]) if nd else 1
    inner = 1
    for s in shape[axis + 1:]:
        inner *= int(s)
    if scale.numel() != C or zero_point.numel() != C:
        raise RuntimeError("dimensions of scale and zero-point are not consistent with `shape`")
    y = torch.empty(list(shape), dtype=torch.float32, device=codes.device)
    if n:
        lib = _native.load()
        codes = codes.contiguous()
        s, z = _param_on(scale, codes.device), _param_on(zero_point, codes.device)
        with _on_device(codes.device):
            rc = lib.mctq_dequant_affine(_ptr(codes), int(code_mode), int(bool(is_signed)), _ptr(y), n, _ptr(s), _ptr(z),
                                         C, inner, 0, _stream(codes.device))
        _native.check(rc, "mctq_dequant_affine")
    return y


# ---- LUT: per-device copies of the search table and per-(quantizer, device, dtype) prepared decision tables
_LUT_DEV_TABLES = {}      # (table.data_ptr(), device) -> (table_cpu kept alive, table_dev)
_LUT_PREPARED = {}        # key -> (objects kept alive so that data_ptr keys stay unique, prepared_dev or None)
_ROUND_TAG = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


def clear_lut_caches():
    _LUT_DEV_TABLES.clear()
    _LUT_PREPARED.clear()
    _PARAM_COPIES.clear()


def _table_header(table_cpu):
    """(bw, is_signed) out of the search-table blob (LutTableHeader: magic, K, Ks, P, levels, pos0, bw, is_signed, ...)."""
    hdr = table_cpu[:32].numpy().view(np.int32)
    return int(hdr[6]), int(hdr[7])


def _table_on(table, device):
    if table.device == device:
        return table
    key = (table.data_ptr(), str(device))
    hit = _LUT_DEV_TABLES.get(key)
    if hit is None:
        if torch.cuda.is_current_stream_capturing():
            # first use inside a CUDA-graph capture: the upload becomes a node of the graph and must read pinned memory
            # that outlives the graph (kept in the cache entry)
            src = table.pin_memory()
            hit = (table, src.to(device, non_blocking=True), src)
        else:
            hit = (table, table.to(device))
        _LUT_DEV_TABLES[key] = hit
    return hit[1]


def _prepared_for(table, K, device, thr_dev, eps, scalar, divisor, thr_f32, round_dtype):
    """Device blob of per-channel decision tables for this (centroid list, thresholds, device, rounding), built once.
    None when the configuration is outside the prepared path (table not on the host; a grid of more than 10 bits with a
    centroid list too dense for the cell table)."""
    if table.device.type != 'cpu':
        return None
    if scalar:
        key = (table.data_ptr(), int(K), str(device), 's', int(scalar), float(divisor), float(thr_f32), int(round_dtype))
        C = 1
    else:
        key = (table.data_ptr(), int(K), str(device), 't', thr_dev.data_ptr(), _ver(thr_dev), thr_dev.numel(), float(eps))
        C = thr_dev.numel()
    hit = _LUT_PREPARED.get(key)
    if hit is None:
        if torch.cuda.is_current_stream_capturing():
            return None                     # preparation synchronises: not inside a CUDA-graph capture (generic kernel instead)
        if len(_LUT_PREPARED) >= 1024:      # bounded like _AFFINE_PREPARED: entries pin a threshold tensor and a device blob
            _LUT_PREPARED.clear()
        lib = _native.load()
        bw, signed = _table_header(table)
        nbytes = lib.mctq_lut_prepared_bytes(int(K), bw, signed, C)
        blob = None
        if nbytes:
            blob = torch.empty(nbytes, dtype=torch.uint8, device=device)
            with _on_device(device):
                rc = lib.mctq_lut_prepare(_ptr(table), int(K), _ptr(thr_dev) if not scalar else None, C,
                                          float(np.float32(eps)), int(scalar), float(np.float32(divisor)),
                                          float(np.float32(thr_f32)), int(round_dtype), _ptr(blob), nbytes, _stream(device))
            if rc == -3:                                         # MCTQ_E_RANGE: a grid of more than 10 bits whose centroids are too
                blob = None                                      # dense for the coarse cell table -> generic kernel
            else:
                _native.check(rc, "mctq_lut_prepare")
                torch.cuda.current_stream(device).synchronize()  # one-off: the blob may be used from any stream afterwards
        hit = ((table, thr_dev), blob, bw, signed)
        _LUT_PREPARED[key] = hit
    return hit


def _lut_launch(xd, y, idx, idx_mode, table, K, C, inner, thr_dev, eps, scalar, divisor, thr_f32, round_flag):
    """Prepared kernel when possible, generic kernel otherwise."""
    lib = _native.load()
    tag = _dtype_tag(xd)
    n = xd.numel()
    round_dtype = _ROUND_TAG[xd.dtype] if (scalar and round_flag) else 0
    prep = _prepared_for(table, K, xd.device, thr_dev, eps, scalar, divisor, thr_f32, round_dtype)
    with _on_device(xd.device):
        if prep is not None and prep[1] is not None:
            rc = lib.mctq_fq_lut_prepared(_ptr(xd), _ptr(y), _ptr(idx), n, tag, _ptr(prep[1]), int(K), prep[2], prep[3],
                                          C, inner, 0, int(idx_mode), _stream(xd.device))
            if rc == 0:
                return
            if rc not in (-1, -3):                      # BADARG (misaligned view) / RANGE (window too wide): generic path
                _native.check(rc, "mctq_fq_lut_prepared")
        t = _table_on(table, xd.device)
        if scalar:
            rc = lib.mctq_fq_lut_scalar(_ptr(xd), _ptr(y), _ptr(idx), n, tag, _ptr(t), int(K), float(np.float32(divisor)),
                                        float(np.float32(thr_f32)), int(bool(round_flag)) | (2 if scalar == 2 else 0), int(idx_mode),
                                        _stream(xd.device))
        else:
            rc = lib.mctq_fq_lut(_ptr(xd), _ptr(y), _ptr(idx), n, tag, _ptr(t), int(K), _ptr(thr_dev), C, inner, 0,
                                 float(np.float32(eps)), int(idx_mode), _stream(xd.device))
    _native.check(rc, "mctq_fq_lut")


def _lut_tensor_launch(x, table, K, threshold, per_channel, axis, eps, idx_mode, want_values):
    _dtype_tag(x)
    if threshold.dtype != torch.float32:
        raise RuntimeError(f"threshold must be Float, found {threshold.dtype}")
    if per_channel:
        if threshold.numel() != x.shape[axis]:
            raise RuntimeError(f"shape '{[1] * x.dim()}' is invalid for threshold of size {threshold.numel()} "
                               f"(input has {x.shape[axis]} channels on axis {axis})")
        xd, C, inner = _channel_layout(x.contiguous(), axis)     # row-major output like the reference's eager composition
    else:
        if threshold.numel() != 1:
            raise RuntimeError("per-tensor LUT quantization needs a single threshold")
        xd, C, inner = x.contiguous(), 1, 1
    n = xd.numel()
    y = torch.empty_like(xd, dtype=torch.float32) if want_values else None
    idx = None
    if idx_mode == _native.CODES_INT8:
        idx = torch.empty_like(xd, dtype=torch.uint8)
    elif idx_mode == _native.CODES_INT4:
        idx = torch.empty(_native.packed_code_bytes(_native.PACK_LUT_I4, n), dtype=torch.uint8, device=xd.device)
    if n:
        thr = _param_on(threshold.contiguous(), xd.device)
        _lut_launch(xd, y, idx, idx_mode, table, K, C, inner, thr, eps, False, 1.0, 1.0, False)
    if y is not None and y.dim() == 0:
        y = y.reshape(1)        # the reference multiplies by the threshold TENSOR of shape (1,): a 0-dim input comes back 1-D
    return y, idx


def lut_weights_direct(x, table, K, threshold, per_channel, axis, eps, cache):
    """Lean launch of the prepared LUT kernel for a weight quantizer (no dispatcher, no per-call validation or cache-key
    building: ~35 us -> ~10 us of host time per call, which matters once a 45 M-element bf16 matrix takes 40 us on the
    device).  `cache` is a dict owned by the quantizer: (shape, dtype, device, thr ptr) -> launch constants.  Anything
    unusual (non-contiguous input, no prepared blob, misaligned view) goes through the general path."""
    if x.is_contiguous() and x.numel() and x.dim():        # (0-dim inputs: general path, which returns them 1-D like the reference)
        key = (x.shape, x.dtype, x.device, threshold.data_ptr(), _ver(threshold))
        hit = cache.get(key)
        if hit is None:
            hit = False
            tag = _DT.get(x.dtype)
            if tag is not None and threshold.dtype == torch.float32 and (not per_channel or threshold.numel() == x.shape[axis]) \
                    and (per_channel or threshold.numel() == 1):
                if per_channel:
                    _, C, inner = _channel_layout(x, axis)
                else:
                    C, inner = 1, 1
                thr = _param_on(threshold.contiguous(), x.device)
                prep = _prepared_for(table, K, x.device, thr, eps, False, 1.0, 1.0, 0)
                if prep is not None and prep[1] is not None:
                    hit = (tag, int(K), prep[2], prep[3], C, inner, prep[1].data_ptr(), (thr, prep), x.device.index)
            if len(cache) > 16:
                cache.clear()
            if hit or not torch.cuda.is_current_stream_capturing():     # a capture only postpones the preparation
                cache[key] = hit
        if hit:
            tag, K_, bw, signed, C, inner, blob_ptr, _, index = hit
            if (x.data_ptr() & 15) == 0:
                y = torch.empty(x.shape, dtype=torch.float32, device=x.device)
                lib = _native._lib or _native.load()
                prev = _get_device()
                if prev != index:
                    _set_device(index)
                fast = _native.fast
                rc = (fast.fq_lut_prepared if fast is not None else lib.mctq_fq_lut_prepared)(
                    x.data_ptr(), y.data_ptr(), None, x.numel(), tag, blob_ptr, K_, bw, signed, C, inner, 0, 0, _raw_stream(index))
                if prev != index:
                    _set_device(prev)
                if rc == 0:
                    return y
    return _lut_tensor_cuda(x, table, K, threshold, per_channel, axis, eps)


def _lut_tensor_cuda(x, table, K, threshold, per_channel, axis, eps):
    return _lut_tensor_launch(x, table, K, threshold, per_channel, axis, eps, 0, True)[0]


def _lut_indices_cuda(x, table, K, threshold, per_channel, axis, eps, idx_mode):
    if idx_mode not in (_native.CODES_INT8, _native.CODES_INT4):
        raise RuntimeError("idx_mode must be 1 (uint8) or 2 (packed 4-bit)")
    return _lut_tensor_launch(x, table, K, threshold, per_channel, axis, eps, idx_mode, False)[1]


def lut_quotients(lut, lut_values_bitwidth, is_signed):
    """q_k = lut_k / 2^(bw - signed) as a host f32 tensor: the division the reference performs before it multiplies by the
    threshold (quantizer_utils.py: `lut_values / 2 ** (lut_values_bitwidth - int(signed))`, CPU f32)."""
    return lut.detach().to("cpu", torch.float32).reshape(-1) / 2 ** (int(lut_values_bitwidth) - int(bool(is_signed)))


def _dequantize_lut_cuda(idx, idx_mode, shape, lut, lut_values_bitwidth, is_signed, threshold, per_channel, axis):
    """y[i] = q[idx[i]] * thr[c(i)] (f32) over the row-major `shape`: the consumer of mctq::lut_indices.  Like fq_lut_tensor,
    a 0-dim `shape` comes back 1-D."""
    if idx_mode == _native.CODES_INT8:
        kind = _native.PACK_LUT_U8
    elif idx_mode == _native.CODES_INT4:
        kind = _native.PACK_LUT_I4
    else:
        raise RuntimeError("idx_mode must be 1 (uint8) or 2 (packed 4-bit)")
    shape = [int(s) for s in shape]
    n = 1
    for s in shape:
        n *= s
    if threshold.dtype != torch.float32:
        raise RuntimeError(f"threshold must be Float, found {threshold.dtype}")
    if per_channel:
        nd = len(shape)
        if not -nd <= axis < nd:
            raise IndexError(f"Dimension out of range (expected to be in range of [{-nd}, {nd - 1}], but got {axis})")
        C, inner = contiguous_layout(shape, axis % nd)
        if threshold.numel() != C:
            raise RuntimeError(f"threshold has {threshold.numel()} entries for {C} channels on axis {axis}")
    else:
        C, inner = 1, 1
        if threshold.numel() != 1:
            raise RuntimeError("per-tensor LUT dequantization needs a single threshold")
    need = _native.packed_code_bytes(kind, n)
    if idx.numel() != need or idx.dtype not in (torch.uint8, torch.int8):
        raise RuntimeError(f"idx must hold {need} bytes for shape {shape} and idx_mode {idx_mode}")
    q = lut_quotients(lut, lut_values_bitwidth, is_signed)
    item = (idx, kind, False, torch.float32, shape if shape else [1], None, C, inner, threshold.reshape(-1), None, q)
    return UnpackPlan([item]).run()[0]


def _packed_desc(codes, kind, is_signed, dtype, n, C, inner, scale, zero_point, lut_quotients, device, what):
    """The MctqPackedDesc of n packed elements (y unset), parameters placed on `device`: (desc, the tensors it points into).
    `what` names the tensor in the ValueError messages."""
    if codes.dtype not in (torch.uint8, torch.int8) or codes.numel() != _native.packed_code_bytes(kind, n):
        raise ValueError(f"{what}: codes ({codes.dtype}, {codes.numel()} bytes) do not hold {n} elements of kind {kind}")
    codes = codes.contiguous()
    s = _param_on(scale.detach().reshape(-1).contiguous(), device)
    z = _param_on(zero_point.detach().reshape(-1).contiguous(), device) if zero_point is not None else None
    q = _param_on(lut_quotients.detach().reshape(-1).contiguous(), device) if lut_quotients is not None else None
    if s.dtype != torch.float32 or (z is not None and z.dtype != torch.int32) or (q is not None and q.dtype != torch.float32):
        raise ValueError(f"{what}: scale / threshold and quotients must be float32, zero points int32")
    d = _native.MctqPackedDesc()
    d.codes, d.y, d.n, d.C, d.inner = codes.data_ptr(), None, n, int(C), int(inner)
    d.kind, d.is_signed, d.y_dtype = int(kind), int(bool(is_signed)), _DT.get(dtype, -1)
    d.K = q.numel() if q is not None else 0
    d.scale, d.zp, d.lut_quotients = s.data_ptr(), _ptr(z), _ptr(q)
    return d, (codes, s, z, q)


class PackedLinear:
    """Launch state of one packed [out_features, in_features] weight for mctq_packed_linear: the descriptor is built once, and
    a call is one C-ABI call with pointers and the row count.
        codes, kind, is_signed   the packed weight (kind: _native.PACK_*), row-major [out][in]
        dtype                    the rebuilt weight's dtype (f32 for the LUT kinds): x, bias and y have it
        scale                    f32, 1 (per tensor) or out_features entries (affine scale or LUT threshold)
        zero_point               int32 like scale (affine) or None; lut_quotients f32 [K] (LUT kinds) or None
    `__call__(x, bias)` returns x @ W^T + bias for a contiguous x of `dtype` on the codes' device, enqueued on the current
    stream; W is exactly the weight UnpackPlan rebuilds, the sum is accumulated in f32 in a fixed order.  `batched(x, bias)`
    computes the same product with mctq_packed_linear_batched (tensor cores, for tens to hundreds of rows); for the LUT kinds
    it reads the quotients on the host (_quotients_host: one synchronising copy per table contents, none when they are on
    the CPU), so capture a batched LUT call in a CUDA graph after one eager call."""

    def __init__(self, codes, kind, is_signed, dtype, out_features, in_features, scale, zero_point, lut_quotients):
        self.device = codes.device
        if self.device.type != "cuda":
            raise ValueError("PackedLinear needs CUDA tensors")
        self.out_features, self.in_features, self.dtype = int(out_features), int(in_features), dtype
        C, inner = (scale.numel(), self.in_features) if scale.numel() > 1 else (1, 1)
        self._desc, self._keep = _packed_desc(codes, kind, is_signed, dtype, self.out_features * self.in_features, C, inner,
                                              scale, zero_point, lut_quotients, self.device, "PackedLinear")
        s, z = self._keep[1], self._keep[2]
        if s.numel() not in (1, self.out_features) or (z is not None and z.numel() != s.numel()):
            raise ValueError(f"{s.numel()} parameters for {out_features} output channels (per tensor or per output channel)")
        self._quot_src = lut_quotients.detach().reshape(-1) if lut_quotients is not None else None
        self._desc_ptr = ctypes.addressof(self._desc)

    def __call__(self, x, bias=None):
        return self._run(x, bias, False)

    def batched(self, x, bias=None):
        return self._run(x, bias, True)

    def _run(self, x, bias, batched):
        if x.dtype != self.dtype or (bias is not None and bias.dtype != self.dtype):
            raise RuntimeError(f"packed_linear: x and bias must have the weight's dtype {self.dtype}")
        if x.dim() == 0 or x.shape[-1] != self.in_features:
            raise RuntimeError(f"packed_linear: x of shape {list(x.shape)} does not end in in_features = {self.in_features}")
        if x.device != self.device or (bias is not None and bias.device != self.device):
            raise RuntimeError(f"packed_linear: x and bias must live on {self.device}")
        if bias is not None and bias.numel() != self.out_features:
            raise RuntimeError(f"packed_linear: bias has {bias.numel()} entries for {self.out_features} outputs")
        x = x.contiguous()
        y = torch.empty(tuple(x.shape[:-1]) + (self.out_features,), dtype=self.dtype, device=self.device)
        M = x.numel() // self.in_features
        if M:
            b = bias.contiguous() if bias is not None else None
            fast = _native.fast
            with _on_device(self.device):
                args = (self._desc_ptr, self.out_features, self.in_features, x.data_ptr(), _DT[self.dtype], M, _ptr(b),
                        y.data_ptr())
                if batched:
                    qh = _quotients_host(self._quot_src)
                    args += (qh.ctypes.data if qh is not None else None, _stream(self.device))
                    rc = fast.packed_linear_batched(*args) if fast is not None else \
                        _native.load().mctq_packed_linear_batched(*args)
                else:
                    args += (_stream(self.device),)
                    rc = fast.packed_linear(*args) if fast is not None else _native.load().mctq_packed_linear(*args)
            _native.check(rc, "mctq_packed_linear_batched" if batched else "mctq_packed_linear")
        return y


_QUOT_HOST = {}


def _quotients_host(q):
    """The f32 LUT quotients `q` as a host numpy array for mctq_packed_linear_batched, cached by storage and version like
    _param_on: a device tensor is copied (and synchronised) once per contents, so that later calls, CUDA-graph capture
    included, need no copy; an in-place update (load_state_dict) bumps the version and is read again."""
    if q is None:
        return None
    key = (q.data_ptr(), _ver(q), q.numel(), q.dtype, str(q.device))
    hit = _QUOT_HOST.get(key)
    if hit is None:
        if len(_QUOT_HOST) >= 1024:
            _QUOT_HOST.clear()
        hit = (q, np.ascontiguousarray(q.to("cpu", torch.float32).numpy()))
        _QUOT_HOST[key] = hit
    return hit[1]


def _packed_linear_cuda(x, codes, kind, is_signed, out_features, scale, zero_point, lut_quotients, bias, batched=False):
    """mctq::packed_linear, and mctq::packed_linear_batched with `batched`."""
    _dtype_tag(x)
    if x.dim() == 0:
        raise RuntimeError(f"packed_linear{'_batched' if batched else ''}: x must have at least one dimension")
    _native.load()
    lin = PackedLinear(codes, kind, is_signed, x.dtype, out_features, x.shape[-1], scale, zero_point, lut_quotients)
    return lin._run(x, bias, batched)


_packed_linear_batched_cuda = functools.partial(_packed_linear_cuda, batched=True)


def quantize_rows_i8(x, scale_f32, zero_point, quant_min, quant_max, want_rowsum):
    """(codes, rowsum) of a CUDA tensor x [..., K] under a per-tensor 8-bit affine quantizer (mctq_quantize_rows_i8): codes of
    x's shape, int8 when quant_min < 0 else uint8, exactly the codes mctq_fq_affine_scalar emits; rowsum int32 [M] (M = the
    product of the leading dimensions), or an empty tensor unless `want_rowsum`.  `scale_f32` is already narrowed to f32."""
    tag = _dtype_tag(x)
    if x.dim() == 0:
        raise RuntimeError("quantize_rows_i8: x must have at least one dimension")
    xd = x.contiguous()
    K = xd.shape[-1]
    M = xd.numel() // K if K else 0
    codes = torch.empty(xd.shape, dtype=torch.int8 if quant_min < 0 else torch.uint8, device=xd.device)
    rowsum = torch.empty((M if want_rowsum else 0,), dtype=torch.int32, device=xd.device)
    if M:
        with _on_device(xd.device):
            rc = _native.load().mctq_quantize_rows_i8(xd.data_ptr(), tag, M, K, scale_f32, zero_point, quant_min, quant_max,
                                                       codes.data_ptr(), _ptr(rowsum) if want_rowsum else None,
                                                       _stream(xd.device))
        _native.check(rc, "mctq_quantize_rows_i8")
    return codes, rowsum


def _quantize_rows_i8_cuda(x, scale, zero_point, quant_min, quant_max, want_rowsum):
    _check_range(quant_min, quant_max)
    if not quant_min <= zero_point <= quant_max:
        raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
    return quantize_rows_i8(x, float(np.float32(scale)), int(zero_point), int(quant_min), int(quant_max), bool(want_rowsum))


def quantize_rows_i8_padded(x, ldc, scale_f32, zero_point, quant_min, quant_max, want_rowsum):
    """quantize_rows_i8 with codes [..., ldc] (ldc >= K, a multiple of 4): the columns [K, ldc) hold zero_point and the row
    sums include them (mctq_quantize_rows_i8_padded)."""
    tag = _dtype_tag(x)
    if x.dim() == 0:
        raise RuntimeError("quantize_rows_i8_padded: x must have at least one dimension")
    xd = x.contiguous()
    K = xd.shape[-1]
    M = xd.numel() // K if K else 0
    codes = torch.empty(tuple(xd.shape[:-1]) + (int(ldc),), dtype=torch.int8 if quant_min < 0 else torch.uint8,
                        device=xd.device)
    rowsum = torch.empty((M if want_rowsum else 0,), dtype=torch.int32, device=xd.device)
    if M:
        with _on_device(xd.device):
            rc = _native.load().mctq_quantize_rows_i8_padded(xd.data_ptr(), tag, M, K, int(ldc), scale_f32, zero_point,
                                                              quant_min, quant_max, codes.data_ptr(),
                                                              _ptr(rowsum) if want_rowsum else None, _stream(xd.device))
        _native.check(rc, "mctq_quantize_rows_i8_padded")
    return codes, rowsum


def _quantize_rows_i8_padded_cuda(x, ldc, scale, zero_point, quant_min, quant_max, want_rowsum):
    _check_range(quant_min, quant_max)
    if not quant_min <= zero_point <= quant_max:
        raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
    return quantize_rows_i8_padded(x, int(ldc), float(np.float32(scale)), int(zero_point), int(quant_min), int(quant_max),
                                   bool(want_rowsum))


def _row_step(kind):
    """The GEMM's row granule: 32 codes for 4-bit codes / indices, else 16."""
    return 32 if kind in (_native.PACK_AFFINE_I4, _native.PACK_LUT_I4) else 16


def linear_code_pitch(in_features, kind):
    """The padded row length of integer linear mode: in_features rounded up to the GEMM's granule (every pad column a
    channel pad: x code zx, counted in K, Sx and Sw)."""
    step = _row_step(kind)
    return -(-int(in_features) // step) * step


def conv_code_pitch(in_channels, kh, kw, kind):
    """(Cp, K): the pixel pitch of the padded NHWC codes and the conv's row length.  Cin <= 4 / <= 8 take the narrow gather
    (Cp = 4 / 8, K = kh*kw*Cp rounded up to the granule: a row tail); wider Cin is rounded up to 16, or to 32 where 4-bit
    codes need kh*kw*Cp % 32 == 0 (K = kh*kw*Cp)."""
    cin, taps, step = int(in_channels), int(kh) * int(kw), _row_step(kind)
    if cin <= 8:
        cp = 4 if cin <= 4 else 8
    else:
        cp = -(-cin // 16) * 16
        if taps * cp % step:
            cp = -(-cin // 32) * 32
    return cp, conv_row_length(cp, kh, kw, kind)


def conv_row_length(cp, kh, kw, kind):
    """The row length mctq_packed_conv2d_i8_padded sums for a pixel pitch cp: kh*kw*cp, rounded up to the granule for the
    narrow gather (cp = 4 / 8)."""
    n, step = int(kh) * int(kw) * int(cp), _row_step(kind)
    return -(-n // step) * step if cp in (4, 8) else n


def quantize_nhwc_i8_padded(x, cp, scale_f32, zero_point, quant_min, quant_max, want_sums):
    """quantize_nhwc_i8 with a channel pitch cp (4, 8 or a multiple of 16, >= C): codes [N, H, W, cp] whose channels
    [C, cp) hold zero_point, P including them.  A channels_last x is quantized as padded rows of pixels
    (mctq_quantize_rows_i8_padded), any other x as NCHW planes (mctq_quantize_nhwc_i8_padded)."""
    if x.dim() != 4:
        raise RuntimeError(f"quantize_nhwc_i8_padded: x must be 4-D [N, C, H, W], got shape {list(x.shape)}")
    N, C, H, W = x.shape
    if not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last):
        return quantize_rows_i8_padded(x.permute(0, 2, 3, 1), cp, scale_f32, zero_point, quant_min, quant_max, want_sums)
    tag = _dtype_tag(x)
    xd = x.contiguous()
    codes = torch.empty((N, H, W, int(cp)), dtype=torch.int8 if quant_min < 0 else torch.uint8, device=xd.device)
    P = torch.empty((N * H * W if want_sums else 0,), dtype=torch.int32, device=xd.device)
    if xd.numel():
        with _on_device(xd.device):
            rc = _native.load().mctq_quantize_nhwc_i8_padded(xd.data_ptr(), tag, N, C, H, W, int(cp), scale_f32, zero_point,
                                                              quant_min, quant_max, codes.data_ptr(),
                                                              _ptr(P) if want_sums else None, _stream(xd.device))
        _native.check(rc, "mctq_quantize_nhwc_i8_padded")
    return codes, P


def _quantize_nhwc_i8_padded_cuda(x, channel_pitch, scale, zero_point, quant_min, quant_max, want_sums):
    _check_range(quant_min, quant_max)
    if not quant_min <= zero_point <= quant_max:
        raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
    return quantize_nhwc_i8_padded(x, int(channel_pitch), float(np.float32(scale)), int(zero_point), int(quant_min),
                                   int(quant_max), bool(want_sums))


def padded_code_rows(codes, kind, is_signed, out_channels, in_channels, kh, kw, channels_last, cp, row):
    """The int32 codes (or LUT indices) of a packed [Cout, Cin, kh, kw] weight (a Linear weight: kh = kw = 1) in (r, s, c)
    order with a channel pitch cp >= Cin and a row of `row` >= kh*kw*cp columns: [Cout][row], channel pads and the row
    tail holding 0.  `channels_last`: the codes are already in (r, s, c) order."""
    qw = weight_code_values(codes, kind, is_signed, out_channels, in_channels * kh * kw)
    qw = qw.reshape(out_channels, kh, kw, in_channels) if channels_last else \
        qw.reshape(out_channels, in_channels, kh, kw).permute(0, 2, 3, 1)
    qw = torch.nn.functional.pad(qw, (0, cp - in_channels)).reshape(out_channels, kh * kw * cp)
    return torch.nn.functional.pad(qw, (0, row - kh * kw * cp)).contiguous()


def pack_code_rows(qw, kind, is_signed, like):
    """pack_weight_codes of int32 code rows, int8 codes viewed as the dtype of the packed tensor `like`."""
    out = pack_weight_codes(qw, kind, is_signed)
    return out.view(like.dtype) if kind == _native.PACK_AFFINE_I8 else out


def weight_code_values(codes, kind, is_signed, out_features, in_features):
    """The integer codes of a packed affine weight (or the indices of a LUT weight: unsigned, 4-bit ones two per byte like
    int4 codes) as an int32 [out_features, in_features] tensor (one-time set-up of IntegerLinear: the code row sums)."""
    c = codes.reshape(-1).view(torch.uint8).to(torch.int32)
    if kind in (_native.PACK_AFFINE_I4, _native.PACK_LUT_I4):
        c = torch.stack((c & 15, c >> 4), dim=-1).reshape(-1)[:out_features * in_features]
        return (c - 16 * (c >= 8).to(torch.int32) if is_signed else c).reshape(out_features, in_features)
    return (c - 256 * (c >= 128).to(torch.int32) if is_signed else c).reshape(out_features, in_features)


class IntegerLinear:
    """Launch state of one packed affine [out_features, in_features] weight in integer linear mode (mctq_quantize_rows_i8 +
    mctq_packed_linear_i8), built once: the descriptor, the weight code row sums Sw, the factors f = fl32(sx * scale) and the
    input quantizer's launch constants.
        codes, kind, is_signed   the packed weight (kind PACK_AFFINE_I8 / PACK_AFFINE_I4), row-major [out][in]
        dtype                    the rebuilt weight's dtype: x, bias and y have it
        scale, zero_point        f32 / int32, 1 (per tensor) or out_features entries
        x_scale, x_zero_point, x_qmin, x_qmax   the input quantizer Q (per tensor, at most 256 levels)
        lut_values               LUT weights (kind PACK_LUT_I4 / PACK_LUT_U8, indices): their int8 centroid codes, a host
                                 tensor or list (mctq_packed_linear_i8_lut); scale is then sw = thr * 2^-(bw-1), zero_point
                                 None (zw = 0), and the codes qw are the table entries of the indices
    `__call__(x, bias)` returns the integer product of Q's codes of x and the weight codes, scaled (include/mctq.h gives the
    formula), for a CUDA x of `dtype` on the codes' device, enqueued on the current stream.  `quantize` and `gemm` are its two
    launches.  `pad=True` admits an in_features off the GEMM's granule (DESIGN §7f): the launch state then holds a copy of
    the codes padded to ldc = linear_code_pitch(in_features, kind) columns, Q's codes have ldc columns whose pads hold zx,
    and the output is that of the same formula over the real row (mctq_packed_linear_i8_padded)."""

    def __init__(self, codes, kind, is_signed, dtype, out_features, in_features, scale, zero_point, x_scale, x_zero_point,
                 x_qmin, x_qmax, lut_values=None, pad=False):
        _check_range(x_qmin, x_qmax)
        if not ((-128 <= x_qmin and x_qmax <= 127) or (0 <= x_qmin and x_qmax <= 255)):
            raise ValueError(f"IntegerLinear: the input range [{x_qmin}, {x_qmax}] does not fit 8-bit codes")
        if not x_qmin <= x_zero_point <= x_qmax:
            raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
        self.device = codes.device
        self.x_scale, self.x_zp = float(np.float32(x_scale)), int(x_zero_point)
        self.x_qmin, self.x_qmax = int(x_qmin), int(x_qmax)
        s = _param_on(scale.detach().reshape(-1).contiguous().to(torch.float32), self.device)
        factor = torch.tensor(self.x_scale, dtype=torch.float32, device=self.device) * s
        ldc = linear_code_pitch(in_features, kind) if pad else int(in_features)
        if ldc != int(in_features):
            qw = padded_code_rows(codes, kind, is_signed, int(out_features), int(in_features), 1, 1, False, ldc, ldc)
            codes = pack_code_rows(qw, kind, is_signed, codes)
        self._bind(codes, kind, is_signed, dtype, out_features, in_features, factor, zero_point, None, "IntegerLinear",
                   lut_values, ldc)

    @classmethod
    def from_parts(cls, codes, kind, is_signed, dtype, out_features, in_features, factor, zero_point, w_rowsum, x_zero_point,
                   lut_values=None, ldc=None):
        """The launch state from a caller-supplied f and Sw (mctq::packed_linear_i8 / _lut; with `ldc`, codes already padded
        to [out][ldc]: mctq::packed_linear_i8_padded), with the constructor's checks of the weight; only `gemm` is available
        (the input quantizer's scale and range are not known)."""
        lin = cls.__new__(cls)
        lin.device = codes.device
        lin.x_zp, lin.x_scale, lin.x_qmin, lin.x_qmax = int(x_zero_point), None, None, None
        what = "packed_linear_i8_padded" if ldc is not None else \
            "packed_linear_i8" if lut_values is None else "packed_linear_i8_lut"
        lin._bind(codes, kind, is_signed, dtype, out_features, in_features, factor, zero_point, w_rowsum, what, lut_values,
                  ldc)
        return lin

    def _bind(self, codes, kind, is_signed, dtype, out_features, in_features, factor, zero_point, w_rowsum, what,
              lut_values=None, ldc=None):
        """Validate the weight, its factors, zero points (LUT weights: the table) and code row sums (computed from the codes
        when None) and build the descriptor.  `ldc`: the codes are [out][ldc] rows whose columns from in_features on are
        channel pads (None: ldc = in_features)."""
        if self.device.type != "cuda":
            raise ValueError(f"{what} needs CUDA tensors")
        lut = lut_code_table(kind, lut_values, what) if lut_values is not None else None
        if lut is None and kind not in (_native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4):
            raise ValueError(f"{what}: kind {kind} is not an affine int8 / int4 packed weight")
        if dtype not in _DT:
            raise ValueError(f"{what}: output dtype {dtype} is not float32 / bfloat16 / float16")
        if zero_point is None and lut is None:
            raise ValueError(f"{what}: affine weights need their zero points")
        self.out_features, self.in_features, self.dtype = int(out_features), int(in_features), dtype
        self.ldc = int(ldc) if ldc is not None else self.in_features
        if self.ldc < self.in_features:
            raise ValueError(f"{what}: a row pitch of {self.ldc} is shorter than in_features = {self.in_features}")
        N, K = self.out_features, self.ldc
        f = _param_on(factor.detach().reshape(-1).contiguous(), self.device)
        nz = f.numel() if lut is not None else zero_point.numel()
        if f.numel() not in (1, N) or nz != f.numel():
            raise ValueError(f"{what}: {f.numel()} factors and {nz} zero points for {N} output channels "
                             f"(both per tensor or both per output channel)")
        C, inner = (f.numel(), K) if f.numel() > 1 else (1, 1)
        # a LUT weight's descriptor carries the table size K and a table pointer, here the codes as f32 (never read)
        self._desc, self._keep = _packed_desc(codes, kind, is_signed, dtype, N * K, C, inner, f,
                                              None if lut is not None else zero_point,
                                              torch.from_numpy(lut.astype(np.float32)) if lut is not None else None,
                                              self.device, what)
        self.factor, z = self._keep[1], self._keep[2]
        self.lut = lut
        if w_rowsum is None:
            qw = weight_code_values(self._keep[0], kind, is_signed, N, K)
            if lut is not None:
                qw = torch.from_numpy(lut.astype(np.int32)).to(self.device)[qw]
            w_rowsum = qw.sum(1, dtype=torch.int32)
        self.w_rowsum = _param_on(w_rowsum.detach().reshape(-1).contiguous(), self.device)
        if self.w_rowsum.dtype != torch.int32 or self.w_rowsum.numel() != N:
            raise ValueError(f"{what}: w_rowsum must be int32 [{N}]")
        self.needs_x_rowsum = lut is None and bool((z != 0).any())
        self._desc_ptr = ctypes.addressof(self._desc)

    def __call__(self, x, bias=None):
        if x.dtype != self.dtype or (bias is not None and bias.dtype != self.dtype):
            raise RuntimeError(f"packed_linear_i8: x and bias must have the weight's dtype {self.dtype}")
        qx, rowsum = self.quantize(x)
        return self.gemm(qx, rowsum if self.needs_x_rowsum else None, bias)

    def quantize(self, x):
        """Q's codes of x and their row sums (empty when no weight zero point needs them)."""
        if x.dim() == 0 or x.shape[-1] != self.in_features:
            raise RuntimeError(f"packed_linear_i8: x of shape {list(x.shape)} does not end in in_features = {self.in_features}")
        if x.device != self.device:
            raise RuntimeError(f"packed_linear_i8: x must live on {self.device}")
        if self.ldc != self.in_features:
            return quantize_rows_i8_padded(x, self.ldc, self.x_scale, self.x_zp, self.x_qmin, self.x_qmax, self.needs_x_rowsum)
        return quantize_rows_i8(x, self.x_scale, self.x_zp, self.x_qmin, self.x_qmax, self.needs_x_rowsum)

    def gemm(self, x_codes, x_rowsum=None, bias=None, out=None):
        """y from x codes [..., in_features] (int8 or uint8, zero point x_zero_point; padded: [..., ldc], the pads holding
        zx) and their row sums.  `out`: a 2-D [M, out_features] CUDA tensor of `dtype` with unit column stride (its rows may
        be further apart) to write into."""
        if x_codes.dtype not in (torch.int8, torch.uint8) or x_codes.dim() == 0 or x_codes.shape[-1] != self.ldc:
            raise RuntimeError(f"packed_linear_i8: x codes ({x_codes.dtype}, {list(x_codes.shape)}) are not int8 / uint8 "
                               f"rows of " + (f"in_features = {self.in_features}" if self.ldc == self.in_features else
                                              f"ldc = {self.ldc} (in_features = {self.in_features}, padded)"))
        if x_codes.device != self.device or (bias is not None and bias.device != self.device):
            raise RuntimeError(f"packed_linear_i8: x codes and bias must live on {self.device}")
        if bias is not None and (bias.numel() != self.out_features or bias.dtype != self.dtype):
            raise RuntimeError(f"packed_linear_i8: bias must hold {self.out_features} entries of {self.dtype}")
        if self.needs_x_rowsum and x_rowsum is None:
            raise RuntimeError("packed_linear_i8: a weight zero point is not 0, so the x code row sums are needed")
        qx = x_codes.contiguous()
        M = qx.numel() // self.ldc
        if out is None:
            y = torch.empty(tuple(qx.shape[:-1]) + (self.out_features,), dtype=self.dtype, device=self.device)
            ldy = self.out_features
        else:
            if out.dim() != 2 or tuple(out.shape) != (M, self.out_features) or out.stride(1) != 1 or out.dtype != self.dtype \
                    or out.device != self.device:
                raise RuntimeError(f"packed_linear_i8: out must be a [{M}, {self.out_features}] {self.dtype} tensor with "
                                   f"unit column stride on {self.device}")
            y, ldy = out, max(out.stride(0), self.out_features)
        if M:
            rs = x_rowsum.reshape(-1).contiguous() if x_rowsum is not None and self.needs_x_rowsum else None
            if rs is not None and (rs.dtype != torch.int32 or rs.numel() != M or rs.device != self.device):
                raise RuntimeError(f"packed_linear_i8: x_rowsum must be int32 [{M}] on {self.device}")
            b = bias.contiguous() if bias is not None else None
            args = (self._desc_ptr, self.out_features, self.in_features, qx.data_ptr(), int(qx.dtype == torch.int8),
                    self.x_zp, M, _ptr(rs), self.w_rowsum.data_ptr(), self.factor.data_ptr(), _ptr(b), _DT[self.dtype],
                    y.data_ptr(), ldy)
            lib = _native.load()
            if self.ldc != self.in_features:
                with _on_device(self.device):
                    rc = lib.mctq_packed_linear_i8_padded(*args[:3], self.ldc, *args[3:],
                                                          self.lut.ctypes.data if self.lut is not None else None,
                                                          _stream(self.device))
                _native.check(rc, "mctq_packed_linear_i8_padded")
                return y
            with _on_device(self.device):
                if self.lut is not None:
                    rc = lib.mctq_packed_linear_i8_lut(*args, self.lut.ctypes.data, _stream(self.device))
                else:
                    rc = lib.mctq_packed_linear_i8(*args, _stream(self.device))
            _native.check(rc, "mctq_packed_linear_i8_lut" if self.lut is not None else "mctq_packed_linear_i8")
        return y


def lut_code_table(kind, lut_values, what):
    """The int8 centroid codes of a LUT weight as a host numpy int8 array (the table mctq_packed_linear_i8_lut /
    mctq_packed_conv2d_i8_lut take by value): 1..16 entries for 4-bit indices, 1..256 for 8-bit ones, integers in
    [-128, 127]."""
    if kind not in _native.PACK_LUT_KINDS:
        raise ValueError(f"{what}: kind {kind} is not a LUT packed weight, but LUT values were given")
    v = np.asarray(lut_values.detach().cpu().numpy() if isinstance(lut_values, torch.Tensor) else lut_values,
                   dtype=np.float64).reshape(-1)
    if not 1 <= v.size <= (16 if kind == _native.PACK_LUT_I4 else 256):
        raise ValueError(f"{what}: {v.size} LUT values for kind {kind}")
    if not (np.all(v == np.round(v)) and np.all(v >= -128) and np.all(v <= 127)):
        raise ValueError(f"{what}: the LUT values are not integers in [-128, 127]")
    return np.ascontiguousarray(v.astype(np.int8))


def _packed_linear_i8_cuda(x_codes, x_zero_point, x_rowsum, codes, kind, is_signed, out_features, zero_point, w_rowsum,
                           factor, bias, dtype):
    """mctq::packed_linear_i8: the caller supplies Sw and f (IntegerLinear derives them from the weight and Q); x_rowsum may
    be None only when every weight zero point is 0."""
    if x_codes.dim() == 0:
        raise RuntimeError("packed_linear_i8: x codes must have at least one dimension")
    _native.load()
    lin = IntegerLinear.from_parts(codes, kind, is_signed, dtype, out_features, x_codes.shape[-1], factor, zero_point,
                                   w_rowsum, x_zero_point)
    return lin.gemm(x_codes, x_rowsum, bias)


def _packed_linear_i8_lut_cuda(x_codes, x_zero_point, codes, kind, out_features, lut_values, w_rowsum, factor, bias):
    """mctq::packed_linear_i8_lut: packed_linear_i8 for LUT indices `codes` with the int8 centroid codes `lut_values` (f32
    output, zw = 0: no x row sums)."""
    if x_codes.dim() == 0:
        raise RuntimeError("packed_linear_i8_lut: x codes must have at least one dimension")
    _native.load()
    lin = IntegerLinear.from_parts(codes, kind, False, torch.float32, out_features, x_codes.shape[-1], factor, None,
                                   w_rowsum, x_zero_point, lut_values)
    return lin.gemm(x_codes, None, bias)


def quantize_nhwc_i8(x, scale_f32, zero_point, quant_min, quant_max, want_sums):
    """(codes, P) of a 4-D CUDA tensor x [N, C, H, W] under a per-tensor 8-bit affine quantizer: codes [N, H, W, C]
    (contiguous, int8 when quant_min < 0 else uint8), exactly the codes mctq_fq_affine_scalar emits, and P int32 [N*H*W]
    (the sum of a pixel's channel codes), or an empty tensor unless `want_sums`.  A channels_last x is quantized as rows of
    pixels (mctq_quantize_rows_i8), any other x as NCHW planes (mctq_quantize_nhwc_i8, after .contiguous() when needed)."""
    if x.dim() != 4:
        raise RuntimeError(f"quantize_nhwc_i8: x must be 4-D [N, C, H, W], got shape {list(x.shape)}")
    N, C, H, W = x.shape
    if not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last):
        codes, P = quantize_rows_i8(x.permute(0, 2, 3, 1), scale_f32, zero_point, quant_min, quant_max, want_sums)
        return codes, P
    tag = _dtype_tag(x)
    xd = x.contiguous()
    codes = torch.empty((N, H, W, C), dtype=torch.int8 if quant_min < 0 else torch.uint8, device=xd.device)
    P = torch.empty((N * H * W if want_sums else 0,), dtype=torch.int32, device=xd.device)
    if xd.numel():
        with _on_device(xd.device):
            rc = _native.load().mctq_quantize_nhwc_i8(xd.data_ptr(), tag, N, C, H, W, scale_f32, zero_point, quant_min,
                                                       quant_max, codes.data_ptr(), _ptr(P) if want_sums else None,
                                                       _stream(xd.device))
        _native.check(rc, "mctq_quantize_nhwc_i8")
    return codes, P


def _quantize_nhwc_i8_cuda(x, scale, zero_point, quant_min, quant_max, want_sums):
    _check_range(quant_min, quant_max)
    if not quant_min <= zero_point <= quant_max:
        raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
    return quantize_nhwc_i8(x, float(np.float32(scale)), int(zero_point), int(quant_min), int(quant_max), bool(want_sums))


def conv_output_hw(H, W, kernel_size, stride, dilation, padding):
    """(Ho, Wo) of a convolution of an H x W image; padding = (pt, pb, pl, pr)."""
    (kh, kw), (sh, sw), (dh, dw), (pt, pb, pl, pr) = kernel_size, stride, dilation, padding
    return (H + pt + pb - dh * (kh - 1) - 1) // sh + 1, (W + pl + pr - dw * (kw - 1) - 1) // sw + 1


def conv_padding(layer):
    """(pt, pb, pl, pr) of a torch.nn.Conv2d, from `_reversed_padding_repeated_twice` ((left, right, top, bottom)): numeric
    padding, 'valid' and the asymmetric 'same'."""
    pl, pr, pt, pb = (int(p) for p in layer._reversed_padding_repeated_twice)
    return pt, pb, pl, pr


def pack_weight_codes(qw, kind, is_signed):
    """Packed codes (int8 / uint8 bytes, or int4 nibbles two per byte, element 2j in the low nibble) of the integer codes
    qw, in qw's element order: the inverse of weight_code_values."""
    q = qw.reshape(-1)
    if kind in (_native.PACK_AFFINE_I4, _native.PACK_LUT_I4):
        u = (q & 15).to(torch.uint8)
        if u.numel() % 2:
            u = torch.cat((u, u.new_zeros(1)))
        u = u.reshape(-1, 2)
        return (u[:, 0] | (u[:, 1] << 4)).contiguous()
    return q.to(torch.int8 if is_signed else torch.uint8).contiguous()


def conv_codes_rsc(codes, kind, is_signed, out_channels, in_channels, kh, kw):
    """The packed codes (or LUT indices) of a contiguous [Cout, Cin, kh, kw] weight ((c, r, s) order per output channel)
    reordered to the (r, s, c) order of mctq_packed_conv2d_i8 (one-time set-up of IntegerConv2d)."""
    qw = weight_code_values(codes, kind, is_signed, out_channels, in_channels * kh * kw)
    qw = qw.reshape(out_channels, in_channels, kh, kw).permute(0, 2, 3, 1)
    out = pack_weight_codes(qw.contiguous(), kind, is_signed)
    return out.view(codes.dtype) if kind == _native.PACK_AFFINE_I8 else out


def conv_window_sums(P, N, H, W, Cin, kernel_size, stride, dilation, padding, x_zero_point):
    """Sx [N*Ho*Wo] (int32) from the per-pixel channel sums P [N*H*W]: the sum of P over each output pixel's window, a tap
    outside the image counting Cin * zx.  Exact int32 torch ops (no host synchronisation, capturable)."""
    (kh, kw), (sh, sw), (dh, dw), (pt, pb, pl, pr) = kernel_size, stride, dilation, padding
    Ho, Wo = conv_output_hw(H, W, kernel_size, stride, dilation, padding)
    p = torch.nn.functional.pad(P.reshape(N, H, W), (pl, pr, pt, pb), value=Cin * int(x_zero_point))
    sx = torch.zeros((N, Ho, Wo), dtype=torch.int32, device=P.device)
    for r in range(kh):
        for s in range(kw):
            sx += p[:, r * dh: r * dh + (Ho - 1) * sh + 1: sh, s * dw: s * dw + (Wo - 1) * sw + 1: sw]
    return sx.reshape(-1)


def _suggests_channels_last(shape, stride):
    from torch._prims_common import suggest_memory_format
    return suggest_memory_format(torch.empty_strided(tuple(shape), tuple(stride), device="meta")) == torch.channels_last


class IntegerConv2d:
    """Launch state of one packed affine Conv2d weight [Cout, Cin, kh, kw] (groups 1, zero padding) in integer convolution
    mode (mctq_quantize_nhwc_i8 + mctq_packed_conv2d_i8), built once, like IntegerLinear: the weight codes in (r, s, c) order,
    the descriptor, Sw, f = fl32(sx * scale), the geometry and the input quantizer's launch constants.
        codes, kind, is_signed   the packed weight (PACK_AFFINE_I8 / PACK_AFFINE_I4)
        weight_stride            the rebuilt weight's strides: contiguous codes are reordered once, channels_last codes
                                 already have the (r, s, c) order and are used as they are
        dtype                    the rebuilt weight's dtype: x, bias and y have it
        kernel_size, stride, dilation   pairs;  padding = (pt, pb, pl, pr)
        scale, zero_point        f32 / int32, 1 (per tensor) or Cout entries
        x_scale, x_zero_point, x_qmin, x_qmax   the input quantizer Q (per tensor, at most 256 levels)
        lut_values               LUT weights (PACK_LUT_I4 / PACK_LUT_U8 indices): their int8 centroid codes, as for
                                 IntegerLinear (mctq_packed_conv2d_i8_lut)
        pad                      admit a Cin off the gather's 16 channels (or a K off 32 for 4-bit codes; DESIGN §7f): the
                                 codes are then copied in (r, s, c) order with a channel pitch Cp = conv_code_pitch(..), Q's
                                 NHWC codes get Cp channels whose pads hold zx (mctq_packed_conv2d_i8_padded)
    `__call__(x, bias)` returns the integer convolution of Q's codes of a 4-D CUDA x of `dtype` on the codes' device with the
    weight codes, scaled (include/mctq.h gives the formula), in the memory format F.conv2d gives for x and the rebuilt
    weight.  `quantize` and `gemm` are its launches."""

    def __init__(self, codes, kind, is_signed, dtype, out_channels, in_channels, kernel_size, weight_stride, stride,
                 dilation, padding, scale, zero_point, x_scale, x_zero_point, x_qmin, x_qmax, lut_values=None, pad=False):
        _check_range(x_qmin, x_qmax)
        if not ((-128 <= x_qmin and x_qmax <= 127) or (0 <= x_qmin and x_qmax <= 255)):
            raise ValueError(f"IntegerConv2d: the input range [{x_qmin}, {x_qmax}] does not fit 8-bit codes")
        if not x_qmin <= x_zero_point <= x_qmax:
            raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
        self.device = codes.device
        self.x_scale, self.x_zp = float(np.float32(x_scale)), int(x_zero_point)
        self.x_qmin, self.x_qmax = int(x_qmin), int(x_qmax)
        kh, kw = (int(k) for k in kernel_size)
        shape = (int(out_channels), int(in_channels), kh, kw)
        self.weight_channels_last = _suggests_channels_last(shape, weight_stride)
        contiguous = tuple(weight_stride) == tuple(torch.empty(shape, device="meta").stride())
        if not contiguous and \
                tuple(weight_stride) != tuple(torch.empty(shape, device="meta").to(memory_format=torch.channels_last).stride()):
            raise ValueError(f"IntegerConv2d: weight strides {tuple(weight_stride)} are neither contiguous nor channels_last")
        cp, row, w_rowsum = None, None, None
        if pad and (shape[1] % 16 or shape[1] * kh * kw % _row_step(kind)):
            # the padded copy in (r, s, c) order; Sw over the counted columns (the narrow gather's row tail is not counted)
            cp, row = conv_code_pitch(shape[1], kh, kw, kind)
            qw = padded_code_rows(codes, kind, is_signed, shape[0], shape[1], kh, kw, not contiguous, cp, row)
            counted = qw[:, :kh * kw * cp]
            if lut_values is not None:
                table = lut_code_table(kind, lut_values, "IntegerConv2d")
                counted = torch.from_numpy(table.astype(np.int32)).to(self.device)[counted]
            w_rowsum = counted.sum(1, dtype=torch.int32)
            codes = pack_code_rows(qw, kind, is_signed, codes)
        elif contiguous:
            codes = conv_codes_rsc(codes, kind, is_signed, *shape)
        s = _param_on(scale.detach().reshape(-1).contiguous().to(torch.float32), self.device)
        factor = torch.tensor(self.x_scale, dtype=torch.float32, device=self.device) * s
        self._bind(codes, kind, is_signed, dtype, shape, stride, dilation, padding, factor, zero_point, w_rowsum,
                   "IntegerConv2d", lut_values, cp)

    @classmethod
    def from_parts(cls, codes, kind, is_signed, dtype, out_channels, in_channels, kernel_size, stride, dilation, padding,
                   factor, zero_point, w_rowsum, x_zero_point, lut_values=None, cp=None):
        """The launch state from caller-supplied (r, s, c)-ordered codes, f and Sw (mctq::packed_conv2d_i8; with `cp`, codes
        already padded to [Cout][conv_row_length(cp, ..)]: mctq::packed_conv2d_i8_padded), with the constructor's checks of
        the weight; only `gemm` is available."""
        conv = cls.__new__(cls)
        conv.device = codes.device
        conv.x_zp, conv.x_scale, conv.x_qmin, conv.x_qmax = int(x_zero_point), None, None, None
        conv.weight_channels_last = False
        shape = (int(out_channels), int(in_channels), int(kernel_size[0]), int(kernel_size[1]))
        what = "packed_conv2d_i8_padded" if cp is not None else \
            "packed_conv2d_i8" if lut_values is None else "packed_conv2d_i8_lut"
        conv._bind(codes, kind, is_signed, dtype, shape, stride, dilation, padding, factor, zero_point, w_rowsum, what,
                   lut_values, cp)
        return conv

    def _bind(self, codes, kind, is_signed, dtype, shape, stride, dilation, padding, factor, zero_point, w_rowsum, what,
              lut_values=None, cp=None):
        if len(stride) != 2 or len(dilation) != 2 or len(padding) != 4:
            raise ValueError(f"{what}: stride and dilation are pairs, padding is (top, bottom, left, right)")
        self.stride, self.dilation = tuple(int(v) for v in stride), tuple(int(v) for v in dilation)
        self.padding = tuple(int(v) for v in padding)
        self.out_channels, self.in_channels = shape[0], shape[1]
        self.kernel_size = shape[2:]
        # cp: the pixel pitch of the x codes (padded: the codes are [Cout][conv_row_length(cp, ..)]; Cin = 4 / 8 keeps
        # cp == Cin but takes the narrow gather)
        self.padded = cp is not None
        self.cp = int(cp) if self.padded else shape[1]
        K = conv_row_length(self.cp, shape[2], shape[3], kind) if cp is not None else shape[1] * shape[2] * shape[3]
        # the weight as a [Cout][K] matrix: IntegerLinear's checks and launch state
        self._w = IntegerLinear.__new__(IntegerLinear)
        self._w.device, self._w.x_zp = self.device, self.x_zp
        self._w._bind(codes, kind, is_signed, dtype, shape[0], K, factor, zero_point, w_rowsum, what, lut_values)
        self.dtype, self.factor, self.w_rowsum = dtype, self._w.factor, self._w.w_rowsum
        self.needs_x_rowsum = self._w.needs_x_rowsum

    def output_hw(self, H, W):
        return conv_output_hw(H, W, self.kernel_size, self.stride, self.dilation, self.padding)

    def __call__(self, x, bias=None):
        if x.dtype != self.dtype or (bias is not None and bias.dtype != self.dtype):
            raise RuntimeError(f"packed_conv2d_i8: x and bias must have the weight's dtype {self.dtype}")
        cl = self.weight_channels_last or _suggests_channels_last(x.shape, x.stride())
        qx, sx = self.quantize(x)
        return self.gemm(qx, sx, bias, channels_last=cl)

    def quantize(self, x):
        """Q's NHWC codes of x and Sx (empty when no weight zero point needs it)."""
        if x.dim() != 4 or x.shape[1] != self.in_channels:
            raise RuntimeError(f"packed_conv2d_i8: x of shape {list(x.shape)} is not [N, {self.in_channels}, H, W]")
        if x.device != self.device:
            raise RuntimeError(f"packed_conv2d_i8: x must live on {self.device}")
        if self.padded:
            qx, P = quantize_nhwc_i8_padded(x, self.cp, self.x_scale, self.x_zp, self.x_qmin, self.x_qmax,
                                            self.needs_x_rowsum)
        else:
            qx, P = quantize_nhwc_i8(x, self.x_scale, self.x_zp, self.x_qmin, self.x_qmax, self.needs_x_rowsum)
        if not self.needs_x_rowsum:
            return qx, None
        N, _, H, W = x.shape
        # the pad channels are channel pads: a tap outside the image counts cp * zx
        return qx, conv_window_sums(P, N, H, W, self.cp, self.kernel_size, self.stride, self.dilation, self.padding,
                                    self.x_zp)

    def gemm(self, x_codes, x_rowsum=None, bias=None, channels_last=False):
        """y [N, Cout, Ho, Wo] from NHWC x codes [N, H, W, Cin] (int8 or uint8, zero point x_zero_point; padded:
        [N, H, W, cp], the pads holding zx) and Sx [N*Ho*Wo]; channels_last: y's memory format (the kernel writes it
        directly)."""
        if x_codes.dtype not in (torch.int8, torch.uint8) or x_codes.dim() != 4 or x_codes.shape[-1] != self.cp:
            raise RuntimeError(f"packed_conv2d_i8: x codes ({x_codes.dtype}, {list(x_codes.shape)}) are not int8 / uint8 "
                               f"NHWC codes of {self.in_channels} channels" +
                               (f" padded to {self.cp}" if self.padded else ""))
        if x_codes.device != self.device or (bias is not None and bias.device != self.device):
            raise RuntimeError(f"packed_conv2d_i8: x codes and bias must live on {self.device}")
        if bias is not None and (bias.numel() != self.out_channels or bias.dtype != self.dtype):
            raise RuntimeError(f"packed_conv2d_i8: bias must hold {self.out_channels} entries of {self.dtype}")
        if self.needs_x_rowsum and x_rowsum is None:
            raise RuntimeError("packed_conv2d_i8: a weight zero point is not 0, so the window code sums Sx are needed")
        qx = x_codes.contiguous()
        N, H, W, _ = qx.shape
        Ho, Wo = self.output_hw(H, W)
        if Ho < 1 or Wo < 1:
            raise RuntimeError(f"packed_conv2d_i8: a {H} x {W} input is smaller than the dilated kernel")
        Cout = self.out_channels
        if channels_last:
            y = torch.empty((N, Ho, Wo, Cout), dtype=self.dtype, device=self.device).permute(0, 3, 1, 2)
        else:
            y = torch.empty((N, Cout, Ho, Wo), dtype=self.dtype, device=self.device)
        M = N * Ho * Wo
        if M:
            rs = x_rowsum.reshape(-1).contiguous() if x_rowsum is not None and self.needs_x_rowsum else None
            if rs is not None and (rs.dtype != torch.int32 or rs.numel() != M or rs.device != self.device):
                raise RuntimeError(f"packed_conv2d_i8: x_rowsum must be int32 [{M}] on {self.device}")
            b = bias.contiguous() if bias is not None else None
            g = _native.MctqConv2dGeom(N, H, W, self.in_channels, Ho, Wo, *self.kernel_size, *self.stride, *self.dilation,
                                       *self.padding)
            args = (self._w._desc_ptr, ctypes.addressof(g), Cout, qx.data_ptr(), int(qx.dtype == torch.int8), self.x_zp,
                    _ptr(rs), self.w_rowsum.data_ptr(), self.factor.data_ptr(), _ptr(b), _DT[self.dtype], y.data_ptr(),
                    0 if channels_last else 1)
            lut = self._w.lut
            lib = _native.load()
            if self.padded:
                with _on_device(self.device):
                    rc = lib.mctq_packed_conv2d_i8_padded(args[0], args[1], self.cp, *args[2:],
                                                          lut.ctypes.data if lut is not None else None, _stream(self.device))
                _native.check(rc, "mctq_packed_conv2d_i8_padded")
                return y
            with _on_device(self.device):
                if lut is not None:
                    rc = lib.mctq_packed_conv2d_i8_lut(*args, lut.ctypes.data, _stream(self.device))
                else:
                    rc = lib.mctq_packed_conv2d_i8(*args, _stream(self.device))
            _native.check(rc, "mctq_packed_conv2d_i8_lut" if lut is not None else "mctq_packed_conv2d_i8")
        return y


def _packed_conv2d_i8_cuda(x_codes, x_zero_point, x_rowsum, codes, kind, is_signed, out_channels, kernel_size, stride,
                           dilation, padding, zero_point, w_rowsum, factor, bias, dtype, channels_last):
    """mctq::packed_conv2d_i8: NHWC x codes, (r, s, c)-ordered weight codes, caller-supplied Sw and f; x_rowsum (Sx) may be
    None only when every weight zero point is 0."""
    if x_codes.dim() != 4:
        raise RuntimeError("packed_conv2d_i8: x codes must be 4-D NHWC")
    if len(kernel_size) != 2:
        raise ValueError("packed_conv2d_i8: kernel_size is a pair")
    _native.load()
    conv = IntegerConv2d.from_parts(codes, kind, is_signed, dtype, out_channels, x_codes.shape[-1], kernel_size, stride,
                                    dilation, padding, factor, zero_point, w_rowsum, x_zero_point)
    return conv.gemm(x_codes, x_rowsum, bias, channels_last)


def _packed_conv2d_i8_lut_cuda(x_codes, x_zero_point, codes, kind, out_channels, kernel_size, stride, dilation, padding,
                               lut_values, w_rowsum, factor, bias, channels_last):
    """mctq::packed_conv2d_i8_lut: packed_conv2d_i8 for (r, s, c)-ordered LUT indices with the int8 centroid codes
    `lut_values` (f32 output, zw = 0: no window code sums)."""
    if x_codes.dim() != 4:
        raise RuntimeError("packed_conv2d_i8_lut: x codes must be 4-D NHWC")
    if len(kernel_size) != 2:
        raise ValueError("packed_conv2d_i8_lut: kernel_size is a pair")
    _native.load()
    conv = IntegerConv2d.from_parts(codes, kind, False, torch.float32, out_channels, x_codes.shape[-1], kernel_size, stride,
                                    dilation, padding, factor, None, w_rowsum, x_zero_point, lut_values)
    return conv.gemm(x_codes, None, bias, channels_last)


def _packed_linear_i8_padded_cuda(x_codes, in_features, x_zero_point, x_rowsum, codes, kind, is_signed, out_features,
                                  zero_point, w_rowsum, factor, bias, dtype, lut_values):
    """mctq::packed_linear_i8_padded: x codes [..., ldc] whose columns from in_features on hold zx, codes [out][ldc] (affine
    with zero_point, or LUT indices with `lut_values` and f32 output), caller-supplied Sw over the ldc columns and f."""
    if x_codes.dim() == 0:
        raise RuntimeError("packed_linear_i8_padded: x codes must have at least one dimension")
    _native.load()
    lut = lut_values is not None
    lin = IntegerLinear.from_parts(codes, kind, False if lut else is_signed, torch.float32 if lut else dtype, out_features,
                                   in_features, factor, None if lut else zero_point, w_rowsum, x_zero_point, lut_values,
                                   ldc=x_codes.shape[-1])
    return lin.gemm(x_codes, None if lut else x_rowsum, bias)


def _packed_conv2d_i8_padded_cuda(x_codes, in_channels, x_zero_point, x_rowsum, codes, kind, is_signed, out_channels,
                                  kernel_size, stride, dilation, padding, zero_point, w_rowsum, factor, bias, dtype,
                                  channels_last, lut_values):
    """mctq::packed_conv2d_i8_padded: NHWC x codes [N, H, W, cp] whose channels from in_channels on hold zx, codes
    [Cout][conv_row_length(cp, ..)] in (r, s, c) order (affine with zero_point, or LUT indices with `lut_values` and f32
    output), caller-supplied Sw over the counted columns and f."""
    if x_codes.dim() != 4:
        raise RuntimeError("packed_conv2d_i8_padded: x codes must be 4-D NHWC")
    if len(kernel_size) != 2:
        raise ValueError("packed_conv2d_i8_padded: kernel_size is a pair")
    _native.load()
    lut = lut_values is not None
    conv = IntegerConv2d.from_parts(codes, kind, False if lut else is_signed, torch.float32 if lut else dtype, out_channels,
                                    in_channels, kernel_size, stride, dilation, padding, factor,
                                    None if lut else zero_point, w_rowsum, x_zero_point, lut_values, cp=x_codes.shape[-1])
    return conv.gemm(x_codes, None if lut else x_rowsum, bias, channels_last)


class IntegerDepthwiseConv2d:
    """Launch state of one packed depthwise Conv2d weight [Cout, 1, kh, kw] (groups = in_channels, Cout a multiple of it) in
    integer convolution mode (mctq_packed_dwconv2d_i8), built once: the descriptor of the weight as a [Cout][kh*kw] matrix,
    f = fl32(sx * scale), the geometry and the input quantizer's launch constants.  The arguments are IntegerConv2d's; the
    codes are used as they are (a contiguous and a channels_last [Cout, 1, kh, kw] weight have the same memory order).
    `__call__(x, bias)` returns the depthwise convolution of Q's codes of a 4-D CUDA x of `dtype` on the codes' device with
    the weight codes, scaled (include/mctq.h gives the formula), in the memory format F.conv2d gives for x and the rebuilt
    weight.  The kernel reads x itself and computes Q's codes in registers: one launch, no code tensor."""

    def __init__(self, codes, kind, is_signed, dtype, out_channels, in_channels, kernel_size, weight_stride, stride,
                 dilation, padding, scale, zero_point, x_scale, x_zero_point, x_qmin, x_qmax, lut_values=None):
        shape = (int(out_channels), 1, int(kernel_size[0]), int(kernel_size[1]))
        self.weight_channels_last = _suggests_channels_last(shape, weight_stride)
        dense = torch.empty(shape, device="meta")
        if tuple(weight_stride) not in (dense.stride(), dense.to(memory_format=torch.channels_last).stride()):
            raise ValueError(f"IntegerDepthwiseConv2d: weight strides {tuple(weight_stride)} are neither contiguous nor "
                             f"channels_last")
        s = _param_on(scale.detach().reshape(-1).contiguous().to(torch.float32), codes.device)
        factor = torch.tensor(float(np.float32(x_scale)), dtype=torch.float32, device=codes.device) * s
        self._bind(codes, kind, is_signed, dtype, shape[0], in_channels, shape[2:], stride, dilation, padding, factor,
                   zero_point, x_scale, x_zero_point, x_qmin, x_qmax, "IntegerDepthwiseConv2d", lut_values)

    @classmethod
    def from_parts(cls, codes, kind, is_signed, dtype, out_channels, in_channels, kernel_size, stride, dilation, padding,
                   factor, zero_point, x_scale, x_zero_point, x_qmin, x_qmax, lut_values=None):
        """The launch state from caller-supplied [Cout][kh*kw] codes and f (mctq::packed_dwconv2d_i8)."""
        conv = cls.__new__(cls)
        conv.weight_channels_last = False
        conv._bind(codes, kind, is_signed, dtype, out_channels, in_channels, kernel_size, stride, dilation, padding, factor,
                   zero_point, x_scale, x_zero_point, x_qmin, x_qmax, "packed_dwconv2d_i8", lut_values)
        return conv

    def _bind(self, codes, kind, is_signed, dtype, out_channels, in_channels, kernel_size, stride, dilation, padding, factor,
              zero_point, x_scale, x_zero_point, x_qmin, x_qmax, what, lut_values):
        _check_range(x_qmin, x_qmax)
        if not ((-128 <= x_qmin and x_qmax <= 127) or (0 <= x_qmin and x_qmax <= 255)):
            raise ValueError(f"{what}: the input range [{x_qmin}, {x_qmax}] does not fit 8-bit codes")
        if not x_qmin <= x_zero_point <= x_qmax:
            raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
        if len(kernel_size) != 2 or len(stride) != 2 or len(dilation) != 2 or len(padding) != 4:
            raise ValueError(f"{what}: kernel_size, stride and dilation are pairs, padding is (top, bottom, left, right)")
        self.out_channels, self.in_channels = int(out_channels), int(in_channels)
        if self.in_channels < 1 or self.out_channels % self.in_channels:
            raise ValueError(f"{what}: out_channels = {out_channels} is not a multiple of in_channels = {in_channels}")
        self.device = codes.device
        self.x_scale, self.x_zp = float(np.float32(x_scale)), int(x_zero_point)
        self.x_qmin, self.x_qmax = int(x_qmin), int(x_qmax)
        self.kernel_size = tuple(int(k) for k in kernel_size)
        self.stride, self.dilation = tuple(int(v) for v in stride), tuple(int(v) for v in dilation)
        self.padding = tuple(int(v) for v in padding)
        # the weight as a [Cout][kh * kw] matrix: IntegerLinear's checks and descriptor
        self._w = IntegerLinear.__new__(IntegerLinear)
        self._w.device, self._w.x_zp = self.device, self.x_zp
        self._w._bind(codes, kind, is_signed, dtype, self.out_channels, self.kernel_size[0] * self.kernel_size[1], factor,
                      zero_point, torch.zeros(self.out_channels, dtype=torch.int32), what, lut_values)
        self.dtype, self.factor = dtype, self._w.factor

    def output_hw(self, H, W):
        return conv_output_hw(H, W, self.kernel_size, self.stride, self.dilation, self.padding)

    def __call__(self, x, bias=None):
        return self.conv(x, bias, self.weight_channels_last or _suggests_channels_last(x.shape, x.stride()))

    def conv(self, x, bias=None, channels_last=False):
        """y [N, Cout, Ho, Wo] of x [N, in_channels, H, W]; channels_last: the layout of y, and of x in the kernel (x is
        converted when it has another one, which changes no value)."""
        if x.dtype != self.dtype or (bias is not None and bias.dtype != self.dtype):
            raise RuntimeError(f"packed_dwconv2d_i8: x and bias must have the weight's dtype {self.dtype}")
        if x.dim() != 4 or x.shape[1] != self.in_channels:
            raise RuntimeError(f"packed_dwconv2d_i8: x of shape {list(x.shape)} is not [N, {self.in_channels}, H, W]")
        if x.device != self.device or (bias is not None and bias.device != self.device):
            raise RuntimeError(f"packed_dwconv2d_i8: x and bias must live on {self.device}")
        if bias is not None and bias.numel() != self.out_channels:
            raise RuntimeError(f"packed_dwconv2d_i8: bias must hold {self.out_channels} entries of {self.dtype}")
        fmt = torch.channels_last if channels_last else torch.contiguous_format
        if not x.is_contiguous(memory_format=fmt):
            x = x.contiguous(memory_format=fmt)
        N, _, H, W = x.shape
        Ho, Wo = self.output_hw(H, W)
        if Ho < 1 or Wo < 1:
            raise RuntimeError(f"packed_dwconv2d_i8: a {H} x {W} input is smaller than the dilated kernel")
        Cout = self.out_channels
        if channels_last:
            y = torch.empty((N, Ho, Wo, Cout), dtype=self.dtype, device=self.device).permute(0, 3, 1, 2)
        else:
            y = torch.empty((N, Cout, Ho, Wo), dtype=self.dtype, device=self.device)
        if y.numel():
            b = bias.contiguous() if bias is not None else None
            g = _native.MctqConv2dGeom(N, H, W, self.in_channels, Ho, Wo, *self.kernel_size, *self.stride, *self.dilation,
                                       *self.padding)
            lut = self._w.lut
            with _on_device(self.device):
                rc = _native.load().mctq_packed_dwconv2d_i8(
                    self._w._desc_ptr, ctypes.addressof(g), Cout, x.data_ptr(), _DT[self.dtype], int(bool(channels_last)),
                    self.x_scale, self.x_zp, self.x_qmin, self.x_qmax, self.factor.data_ptr(), _ptr(b), y.data_ptr(),
                    lut.ctypes.data if lut is not None else None, _stream(self.device))
            _native.check(rc, "mctq_packed_dwconv2d_i8")
        return y


def dwconv_plan(N, C, H, W, out_channels, kernel_size, stride, dilation, padding, channels_last=False):
    """The tile plan mctq_packed_dwconv2d_i8 launches for x [N, C, H, W] (mctq_packed_dwconv2d_i8_plan, host only): a dict
    of S (slots per work unit), TH x TW (output tile), IH x IW (window tile) and smem_bytes, or None when the dilated window
    does not fit the kernel's shared memory even for one output of one channel (the launch returns MCTQ_E_RANGE)."""
    Ho, Wo = conv_output_hw(H, W, kernel_size, stride, dilation, padding)
    g = _native.MctqConv2dGeom(N, H, W, C, Ho, Wo, *kernel_size, *stride, *dilation, *padding)
    plan = _native.MctqDwPlan()
    rc = _native.load().mctq_packed_dwconv2d_i8_plan(ctypes.addressof(g), out_channels, int(bool(channels_last)),
                                                     ctypes.addressof(plan))
    if rc == -3:                                                 # MCTQ_E_RANGE
        return None
    _native.check(rc, "mctq_packed_dwconv2d_i8_plan")
    return {f: getattr(plan, f) for f, _ in _native.MctqDwPlan._fields_}


def _packed_dwconv2d_i8_cuda(x, x_scale, x_zero_point, x_qmin, x_qmax, codes, kind, is_signed, out_channels, kernel_size,
                             stride, dilation, padding, zero_point, factor, lut_values, bias, channels_last):
    """mctq::packed_dwconv2d_i8: the [Cout][kh*kw] weight codes (or LUT indices with their int8 centroid codes
    `lut_values`) and f supplied by the caller; y in x's dtype, channels_last or NCHW."""
    if x.dim() != 4:
        raise RuntimeError("packed_dwconv2d_i8: x must be 4-D [N, C, H, W]")
    _native.load()
    conv = IntegerDepthwiseConv2d.from_parts(codes, kind, is_signed, x.dtype, out_channels, x.shape[1], kernel_size, stride,
                                             dilation, padding, factor, zero_point, x_scale, x_zero_point, x_qmin, x_qmax,
                                             lut_values)
    return conv.conv(x, bias, channels_last)


def _lut_scalar_cuda(x, table, K, divisor, threshold, round_to_input_dtype, multiply=False):
    """`multiply`: normalise with x * (float)(1.0 / divisor) -- the reference's CUDA flavour of `tensor / python_number`
    (quantizer_utils.reference_arithmetic) -- instead of the true division x / (float)divisor."""
    _dtype_tag(x)
    xd = x.contiguous()        # the reference's eager composition (argmin + gather) returns a row-major tensor whatever x's strides
    y = torch.empty_like(xd, dtype=torch.float32)
    if xd.numel():
        if multiply:
            _lut_launch(xd, y, None, 0, table, K, 1, 1, None, 0.0, 2, float(np.float32(1.0 / divisor)), threshold, round_to_input_dtype)
        else:
            _lut_launch(xd, y, None, 0, table, K, 1, 1, None, 0.0, 1, divisor, threshold, round_to_input_dtype)
    return y


class private_stream:
    """Context manager for back-to-back calls on tensors that ALREADY EXIST (per-layer weight quantization of a model,
    sweeps over recorded activations): inside the block consecutive launches of this package on a stream may OVERLAP.  A
    launch whose buffers are disjoint from those of every launch still in flight does not wait for its predecessor at all
    (at most two such launches in a row), one whose input is merely not produced by a launch in flight issues its loads
    before it waits -- the drain of one kernel and the ramp of the next disappear (programmatic dependent launch, orders
    "free" and "early" in csrc/mctq_common.cuh; every dependency between this package's own launches is detected from
    their address ranges and honoured).

    The caller guarantees that, inside the block, the streams used carry NO OTHER work than this package's calls: the
    library cannot see foreign kernels (a cuDNN kernel may release its dependents before its stores are visible; the
    caching allocator may recycle a foreign kernel's input buffer as one of our outputs).  Entering and leaving the block
    make the next launch on every stream wait for everything before it.  Process-wide setting."""

    def __enter__(self):
        self._prev = _native.load().mctq_set_tuning(3, 3)
        return self

    def __exit__(self, *exc):
        _native.load().mctq_set_tuning(3, self._prev)
        return False


# --------------------------------------------------------------------------------------------- CPU-tensor impls
# A host tensor is streamed through the GPU in chunks (pinned memory overlaps copies and kernels).
class host_pipeline:
    """Context manager: quantizer / holder / wrapper calls on HOST (pinned) tensors inside the block are only
    *enqueued* -- their results are complete when the block exits.  The H2D -> kernel -> D2H pipeline then keeps
    running across the tensors of a model instead of filling and draining once per call (mctq_host_set_deferred /
    mctq_host_wait).  Inputs must not be modified inside the block; the block keeps them (and the outputs) alive.

        with mct_quantizers_b200.host_pipeline():
            outs = [holder(x) for holder, x in zip(holders, pinned_host_tensors)]
        # outs are complete here
    """
    _active = {}          # device index -> innermost active scope

    def __init__(self, device=None):
        self._device = device
        self._keep = []
        self._outer = None

    def __enter__(self):
        dev = _require_cuda_for_host_path() if self._device is None else torch.device(self._device).index
        self._dev = dev
        self._outer = host_pipeline._active.get(dev)
        if self._outer is None:
            _native.check(_native.load().mctq_host_set_deferred(dev, 1), "mctq_host_set_deferred")
        host_pipeline._active[dev] = self
        return self

    def wait(self):
        """Complete everything enqueued so far (the block stays deferred)."""
        _native.check(_native.load().mctq_host_wait(self._dev), "mctq_host_wait")
        self._keep.clear()

    def __exit__(self, *exc):
        try:
            if self._outer is None:
                _native.check(_native.load().mctq_host_set_deferred(self._dev, 0), "mctq_host_set_deferred")   # waits
            else:
                self.wait()
        finally:
            self._keep.clear()
            if self._outer is None:
                host_pipeline._active.pop(self._dev, None)
            else:
                host_pipeline._active[self._dev] = self._outer
        return False


def _host_keepalive(dev, *tensors):
    scope = host_pipeline._active.get(dev)
    if scope is not None:
        scope._keep.extend(tensors)


def _affine_host(x, scale_np, zp_np, C, inner, quant_min, quant_max):
    dev = _require_cuda_for_host_path()
    tag = _dtype_tag(x)
    xc = x.contiguous()
    y = torch.empty_like(xc, pin_memory=xc.is_pinned())
    if xc.numel():
        lib = _native.load()
        stg = _staging_buffer(dev)
        rc = lib.mctq_fq_affine_host(_ptr(xc), _ptr(y), xc.numel(), tag, scale_np.ctypes.data_as(c_vp),
                                     zp_np.ctypes.data_as(c_vp), C, inner, int(quant_min), int(quant_max),
                                     _ptr(stg), stg.numel(), dev)
        _native.check(rc, "mctq_fq_affine_host")
        _host_keepalive(dev, xc, y)
    return y


def _affine_scalar_cpu(x, scale, zero_point, quant_min, quant_max):
    _check_range(quant_min, quant_max)
    if not quant_min <= zero_point <= quant_max:
        raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
    return _affine_host(x, np.array([scale], dtype=np.float64).astype(np.float32), np.array([zero_point], dtype=np.int32),
                        1, 1, quant_min, quant_max)


def _affine_tensor_cpu(x, scale, zero_point, quant_min, quant_max):
    _check_range(quant_min, quant_max)
    if scale.numel() != 1 or zero_point.numel() != 1:
        raise RuntimeError(f"a Tensor with {max(scale.numel(), zero_point.numel())} elements cannot be converted to Scalar")
    return _affine_host(x, _host_array(scale, np.float32), _host_array(zero_point, np.int32), 1, 1, quant_min, quant_max)


def _affine_channel_cpu(x, scale, zero_point, axis, quant_min, quant_max):
    _check_range(quant_min, quant_max)
    _check_channel_params(x, scale, zero_point, axis)
    xc = x.contiguous()
    _, C, inner = _channel_layout(xc, axis)
    return _affine_host(xc, _host_array(scale, np.float32), _host_array(zero_point, np.int32), C, inner,
                        quant_min, quant_max)


def _lut_host(x, table, K, thr_np, C, inner, eps, scalar_mode, divisor, thr_f32, round_flag):
    dev = _require_cuda_for_host_path()
    tag = _dtype_tag(x)
    xc = x.contiguous()
    y = torch.empty(xc.shape, dtype=torch.float32, pin_memory=xc.is_pinned())
    if xc.numel():
        lib = _native.load()
        stg = _staging_buffer(dev)
        tab = table.detach().cpu().contiguous()
        rc = lib.mctq_fq_lut_host(_ptr(xc), _ptr(y), xc.numel(), tag, _ptr(tab), int(K),
                                  thr_np.ctypes.data_as(c_vp) if thr_np is not None else None, C, inner,
                                  float(np.float32(eps)), int(scalar_mode), float(np.float32(divisor)),
                                  float(np.float32(thr_f32)), int(round_flag), _ptr(stg), stg.numel(), dev)
        _native.check(rc, "mctq_fq_lut_host")
        _host_keepalive(dev, xc, y)
    return y


def _lut_tensor_cpu(x, table, K, threshold, per_channel, axis, eps):
    xc = x.contiguous()
    if per_channel:
        if threshold.numel() != xc.shape[axis]:
            raise RuntimeError("threshold length does not match the channel axis")
        _, C, inner = _channel_layout(xc, axis)
    else:
        C, inner = 1, 1
    return _lut_host(xc, table, K, _host_array(threshold, np.float32), C, inner, eps, 0, 1.0, 1.0, 0)


def _lut_scalar_cpu(x, table, K, divisor, threshold, round_to_input_dtype, multiply=False):
    # host tensors: the reference would run libtorch's CPU kernels, i.e. a true division, whatever `multiply` says
    return _lut_host(x, table, K, None, 1, 1, 0.0, 1, divisor, threshold, round_to_input_dtype)


def _via_device(cuda_impl, keep=()):
    """Host-tensor implementation of the operators that have no chunked host pipeline of their own (integer codes, LUT
    indices, dequantization, the producer-fused holder): every tensor argument is copied to the current CUDA device, the
    device operator runs there and the results come back as host tensors.  Codes are the cheap direction of this trip:
    one byte (or a nibble) per element returns instead of four.  `keep`: positions of tensor arguments that stay on the
    host (the LUT search table is host data by contract)."""
    def impl(*args):
        dev = torch.device("cuda", _require_cuda_for_host_path())

        def up(a):
            if isinstance(a, torch.Tensor) and not a.is_cuda:
                return a.to(dev, non_blocking=a.is_pinned())
            return a

        out = cuda_impl(*[a if k in keep else up(a) for k, a in enumerate(args)])
        if isinstance(out, (tuple, list)):
            return type(out)(o.cpu() if isinstance(o, torch.Tensor) else o for o in out)
        return out.cpu() if isinstance(out, torch.Tensor) else out
    return impl


_LIB.impl("fq_affine_scalar", _affine_scalar_cuda, "CUDA")
_LIB.impl("fq_affine_tensor", _affine_tensor_cuda, "CUDA")
_LIB.impl("fq_affine_channel", _affine_channel_cuda, "CUDA")
_LIB.impl("fq_lut_tensor", _lut_tensor_cuda, "CUDA")
_LIB.impl("fq_lut_scalar", _lut_scalar_cuda, "CUDA")
_LIB.impl("quantize_affine_channel", _quantize_affine_channel_cuda, "CUDA")
_LIB.impl("dequantize_affine", _dequantize_affine_cuda, "CUDA")
_LIB.impl("lut_indices", _lut_indices_cuda, "CUDA")
_LIB.impl("dequantize_lut", _dequantize_lut_cuda, "CUDA")
_LIB.impl("packed_linear", _packed_linear_cuda, "CUDA")
_LIB.impl("packed_linear_batched", _packed_linear_batched_cuda, "CUDA")
_LIB.impl("quantize_rows_i8", _quantize_rows_i8_cuda, "CUDA")
_LIB.impl("packed_linear_i8", _packed_linear_i8_cuda, "CUDA")
_LIB.impl("quantize_nhwc_i8", _quantize_nhwc_i8_cuda, "CUDA")
_LIB.impl("packed_conv2d_i8", _packed_conv2d_i8_cuda, "CUDA")
_LIB.impl("packed_linear_i8_lut", _packed_linear_i8_lut_cuda, "CUDA")
_LIB.impl("packed_conv2d_i8_lut", _packed_conv2d_i8_lut_cuda, "CUDA")
_LIB.impl("packed_dwconv2d_i8", _packed_dwconv2d_i8_cuda, "CUDA")
_LIB.impl("quantize_rows_i8_padded", _quantize_rows_i8_padded_cuda, "CUDA")
_LIB.impl("quantize_nhwc_i8_padded", _quantize_nhwc_i8_padded_cuda, "CUDA")
_LIB.impl("packed_linear_i8_padded", _packed_linear_i8_padded_cuda, "CUDA")
_LIB.impl("packed_conv2d_i8_padded", _packed_conv2d_i8_padded_cuda, "CUDA")

_LIB.impl("fq_affine_scalar_pre", _affine_scalar_pre_cuda, "CUDA")
_LIB.impl("fq_affine_scalar_pre", _via_device(_affine_scalar_pre_cuda), "CPU")
_LIB.impl("fq_affine_scalar", _affine_scalar_cpu, "CPU")
_LIB.impl("fq_affine_tensor", _affine_tensor_cpu, "CPU")
_LIB.impl("fq_affine_channel", _affine_channel_cpu, "CPU")
_LIB.impl("fq_lut_tensor", _lut_tensor_cpu, "CPU")
_LIB.impl("fq_lut_scalar", _lut_scalar_cpu, "CPU")
_LIB.impl("quantize_affine_channel", _via_device(_quantize_affine_channel_cuda), "CPU")
_LIB.impl("dequantize_affine", _via_device(_dequantize_affine_cuda), "CPU")
_LIB.impl("lut_indices", _via_device(_lut_indices_cuda, keep=(1,)), "CPU")
_LIB.impl("dequantize_lut", _via_device(_dequantize_lut_cuda, keep=(3,)), "CPU")
_LIB.impl("packed_linear", _via_device(_packed_linear_cuda), "CPU")
_LIB.impl("packed_linear_batched", _via_device(_packed_linear_batched_cuda), "CPU")
_LIB.impl("quantize_rows_i8", _via_device(_quantize_rows_i8_cuda), "CPU")
_LIB.impl("packed_linear_i8", _via_device(_packed_linear_i8_cuda), "CPU")
_LIB.impl("quantize_nhwc_i8", _via_device(_quantize_nhwc_i8_cuda), "CPU")
_LIB.impl("packed_conv2d_i8", _via_device(_packed_conv2d_i8_cuda), "CPU")
_LIB.impl("packed_linear_i8_lut", _via_device(_packed_linear_i8_lut_cuda), "CPU")
_LIB.impl("packed_conv2d_i8_lut", _via_device(_packed_conv2d_i8_lut_cuda), "CPU")
_LIB.impl("packed_dwconv2d_i8", _via_device(_packed_dwconv2d_i8_cuda, keep=(15,)), "CPU")
_LIB.impl("quantize_rows_i8_padded", _via_device(_quantize_rows_i8_padded_cuda), "CPU")
_LIB.impl("quantize_nhwc_i8_padded", _via_device(_quantize_nhwc_i8_padded_cuda), "CPU")
_LIB.impl("packed_linear_i8_padded", _via_device(_packed_linear_i8_padded_cuda), "CPU")
_LIB.impl("packed_conv2d_i8_padded", _via_device(_packed_conv2d_i8_padded_cuda), "CPU")


# --------------------------------------------------------------------------------------------- fake / meta impls
@torch.library.register_fake("mctq::fq_affine_scalar")
def _(x, scale, zero_point, quant_min, quant_max):
    return torch.empty_like(x)


@torch.library.register_fake("mctq::fq_affine_scalar_pre")
def _(x, other, pre_op, scale, zero_point, quant_min, quant_max):
    return torch.empty_like(x)


@torch.library.register_fake("mctq::fq_affine_tensor")
def _(x, scale, zero_point, quant_min, quant_max):
    return torch.empty_like(x)


@torch.library.register_fake("mctq::fq_affine_channel")
def _(x, scale, zero_point, axis, quant_min, quant_max):
    return torch.empty_like(x)


@torch.library.register_fake("mctq::fq_lut_tensor")
def _(x, table, K, threshold, per_channel, axis, eps):
    return torch.empty_like(x, dtype=torch.float32)


@torch.library.register_fake("mctq::fq_lut_scalar")
def _(x, table, K, divisor, threshold, round_to_input_dtype, multiply=False):
    return torch.empty_like(x, dtype=torch.float32)


@torch.library.register_fake("mctq::quantize_affine_channel")
def _(x, scale, zero_point, axis, quant_min, quant_max, code_mode, want_values):
    if code_mode == _native.CODES_INT4:
        codes = x.new_empty(((x.numel() + 1) // 2,), dtype=torch.uint8)
    else:
        codes = torch.empty_like(x, dtype=torch.int8 if quant_min < 0 else torch.uint8)
    return codes, (torch.empty_like(x) if want_values else x.new_empty((0,)))


@torch.library.register_fake("mctq::dequantize_affine")
def _(codes, code_mode, is_signed, shape, scale, zero_point, axis):
    return codes.new_empty(list(shape), dtype=torch.float32)


@torch.library.register_fake("mctq::lut_indices")
def _(x, table, K, threshold, per_channel, axis, eps, idx_mode):
    if idx_mode == _native.CODES_INT4:
        return x.new_empty(((x.numel() + 1) // 2,), dtype=torch.uint8)
    return torch.empty_like(x, dtype=torch.uint8)


@torch.library.register_fake("mctq::dequantize_lut")
def _(idx, idx_mode, shape, lut, lut_values_bitwidth, is_signed, threshold, per_channel, axis):
    return idx.new_empty(list(shape) if len(shape) else [1], dtype=torch.float32)


@torch.library.register_fake("mctq::packed_linear")
def _(x, codes, kind, is_signed, out_features, scale, zero_point, lut_quotients, bias):
    return x.new_empty(tuple(x.shape[:-1]) + (out_features,))


@torch.library.register_fake("mctq::packed_linear_batched")
def _(x, codes, kind, is_signed, out_features, scale, zero_point, lut_quotients, bias):
    return x.new_empty(tuple(x.shape[:-1]) + (out_features,))


@torch.library.register_fake("mctq::quantize_rows_i8")
def _(x, scale, zero_point, quant_min, quant_max, want_rowsum):
    M = x.numel() // x.shape[-1] if x.dim() and x.shape[-1] else 0
    return (torch.empty_like(x, dtype=torch.int8 if quant_min < 0 else torch.uint8),
            x.new_empty((M if want_rowsum else 0,), dtype=torch.int32))


@torch.library.register_fake("mctq::packed_linear_i8")
def _(x_codes, x_zero_point, x_rowsum, codes, kind, is_signed, out_features, zero_point, w_rowsum, factor, bias, dtype):
    return x_codes.new_empty(tuple(x_codes.shape[:-1]) + (out_features,), dtype=dtype)


@torch.library.register_fake("mctq::quantize_nhwc_i8")
def _(x, scale, zero_point, quant_min, quant_max, want_sums):
    N, C, H, W = x.shape
    return (x.new_empty((N, H, W, C), dtype=torch.int8 if quant_min < 0 else torch.uint8),
            x.new_empty((N * H * W if want_sums else 0,), dtype=torch.int32))


@torch.library.register_fake("mctq::packed_conv2d_i8")
def _(x_codes, x_zero_point, x_rowsum, codes, kind, is_signed, out_channels, kernel_size, stride, dilation, padding,
      zero_point, w_rowsum, factor, bias, dtype, channels_last):
    N, H, W, _ = x_codes.shape
    Ho, Wo = conv_output_hw(H, W, kernel_size, stride, dilation, padding)
    if channels_last:
        return x_codes.new_empty((N, Ho, Wo, out_channels), dtype=dtype).permute(0, 3, 1, 2)
    return x_codes.new_empty((N, out_channels, Ho, Wo), dtype=dtype)


@torch.library.register_fake("mctq::packed_linear_i8_lut")
def _(x_codes, x_zero_point, codes, kind, out_features, lut_values, w_rowsum, factor, bias):
    return x_codes.new_empty(tuple(x_codes.shape[:-1]) + (out_features,), dtype=torch.float32)


@torch.library.register_fake("mctq::packed_conv2d_i8_lut")
def _(x_codes, x_zero_point, codes, kind, out_channels, kernel_size, stride, dilation, padding, lut_values, w_rowsum, factor,
      bias, channels_last):
    N, H, W, _ = x_codes.shape
    Ho, Wo = conv_output_hw(H, W, kernel_size, stride, dilation, padding)
    if channels_last:
        return x_codes.new_empty((N, Ho, Wo, out_channels), dtype=torch.float32).permute(0, 3, 1, 2)
    return x_codes.new_empty((N, out_channels, Ho, Wo), dtype=torch.float32)


@torch.library.register_fake("mctq::packed_dwconv2d_i8")
def _(x, x_scale, x_zero_point, x_qmin, x_qmax, codes, kind, is_signed, out_channels, kernel_size, stride, dilation, padding,
      zero_point, factor, lut_values, bias, channels_last):
    N, _, H, W = x.shape
    Ho, Wo = conv_output_hw(H, W, kernel_size, stride, dilation, padding)
    if channels_last:
        return x.new_empty((N, Ho, Wo, out_channels)).permute(0, 3, 1, 2)
    return x.new_empty((N, out_channels, Ho, Wo))


@torch.library.register_fake("mctq::quantize_rows_i8_padded")
def _(x, ldc, scale, zero_point, quant_min, quant_max, want_rowsum):
    M = x.numel() // x.shape[-1] if x.dim() and x.shape[-1] else 0
    return (x.new_empty(tuple(x.shape[:-1]) + (ldc,), dtype=torch.int8 if quant_min < 0 else torch.uint8),
            x.new_empty((M if want_rowsum else 0,), dtype=torch.int32))


@torch.library.register_fake("mctq::quantize_nhwc_i8_padded")
def _(x, channel_pitch, scale, zero_point, quant_min, quant_max, want_sums):
    N, C, H, W = x.shape
    return (x.new_empty((N, H, W, channel_pitch), dtype=torch.int8 if quant_min < 0 else torch.uint8),
            x.new_empty((N * H * W if want_sums else 0,), dtype=torch.int32))


@torch.library.register_fake("mctq::packed_linear_i8_padded")
def _(x_codes, in_features, x_zero_point, x_rowsum, codes, kind, is_signed, out_features, zero_point, w_rowsum, factor, bias,
      dtype, lut_values):
    return x_codes.new_empty(tuple(x_codes.shape[:-1]) + (out_features,),
                             dtype=torch.float32 if lut_values is not None else dtype)


@torch.library.register_fake("mctq::packed_conv2d_i8_padded")
def _(x_codes, in_channels, x_zero_point, x_rowsum, codes, kind, is_signed, out_channels, kernel_size, stride, dilation,
      padding, zero_point, w_rowsum, factor, bias, dtype, channels_last, lut_values):
    N, H, W, _ = x_codes.shape
    Ho, Wo = conv_output_hw(H, W, kernel_size, stride, dilation, padding)
    dt = torch.float32 if lut_values is not None else dtype
    if channels_last:
        return x_codes.new_empty((N, Ho, Wo, out_channels), dtype=dt).permute(0, 3, 1, 2)
    return x_codes.new_empty((N, out_channels, Ho, Wo), dtype=dt)


# --------------------------------------------------------------------------------------------- whole-model launch
class MultiTensorPlan:
    """One-launch fake-quant of many weight tensors (C ABI: mctq_fq_affine_multi).

    Build once from [(x, scale, zp, axis, qmin, qmax)] (all CUDA, same device): outputs are allocated here and
    reused by every run(); the descriptor table is uploaded once.  run() enqueues ONE kernel on the current
    stream.  Reference loop being replaced: quantize_wrapper.py:228-240 / :260-270."""

    @staticmethod
    def accepts(item):
        """Whether a tensor can be part of a plan: CUDA, supported dtype, non-empty, dense in memory (the plan captures
        pointers, so no hidden copies), parameters of the right length."""
        x, scale, zp, axis, qmin, qmax = item
        if not x.is_cuda or x.dtype not in _DT or x.numel() == 0 or not _is_dense_permutation(x):
            return False
        try:
            if axis is None:
                if scale.numel() != 1 or zp.numel() != 1:
                    return False
                xd = _dense(x)
            else:
                _check_channel_params(x, scale, zp, axis)
                xd = _channel_layout(x, axis)[0]
        except (RuntimeError, IndexError):
            return False
        return xd.data_ptr() == x.data_ptr() and scale.dtype == torch.float32 and zp.dtype == torch.int32

    def __init__(self, items):
        lib = _native.load()
        if not items:
            raise ValueError("MultiTensorPlan needs at least one tensor")
        self.device = items[0][0].device
        self.inputs, self.outputs, self._keep = [], [], []
        descs = (_native.MctqTensorDesc * len(items))()
        for k, (x, scale, zp, axis, qmin, qmax) in enumerate(items):
            if x.device != self.device or not x.is_cuda:
                raise ValueError("all tensors of a MultiTensorPlan must live on one CUDA device")
            _check_range(qmin, qmax)
            if axis is None:
                xd, C, inner = _dense(x), 1, 1
                if scale.numel() != 1 or zp.numel() != 1:
                    raise RuntimeError("per-tensor entry needs one scale / zero-point")
            else:
                _check_channel_params(x, scale, zp, axis)
                xd, C, inner = _channel_layout(x, axis)
            if xd.data_ptr() != x.data_ptr():
                raise ValueError("MultiTensorPlan needs dense tensors (no hidden copies: the plan captures pointers)")
            y = torch.empty_like(xd)
            s, z = _param_on(scale.contiguous(), self.device), _param_on(zp.contiguous(), self.device)
            self._keep += [s, z]
            self.inputs.append(xd)
            self.outputs.append(y)
            d = descs[k]
            d.x, d.y, d.codes, d.scale, d.zp = xd.data_ptr(), y.data_ptr(), None, s.data_ptr(), z.data_ptr()
            d.n, d.C, d.inner = xd.numel(), C, inner
            d.qmin, d.qmax, d.dtype, d.code_mode = int(qmin), int(qmax), _dtype_tag(xd), 0
        starts = (ctypes.c_int32 * (len(items) + 1))()
        total = lib.mctq_multi_plan(ctypes.cast(descs, c_vp), len(items), ctypes.cast(starts, c_vp))
        if total < 0:
            raise MctqError(f"mctq_multi_plan: {total}")
        self.total_tiles = int(total)
        self.n_desc = len(items)
        self._descs_dev = torch.frombuffer(bytearray(bytes(descs)), dtype=torch.uint8).to(self.device)
        self._starts_dev = torch.frombuffer(bytearray(bytes(starts)), dtype=torch.uint8).to(self.device)

    def run(self):
        lib = _native.load()
        with _on_device(self.device):
            rc = lib.mctq_fq_affine_multi(_ptr(self._descs_dev), _ptr(self._starts_dev), self.n_desc, self.total_tiles,
                                          _stream(self.device))
        _native.check(rc, "mctq_fq_affine_multi")
        return self.outputs


class ScalarSitesPlan:
    """One-launch per-tensor fake-quant of many tensors (C ABI: mctq_fq_affine_scalar_multi).

    Build once from [(x, scale, zero_point, qmin, qmax)] (CUDA tensors of ONE device, dense, 16-byte aligned; scale a Python
    float, narrowed to f32 like ATen does): outputs are allocated here and reused by every run(); the site table is a host
    array that travels as kernel parameters.  run() enqueues ONE kernel per 64 sites on the current stream.
    Reference loop being replaced: one PytorchActivationQuantizationHolder.forward per site
    (activation_quantization_holder.py:43-53)."""

    @staticmethod
    def accepts(x):
        return (x.is_cuda and x.dtype in _DT and x.numel() > 0 and _is_dense_permutation(x) and (x.data_ptr() & 15) == 0)

    def __init__(self, items):
        if not items:
            raise ValueError("ScalarSitesPlan needs at least one tensor")
        self.device = items[0][0].device
        self.inputs, self.outputs = [], []
        self._sites = (_native.MctqSiteDesc * len(items))()
        for k, (x, scale, zp, qmin, qmax) in enumerate(items):
            if x.device != self.device or not self.accepts(x):
                raise ValueError(f"tensor {k} cannot be part of a ScalarSitesPlan (see ScalarSitesPlan.accepts)")
            _check_range(qmin, qmax)
            if not int(qmin) <= int(zp) <= int(qmax):
                raise RuntimeError("`zero_point` must be between `quant_min` and `quant_max`.")
            y = torch.empty_like(x)                         # preserve_format: a dense permutation keeps its strides
            if y.stride() != x.stride():
                raise ValueError(f"tensor {k}: output strides differ from the input's")
            d = self._sites[k]
            d.x, d.y, d.n, d.dtype = x.data_ptr(), y.data_ptr(), x.numel(), _DT[x.dtype]
            d.scale, d.zp, d.qmin, d.qmax = float(np.float32(scale)), int(zp), int(qmin), int(qmax)
            self.inputs.append(x)
            self.outputs.append(y)
        self.n_sites = len(items)
        self._sites_ptr = ctypes.cast(self._sites, c_vp)
        self._sites_addr = ctypes.addressof(self._sites)

    def run(self):
        lib = _native._lib or _native.load()
        index = self.device.index
        prev = _get_device()
        if prev != index:
            _set_device(index)
        fast = _native.fast
        if fast is not None:
            rc = fast.fq_affine_scalar_multi(self._sites_addr, self.n_sites, _raw_stream(index))
        else:
            rc = lib.mctq_fq_affine_scalar_multi(self._sites_ptr, self.n_sites, _raw_stream(index))
        if prev != index:
            _set_device(prev)
        if rc:
            _native.check(rc, "mctq_fq_affine_scalar_multi")
        return self.outputs


def _compile_plan(plan_bytes, plan, descs, n_desc, buf=None):
    """Compile a descriptor array into a host plan blob with a (`*_plan_bytes`, `*_plan`) pair of the C ABI, reusing `buf`
    when it is large enough.  Returns (blob, total tiles, launches): launches = n_chunks of the 64-byte blob header, one per
    kernel variant and 64 tensors."""
    p = ctypes.cast(descs, c_vp)
    nb = plan_bytes(p, n_desc)
    if nb == 0:
        total = plan(p, n_desc, None, 0)
    else:
        if buf is None or len(buf) < nb:
            buf = (ctypes.c_uint8 * nb)()
        total = plan(p, n_desc, ctypes.cast(buf, c_vp), len(buf))
    if total < 0:
        raise MctqError(f"{plan.__name__}: {_native.ERRORS.get(total, total)}")
    return buf, int(total), ctypes.c_int32.from_buffer(buf, 8).value


class LutMultiPlan:
    """One-launch LUT fake-quant of many weight tensors (C ABI: mctq_lut_multi_plan + mctq_fq_lut_prepared_multi).

    Build once from [(x, table, K, threshold, per_channel, axis, eps)] (all CUDA, one device; `table` is the host search
    table of the quantizer): every tensor's decision tables are prepared (or taken from the per-quantizer cache), outputs
    are allocated here and reused by every run(); the plan travels as kernel parameters.  run() enqueues ONE kernel
    per kernel variant and 64 tensors on the current stream -- no launch gaps and no per-launch tails between the tensors
    (Llama-7B: 96 launches -> 2).
    `accepts(item)` tells whether a tensor can be part of a plan (prepared path available, dense, aligned)."""

    @staticmethod
    def _describe(item, device, y=None):
        x, table, K, threshold, per_channel, axis, eps = item
        if not x.is_cuda or x.device != device or x.dtype not in _DT or x.numel() == 0:
            return None
        if threshold.dtype != torch.float32:
            return None
        if per_channel:
            if threshold.numel() != x.shape[axis]:
                return None
            xd, C, inner = _channel_layout(x, axis)
        else:
            if threshold.numel() != 1:
                return None
            xd, C, inner = _dense(x), 1, 1
        if xd.data_ptr() != x.data_ptr():
            return None                                    # the plan captures pointers: no hidden copies
        thr = _param_on(threshold.contiguous(), device)
        prep = _prepared_for(table, K, device, thr, eps, False, 1.0, 1.0, 0)
        if prep is None or prep[1] is None:
            return None
        d = _native.MctqLutTensorDesc()
        d.x, d.y, d.prepared_dev = xd.data_ptr(), (y.data_ptr() if y is not None else xd.data_ptr()), prep[1].data_ptr()
        d.n, d.C, d.inner = xd.numel(), C, inner
        d.dtype, d.K, d.lut_values_bitwidth, d.is_signed = _DT[xd.dtype], int(K), prep[2], prep[3]
        return d, xd, (thr, prep)

    @staticmethod
    def accepts(item):
        x = item[0]
        if not x.is_cuda:
            return False
        got = LutMultiPlan._describe(item, x.device)
        if got is None:
            return False
        lib = _native.load()
        descs = (_native.MctqLutTensorDesc * 1)(got[0])     # y stands in as x here: fresh outputs are at least as aligned
        return lib.mctq_lut_multi_plan_bytes(ctypes.cast(descs, c_vp), 1) > 0

    def __init__(self, items):
        lib = _native.load()
        if not items:
            raise ValueError("LutMultiPlan needs at least one tensor")
        self.device = items[0][0].device
        self.inputs, self.outputs, self._keep = [], [], []
        descs = (_native.MctqLutTensorDesc * len(items))()
        for k, item in enumerate(items):
            x = item[0]
            if not x.is_cuda or x.device != self.device:
                raise ValueError("all tensors of a LutMultiPlan must live on one CUDA device")
            y = torch.empty(x.shape, dtype=torch.float32, device=self.device)
            if not x.is_contiguous():
                y = torch.empty_like(_dense(x), dtype=torch.float32)
            got = self._describe(item, self.device, y)
            if got is None:
                raise ValueError(f"tensor {k} cannot be part of a LutMultiPlan (see LutMultiPlan.accepts)")
            descs[k] = got[0]
            self.inputs.append(got[1])
            self.outputs.append(y)
            self._keep.append(got[2])
        self.n_desc = len(items)
        self._plan_host, self.total_tiles, self.n_launches = _compile_plan(lib.mctq_lut_multi_plan_bytes, lib.mctq_lut_multi_plan,
                                                                           descs, self.n_desc)

    def run(self):
        lib = _native.load()
        with _on_device(self.device):
            rc = lib.mctq_fq_lut_prepared_multi(ctypes.cast(self._plan_host, c_vp), _stream(self.device))
        _native.check(rc, "mctq_fq_lut_prepared_multi")
        return self.outputs



class UnpackPlan:
    """Rebuild many packed tensors in one launch per kernel variant and 64 tensors (C ABI: mctq_unpack_plan +
    mctq_unpack_multi).  The result of each tensor is bit-identical to the fake-quant output its codes were taken from.

    Build once from items (all on one CUDA device)
        (codes, kind, is_signed, dtype, shape, stride, C, inner, scale, zero_point, lut_quotients)
    codes      uint8 / int8 tensor in the layout of `kind` (_native.PACK_*), elements in the output's memory order
    dtype      output dtype (f32 for the LUT kinds); shape / stride of the output (stride None: row-major)
    C, inner   [outer][C][inner] view of the output's memory (C = 1: per tensor)
    scale      f32 [C] (affine scale, or LUT threshold); zero_point int32 [C] (affine) or None
    lut_quotients  f32 [K] (LUT kinds, see lut_quotients()) or None
    `outputs` (optional): tensors to write into instead of plan-owned buffers.
    `fresh=True`: every run() writes into newly allocated tensors (re-planned on the host) and the plan keeps no reference
    to them, so that a caller can drop the rebuilt tensors after use and keep only the codes resident.

    run() enqueues the launches on the current stream and returns the outputs."""

    def __init__(self, items, outputs=None, fresh=False):
        if not items:
            raise ValueError("UnpackPlan needs at least one tensor")
        lib = _native.load()
        self.device = items[0][0].device
        if self.device.type != "cuda":
            raise ValueError("UnpackPlan needs CUDA tensors")
        self.n_desc = len(items)
        self._descs = (_native.MctqPackedDesc * self.n_desc)()
        self._keep, self._out_specs = [], []
        for k, (codes, kind, is_signed, dtype, shape, stride, C, inner, scale, zp, quot) in enumerate(items):
            if codes.device != self.device:
                raise ValueError("all tensors of an UnpackPlan must live on one CUDA device")
            if not codes.is_contiguous() or codes.data_ptr() % 16:      # the kernels load codes in 16-byte aligned vectors
                codes = codes.clone(memory_format=torch.contiguous_format)
            n = 1
            for s_ in shape:
                n *= int(s_)
            self._descs[k], keep = _packed_desc(codes, kind, is_signed, dtype, n, C, inner, scale, zp, quot, self.device,
                                                f"tensor {k}")
            self._keep.append(keep)
            self._out_specs.append((tuple(int(v) for v in shape), None if stride is None else tuple(int(v) for v in stride), dtype))
        self._plan_host, self.fresh = None, fresh
        if fresh:
            if outputs is not None:
                raise ValueError("a fresh UnpackPlan allocates its outputs on every run")
            self._install(self._new_outputs(), lib)       # validates the descriptors once
            self.outputs = None
        elif outputs is not None:
            outputs = list(outputs)
            for k, (y, (shape, stride, dtype)) in enumerate(zip(outputs, self._out_specs)):
                if y.device != self.device or y.dtype != dtype or tuple(y.shape) != shape or \
                        (stride is not None and tuple(y.stride()) != stride) or (stride is None and not y.is_contiguous()):
                    raise ValueError(f"output {k} does not match the packed tensor's device, dtype, shape or strides")
            self._install(outputs, lib)
        else:
            self._install(self._new_outputs(), lib)

    def _new_outputs(self):
        return [torch.empty(shape, dtype=dtype, device=self.device) if stride is None else
                torch.empty_strided(shape, stride, dtype=dtype, device=self.device)
                for shape, stride, dtype in self._out_specs]

    def _install(self, outputs, lib):
        for d, y in zip(self._descs, outputs):
            d.y = y.data_ptr() if y.numel() else None
        self._plan_host, self.total_tiles, self.n_launches = _compile_plan(lib.mctq_unpack_plan_bytes, lib.mctq_unpack_plan,
                                                                           self._descs, self.n_desc, self._plan_host)
        self._plan_nb = len(self._plan_host)
        self.outputs = outputs

    def run(self):
        lib = _native._lib or _native.load()
        if self.fresh:
            self._install(self._new_outputs(), lib)
        with _on_device(self.device):
            rc = lib.mctq_unpack_multi(ctypes.cast(self._plan_host, c_vp), _stream(self.device))
        _native.check(rc, "mctq_unpack_multi")
        outputs = self.outputs
        if self.fresh:
            self.outputs = None
        return outputs
