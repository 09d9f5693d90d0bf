"""Packed weight storage for quantized models: int8 / int4 affine codes and LUT indices instead of float weights.

    report = pack_model_weights(model)        # or wrapper.pack_weights() for one PytorchQuantizationWrapper
    y = model(x)                              # bit-identical to the float model's output

A packed weight keeps only its codes (one byte or one nibble per element) as a `uint8` / `int8` buffer of its wrapper; the
float parameter is deleted.  Every forward of a packed wrapper rebuilds all of its packed weights with ONE unpack launch
(csrc/mctq_unpack.cu), installs them exactly as the float path installs `quantizer(weight)`, runs the layer and drops the
rebuilt tensors again, so that only the codes stay resident.  A rebuilt weight equals `quantizer(float_weight)` bit for bit,
in dtype, shape and strides -- the codes are what the quantizer's own kernels emit (`code_mode` / `idx_mode`), and packing
checks every rebuilt weight against the quantizer's output once.

Which weights pack: those of the five built-in weight quantizers (symmetric, POT, uniform, LUT symmetric, LUT POT) on a CUDA
device whose codes fit 8 bits -- affine ranges of at most 256 levels (int4 codes for ranges of at most 16), LUTs of at most
256 centroids (4-bit indices for at most 16).  Everything else keeps its float weight and its current path; the report says
why for each weight.

Fused linear mode (`pack_model_weights(model, fused_linear=True)`, opt-in): a packed `torch.nn.Linear` wrapper computes
`x @ W^T + b` straight from its codes (csrc/mctq_packed_linear.cu) when the input has at most FUSED_LINEAR_MAX_ROWS rows, so
W is never rebuilt in memory.  W is exactly the rebuilt weight, the sum is accumulated in f32 in a fixed order and rounded
once to x's dtype: deterministic and within f32 rounding of the exact product, but not bit-identical to the float model.
Larger inputs, and every input the fused kernel does not take (see PackedState.fused_forward), run the exact packed path.

Batched linear mode (`pack_model_weights(model, fused_linear=True, batched_linear=True)`, opt-in on top of the fused mode):
inputs of more than FUSED_LINEAR_MAX_ROWS and at most FUSED_BATCHED_MAX_ROWS rows take the tensor-core kernel
(csrc/mctq_packed_gemm.cu) instead of the exact path; smaller inputs keep the fused kernel.  Same contract: W is exactly the
rebuilt weight, f32 accumulation, one rounding to x's dtype, deterministic.  LUT weights qualify when every quotient of the
table is exact in bf16 (integer centroids on grids of up to 8 bits).

Integer linear mode (`pack_model_weights(model, integer_linear=True)`, or `wrapper.pack_weights(integer_linear=True,
input_quantizer=q)` for one wrapper; opt-in): a packed `torch.nn.Linear` wrapper with int8 / int4 affine codes whose input
comes from a per-tensor 8-bit affine activation quantizer Q computes `layer(Q(x))` with integer arithmetic: Q's codes of x
(csrc/mctq_affine.cu, mctq_quantize_rows_i8) times the weight codes as an exact int32 sum on the tensor cores
(csrc/mctq_packed_igemm.cu), then the zero-point corrections and one f32 scaling per output (include/mctq.h gives the formula
bit for bit).  Q is idempotent on its own outputs, so on a holder -> Linear edge this is the fake-quant model's product summed
exactly; it differs from the float model by f32 accumulation rounding (and, for bf16 / f16, by the rounding of the holder's
outputs and of W to that dtype).  It is a numerical contract of its own, so it covers every row count.  The model-level call
traces the model with torch.fx (holders and wrappers as leaves) and switches each eligible wrapper whose input is a holder's
output, directly or through flatten / reshape / view / contiguous; integer mode takes precedence over fused / batched mode.

Integer convolution mode (`pack_model_weights(model, integer_conv=True)`, or `wrapper.pack_weights(integer_conv=True,
input_quantizer=q)`; opt-in, and it may be combined with integer_linear=True): the same arithmetic for a packed
`torch.nn.Conv2d` wrapper (groups 1, zero padding, Cin a multiple of 16) fed by such a holder.  Q's codes of x are written
channels-innermost (NHWC, csrc/mctq_affine.cu, mctq_quantize_nhwc_i8) and the convolution is an implicit GEMM whose x
operand is gathered from each output pixel's window (csrc/mctq_packed_igemm.cu, mctq_packed_conv2d_i8); a padded tap holds
Q's zero-point code and contributes exactly 0.  The output has the memory format F.conv2d gives for x and the rebuilt
weight.  Inputs that are not 4-D (unbatched 3-D inputs included) take the packed path.

Integer depthwise convolution (`integer_depthwise=True` together with integer_conv=True; opt-in): integer convolution mode
for Conv2d layers with groups == in_channels > 1 and any channel multiplier, such as the 3x3 depthwise convs of MobileNetV2.
A depthwise conv is a stencil, not a matrix product: one kernel (csrc/mctq_affine.cu, mctq_packed_dwconv2d_i8) reads the
float x once, computes Q's codes in registers and sums (qx - zx) * (qw - zw) exactly in int32 over each window (include/mctq.h
gives the formula).  With integer_lut=True it takes LUT weights too.

Integer modes for LUT weights (`integer_lut=True` together with integer_linear=True and / or integer_conv=True; opt-in): a
LUT weight rebuilds as fl32(lut_k / 2^(bw-1) * thr[o]) with integer centroids lut_k, i.e. an int8 code lut_k times the scale
sw[o] = thr[o] * 2^-(bw-1) and zero point 0.  When every centroid is an integer in [-128, 127] and every sw[o] is exact and
normal in f32, the integer modes take LUT wrappers too: the GEMM's weight producers look each index up in the table (passed
by value with every launch) and the product is the same exact int32 sum (include/mctq.h).  It differs from the packed path
by the rounding of W to f32 and by f32 accumulation, so it stays opt-in: without the flag LUT wrappers keep their paths.

Padded integer modes (`integer_pad=True` together with integer_linear=True and / or integer_conv=True; opt-in): Linear layers
whose in_features and groups-1 Conv2d layers whose Cin is off the GEMM's granule (16 codes, 32 for 4-bit codes), such as a
stem with Cin = 3 or the squeeze-excitation convs of EfficientNet.  Q's codes get a padded pitch whose pad columns hold Q's
zero-point code and are counted in the corrections, so they contribute exactly 0: every output is the formula over the real
row (include/mctq.h, DESIGN §7f).  Convs with Cin <= 8 take a narrow gather with a pixel pitch of 4 or 8 codes.

Packing is one-way and for inference only:
  * the rebuild dtype is the weight's dtype at packing time; `.half()` does not change it (the codes are integer buffers);
  * the packed state travels with the module: `state_dict` / `load_state_dict` between packed models of the same structure,
    `.to(device)`, `torch.save` + `pytorch_load_quantized_model`;
  * a packed wrapper cannot be traced (ONNX export needs the float weights, which are gone) and cannot be trained.
"""
import functools
import weakref
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
from torch.nn.modules import module as _nn_module

from mct_quantizers_b200 import _native, ops
from mct_quantizers_b200.common.constants import LAYER, POSITIONAL_WEIGHT, QUANTIZED_POSITIONAL_WEIGHT

# Largest number of input rows (the product of x's leading dimensions) a fused-mode wrapper computes with the fused kernel,
# per dtype of the rebuilt weight: above it, rebuilding W and calling F.linear is faster.  The largest M at which the fused
# kernel beat the rebuild in every benchmarked format of the dtype (tools/packed_linear_bench.py, Llama-7B's MLP shapes,
# one B200 at 1000 W, profiles/r04_packed_linear_bench.txt): f32 8 (4-bit LUT; 16 loses), bf16 4 (int4 and int8; 8 loses).
# f16 runs the bf16 code path and takes its value.
FUSED_LINEAR_MAX_ROWS = {torch.float32: 8, torch.bfloat16: 4, torch.float16: 4}

# Largest number of input rows a batched-mode wrapper computes with the tensor-core kernel (above FUSED_LINEAR_MAX_ROWS),
# per dtype of the rebuilt weight: the largest M up to which the kernel beat rebuild + F.linear at every measured M in
# every format of the dtype (tools/packed_batched_bench.py, Llama-7B's MLP shapes, one B200 at 1000 W,
# profiles/r05_packed_batched_bench.txt).  f32: 256 (4-bit LUT, int4 and int8 affine; every M from 8 to 256 wins).  bf16: the kernel lost at
# every M (int4 and int8), so the limit equals FUSED_LINEAR_MAX_ROWS and batched mode leaves bf16 wrappers as they are;
# f16 runs the bf16 code path and takes its value.
FUSED_BATCHED_MAX_ROWS = {torch.float32: 256, torch.bfloat16: 4, torch.float16: 4}

_KIND_NAMES = {_native.PACK_AFFINE_I8: "affine_i8", _native.PACK_AFFINE_I4: "affine_i4",
               _native.PACK_LUT_U8: "lut_u8", _native.PACK_LUT_I4: "lut_i4"}


def _builtin_kind(q) -> Optional[str]:
    """'affine' / 'lut' for the five built-in weight quantizers (exact classes: a subclass may change the arithmetic)."""
    from mct_quantizers_b200.pytorch.quantizers import (WeightsSymmetricInferableQuantizer, WeightsPOTInferableQuantizer,
                                                        WeightsUniformInferableQuantizer, WeightsLUTSymmetricInferableQuantizer,
                                                        WeightsLUTPOTInferableQuantizer)
    t = type(q)
    if t in (WeightsSymmetricInferableQuantizer, WeightsPOTInferableQuantizer, WeightsUniformInferableQuantizer):
        return 'affine'
    if t in (WeightsLUTSymmetricInferableQuantizer, WeightsLUTPOTInferableQuantizer):
        return 'lut'
    return None


def packing_kind(q, w) -> Tuple[Optional[int], str]:
    """(kind, '') when weight `w` of quantizer `q` can be packed (kind: _native.PACK_*), else (None, reason)."""
    if not isinstance(w, torch.Tensor) or not w.is_cuda:
        return None, "the weight is not on a CUDA device"
    return code_kind(q, w)


def code_kind(q, w) -> Tuple[Optional[int], str]:
    """packing_kind without the placement check: the code format weight `w` of quantizer `q` would be packed in."""
    family = _builtin_kind(q)
    if family is None:
        return None, f"quantizer {type(q).__name__} is not a built-in weight quantizer"
    d = q.__dict__
    if d.get('enable_reuse', False):
        return None, "the quantizer reuses its outputs (enable_reuse)"
    if d.get('_use_custom_impl', False):
        return None, "the quantizer is set up for ONNX export (_use_custom_impl)"
    if w.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        return None, f"weight dtype {w.dtype} is not float32 / bfloat16 / float16"
    if family == 'affine':
        if d.get('_zero_point_out_of_range', False):
            return None, "a zero point lies outside the quantization range (the quantizer raises ATen's error)"
        qmin, qmax = int(q.min_quantized_domain), int(q.max_quantized_domain)
        if (-8 <= qmin and qmax <= 7) or (0 <= qmin and qmax <= 15):
            return _native.PACK_AFFINE_I4, ""
        if (-128 <= qmin and qmax <= 127) or (0 <= qmin and qmax <= 255):
            return _native.PACK_AFFINE_I8, ""
        return None, f"quantization range [{qmin}, {qmax}] does not fit 8-bit codes"
    if q.per_channel and q.input_rank is not None and q.input_rank != w.dim():
        return None, "input_rank does not match the weight (the quantizer raises the reference's error)"
    K = int(q._lut_values_torch.numel())
    if K <= 16:
        return _native.PACK_LUT_I4, ""
    if K <= 256:
        return _native.PACK_LUT_U8, ""
    return None, f"{K} LUT entries do not fit 8-bit indices"


class PackedWeight:
    """One packed weight of a wrapper: where its codes live (buffers of the owning wrapper) and how to rebuild it.
    Stands in for the float weight in (name, weight, quantizer) triples, e.g. for ModelWeightPlan; `data_ptr()`, `dtype`,
    `shape` and `stride()` describe the codes, so that a plan notices moved storage.  The owner is held by a weak reference
    (a wrapper and its entries form no reference cycle, so `del model` frees the codes at once); copies and unpickled
    objects are bound to their wrapper again by PackedState.bind."""

    def __init__(self, owner, name, quantizer, kind, is_signed, dtype, shape, stride, C, inner):
        self._owner, self.name, self.quantizer = weakref.ref(owner), name, quantizer
        self.kind, self.is_signed, self.dtype_out = kind, is_signed, dtype
        self.shape_out, self.stride_out, self.C, self.inner = tuple(shape), tuple(stride), C, inner
        self.codes_name, self.quot_name = f"packed_codes_{name}", f"packed_lutq_{name}"

    def __getstate__(self):
        return {**self.__dict__, '_owner': None}

    @property
    def codes(self) -> torch.Tensor:
        return self._owner()._buffers[self.codes_name]

    @property
    def lut_quotients(self) -> Optional[torch.Tensor]:
        # kept as the int32 bit patterns of the f32 quotients, so that `.half()` / `.to(dtype)` leave them alone
        q = self._owner()._buffers.get(self.quot_name)
        return q.view(torch.float32) if q is not None else None

    # the storage signature a WeightPlan compares
    def data_ptr(self):
        return self.codes.data_ptr()

    @property
    def dtype(self):
        return self.codes.dtype

    @property
    def shape(self):
        return self.codes.shape

    def stride(self):
        return self.codes.stride()

    @property
    def is_cuda(self):
        return self.codes.is_cuda

    @property
    def device(self):
        return self.codes.device

    def plan_item(self):
        """The UnpackPlan item of this weight, parameters on the codes' device."""
        q, dev = self.quantizer, self.codes.device
        if self.kind in _native.PACK_LUT_KINDS:
            thr, = q._on(dev, q._threshold_torch)
            return (self.codes, self.kind, False, self.dtype_out, self.shape_out, self.stride_out, self.C, self.inner,
                    thr.reshape(-1), None, self.lut_quotients)
        scales, zps = q._on(dev, q.scales, q.zero_points)
        return (self.codes, self.kind, self.is_signed, self.dtype_out, self.shape_out, self.stride_out, self.C, self.inner,
                scales.reshape(-1), zps.reshape(-1), None)

    def __repr__(self):
        return (f"PackedWeight({self.name!r}, {_KIND_NAMES[self.kind]}, {self.dtype_out}, shape={list(self.shape_out)}, "
                f"{self.codes.numel()} code bytes)")


def _emit_codes(q, w, kind):
    """(codes, is_signed, C, inner) of weight w: the quantizer's kernels in code-emission mode, elements in the memory order
    of quantizer(w)."""
    if kind in _native.PACK_LUT_KINDS:
        if q.__dict__.get('_search_table') is None:
            from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
            q._search_table = lut_search_table(q._lut_values_np, q.lut_values_bitwidth, True)
        thr, = q._on(w.device, q._threshold_torch)
        axis = int(q.channel_axis) if q.per_channel else 0
        idx_mode = _native.CODES_INT4 if kind == _native.PACK_LUT_I4 else _native.CODES_INT8
        codes = torch.ops.mctq.lut_indices(w.detach(), q._search_table, int(q._lut_values_torch.numel()), thr.reshape(-1),
                                           bool(q.per_channel), axis, float(q.eps), idx_mode)
        C, inner = ops.contiguous_layout(tuple(w.shape), axis % max(w.dim(), 1)) if q.per_channel else (1, 1)
        return codes.reshape(-1), False, int(C), int(inner)
    scales, zps = q._on(w.device, q.scales, q.zero_points)
    qmin, qmax = int(q.min_quantized_domain), int(q.max_quantized_domain)
    if q.per_channel:
        xd, C, inner = ops._channel_layout(w.detach(), q.channel_axis)
    else:
        xd, C, inner = ops._dense(w.detach()), 1, 1
    code_mode = _native.CODES_INT4 if kind == _native.PACK_AFFINE_I4 else _native.CODES_INT8
    codes = ops.affine_codes(xd, scales.reshape(-1).contiguous(), zps.reshape(-1).contiguous(), C, inner, qmin, qmax, code_mode)
    return codes, qmin < 0, int(C), int(inner)


def fused_linear_eligibility(wrapper) -> Tuple[bool, str]:
    """(True, '') when `wrapper` can run in fused linear mode, else (False, reason).  Host-only: looks at the wrapper's
    layer, weights and packed layout, never at device memory."""
    d = wrapper.__dict__
    if not d.get('is_str_attr', False):
        return False, "the weights are positional inputs of a functional op"
    layer = d['_modules'].get(LAYER)
    if type(layer) is not torch.nn.Linear:
        return False, f"the layer is {type(layer).__name__}, not torch.nn.Linear"
    if d.get('op_call_args') or d.get('op_call_kwargs') or d.get('is_inputs_as_list'):
        return False, "the wrapper passes extra call arguments to the layer"
    if list(wrapper.weights_quantizers) != ['weight']:
        return False, "the wrapper quantizes weights other than 'weight'"
    state = d.get('_packed')
    e = next((e for e in state.entries if e.name == 'weight'), None) if state is not None else None
    if e is None:
        return False, "the weight is not packed"
    out_f, in_f = layer.out_features, layer.in_features
    if e.shape_out != (out_f, in_f) or e.stride_out != (in_f, 1):
        return False, "the rebuilt weight is not a row-major [out_features, in_features] matrix"
    if not (e.C == 1 or (e.C == out_f and e.inner == in_f)):
        return False, "the parameters are not per tensor or per output channel (channel_axis 0)"
    return True, ""


def _lut_quotients_host(q):
    """The f32 quotients of LUT quantizer q, computed on the host (no device synchronisation): the values a packed wrapper
    registers and batched_linear_eligibility checks."""
    return ops.lut_quotients(torch.as_tensor(q._lut_values_np), q.lut_values_bitwidth, True)


def batched_linear_eligibility(wrapper) -> Tuple[bool, str]:
    """(True, '') when `wrapper` can run in batched linear mode: fused_linear_eligibility, and for LUT weights every quotient
    of the table exact in bf16 (the tensor cores multiply it as a bf16 operand).  Host-only."""
    ok, reason = fused_linear_eligibility(wrapper)
    if not ok:
        return ok, reason
    e = next(e for e in wrapper.__dict__['_packed'].entries if e.name == 'weight')
    if e.kind in _native.PACK_LUT_KINDS:
        bits = _lut_quotients_host(e.quantizer).view(torch.int32)
        if bool(((bits & 0xFFFF) != 0).any()):
            return False, "a LUT quotient is not exact in bfloat16 (the tensor cores take the quotients as bf16 operands)"
    return True, ""


def _input_quantizer_eligibility(input_quantizer) -> Tuple[bool, str]:
    """The conditions integer linear and integer convolution mode put on the input quantizer: per-tensor affine, no reuse
    of its outputs, 8-bit codes."""
    from mct_quantizers_b200.pytorch.fused_activation_holder import affine_scalar_params
    if affine_scalar_params(input_quantizer) is None:
        return False, (f"the input quantizer {type(input_quantizer).__name__} is not a per-tensor affine activation quantizer "
                       f"(ActivationSymmetric / POT / Uniform)")
    if input_quantizer.__dict__.get('enable_reuse', False):
        return False, "the input quantizer reuses its outputs (enable_reuse)"
    qmin, qmax = int(input_quantizer.min_quantized_domain), int(input_quantizer.max_quantized_domain)
    if not ((-128 <= qmin and qmax <= 127) or (0 <= qmin and qmax <= 255)):
        return False, f"the input quantization range [{qmin}, {qmax}] does not fit 8-bit codes"
    return True, ""


def _lut_code_eligibility(e) -> Tuple[bool, str]:
    """The conditions every integer mode puts on a LUT weight (entry e): integer centroids in [-128, 127] and every
    thr[o] * 2^-(bw-1) exact and normal in f32.  Host-only: reads the quantizer's numpy parameters."""
    q = e.quantizer
    v = np.asarray(q._lut_values_np, dtype=np.float64).reshape(-1)
    if not (np.all(v == np.round(v)) and np.all(v >= -128) and np.all(v <= 127)):
        return False, "a LUT value is not an integer in [-128, 127] (the integer modes take the centroids as int8 codes)"
    sw = np.asarray(q._threshold_np, dtype=np.float32).reshape(-1).astype(np.float64) * 2.0 ** -(int(q.lut_values_bitwidth) - 1)
    if not (np.all(np.isfinite(sw)) and np.all(sw.astype(np.float32) == sw) and
            np.all(np.abs(sw) >= np.finfo(np.float32).tiny)):
        return False, "a threshold times 2^-(lut_values_bitwidth - 1) is not exact and normal in float32"
    return True, ""


def _lut_eligibility(e, K, what, x_signed, padded=None) -> Tuple[bool, str]:
    """The conditions the GEMM integer modes put on a LUT weight (entry e, row length K named `what`): _lut_code_eligibility,
    K a multiple of 32 (4-bit indices) or 16 (8-bit indices) and at most the int32 bound of signed weight codes.  `padded`:
    the row length the padded kernel sums instead (integer_pad), which takes the place of the multiple rule."""
    ok, reason = _lut_code_eligibility(e)
    if not ok:
        return ok, reason
    step, bits = (32, 4) if e.kind == _native.PACK_LUT_I4 else (16, 8)
    if padded is None and K % step:
        return False, f"{what} = {K} is not a multiple of {step} ({bits}-bit LUT indices)"
    return _row_bound(K, padded, what, _native.integer_linear_max_k(True, x_signed))


def _row_bound(K, padded, what, bound) -> Tuple[bool, str]:
    """The int32 bound on the row length the kernel sums: K, or `padded` (not None) when the codes are padded."""
    if K > bound:
        return False, f"{what} = {K} exceeds {bound}, the largest row length whose int32 sum of code products cannot overflow"
    if padded is not None and padded > bound:
        return False, (f"{what} = {K} padded to a row of {padded} exceeds {bound}, the largest row length whose int32 sum "
                       f"of code products cannot overflow")
    return True, ""


def integer_linear_eligibility(wrapper, input_quantizer, lut: bool = False, pad: bool = False) -> Tuple[bool, str]:
    """(True, '') when `wrapper` can run in integer linear mode with input quantizer `input_quantizer`: fused_linear_eligibility,
    int8 / int4 affine codes, a per-tensor affine activation quantizer with 8-bit codes, in_features a multiple of 16 (32 for
    int4 codes) and at most the int32 bound of the code signedness pair.  `lut=True` also accepts LUT weights that meet
    _lut_eligibility.  `pad=True` drops the multiple rule: such rows are padded to ops.linear_code_pitch, and the bound
    applies to the padded row.  Host-only."""
    ok, reason = fused_linear_eligibility(wrapper)
    if not ok:
        return ok, reason
    e = next(e for e in wrapper.__dict__['_packed'].entries if e.name == 'weight')
    is_lut = lut and e.kind in _native.PACK_LUT_KINDS
    if e.kind not in (_native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4) and not is_lut:
        return False, f"the weight is packed as {_KIND_NAMES[e.kind]}, not as int8 / int4 affine codes"
    ok, reason = _input_quantizer_eligibility(input_quantizer)
    if not ok:
        return ok, reason
    qmin = int(input_quantizer.min_quantized_domain)
    K = wrapper.layer.in_features
    padded = ops.linear_code_pitch(K, e.kind) if pad and K % ops._row_step(e.kind) else None
    if is_lut:
        return _lut_eligibility(e, K, "in_features", qmin < 0, padded)
    step = 32 if e.kind == _native.PACK_AFFINE_I4 else 16
    if padded is None and K % step:
        return False, f"in_features = {K} is not a multiple of {step}"
    return _row_bound(K, padded, "in_features", _native.integer_linear_max_k(e.is_signed, qmin < 0))


def _conv_eligibility(wrapper, input_quantizer, lut, depthwise):
    """The checks integer convolution mode makes on a Conv2d wrapper, in their order (depthwise: one input channel per
    group instead of groups 1): (True, '', entry, weight shape, is_lut) or (False, reason)."""
    d = wrapper.__dict__
    if not d.get('is_str_attr', False):
        return False, "the weights are positional inputs of a functional op"
    layer = d['_modules'].get(LAYER)
    if type(layer) is not torch.nn.Conv2d:
        return False, f"the layer is {type(layer).__name__}, not torch.nn.Conv2d"
    if d.get('op_call_args') or d.get('op_call_kwargs') or d.get('is_inputs_as_list'):
        return False, "the wrapper passes extra call arguments to the layer"
    if list(wrapper.weights_quantizers) != ['weight']:
        return False, "the wrapper quantizes weights other than 'weight'"
    if depthwise:
        if layer.groups == 1:
            return False, "groups = 1: not a depthwise convolution"
        if layer.groups != layer.in_channels:
            return False, (f"groups = {layer.groups}: a grouped convolution with {layer.in_channels // layer.groups} input "
                           f"channels per group is not depthwise")
    elif layer.groups != 1:
        return False, f"groups = {layer.groups}: a grouped or depthwise convolution is not one matrix product"
    if layer.padding_mode != 'zeros':
        return False, f"padding_mode = {layer.padding_mode!r}: only zero padding is a padding with Q's zero-point code"
    state = d.get('_packed')
    e = next((e for e in state.entries if e.name == 'weight'), None) if state is not None else None
    if e is None:
        return False, "the weight is not packed"
    is_lut = lut and e.kind in _native.PACK_LUT_KINDS
    if e.kind not in (_native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4) and not is_lut:
        return False, f"the weight is packed as {_KIND_NAMES[e.kind]}, not as int8 / int4 affine codes"
    shape = (layer.out_channels, layer.in_channels // layer.groups) + tuple(layer.kernel_size)
    dense = torch.empty(shape, device="meta")
    if e.shape_out != shape or e.stride_out not in (dense.stride(), dense.to(memory_format=torch.channels_last).stride()):
        return False, (f"the rebuilt weight is not a contiguous or channels_last [Cout, {'1' if depthwise else 'Cin'}, kh, kw] "
                       f"tensor")
    K = shape[1] * shape[2] * shape[3]
    if not (e.C == 1 or (e.C == shape[0] and e.inner == K)):
        return False, "the parameters are not per tensor or per output channel (channel_axis 0)"
    ok, reason = _input_quantizer_eligibility(input_quantizer)
    if not ok:
        return ok, reason
    return True, "", e, shape, is_lut


def integer_conv_eligibility(wrapper, input_quantizer, lut: bool = False, pad: bool = False) -> Tuple[bool, str]:
    """(True, '') when `wrapper` can run in integer convolution mode with input quantizer `input_quantizer`: a
    torch.nn.Conv2d layer with string-attribute weights, no extra call arguments and 'weight' its only quantized weight,
    packed as int8 / int4 affine codes, rebuilt as a contiguous or channels_last [Cout, Cin, kh, kw] weight with parameters
    per tensor or per output channel; groups 1 and zero padding; the input quantizer conditions of integer linear mode;
    Cin a multiple of 16, K = Cin * kh * kw a multiple of 32 for int4 codes and at most the int32 bound of the code
    signedness pair.  `lut=True` also accepts LUT weights that meet _lut_eligibility.  `pad=True` drops the channel and
    multiple rules: such codes get the pixel pitch and row length of ops.conv_code_pitch, and the bound applies to that
    row.  Host-only."""
    r = _conv_eligibility(wrapper, input_quantizer, lut, depthwise=False)
    if not r[0]:
        return r
    _, _, e, shape, is_lut = r
    K = shape[1] * shape[2] * shape[3]
    padded = None
    if pad and (shape[1] % 16 or K % ops._row_step(e.kind)):
        padded = ops.conv_code_pitch(shape[1], shape[2], shape[3], e.kind)[1]
    if padded is None and shape[1] % 16:
        return False, f"in_channels = {shape[1]} is not a multiple of 16"
    if is_lut:
        return _lut_eligibility(e, K, "Cin * kh * kw", int(input_quantizer.min_quantized_domain) < 0, padded)
    if padded is None and e.kind == _native.PACK_AFFINE_I4 and K % 32:
        return False, f"Cin * kh * kw = {K} is not a multiple of 32 (int4 codes)"
    bound = _native.integer_linear_max_k(e.is_signed, int(input_quantizer.min_quantized_domain) < 0)
    return _row_bound(K, padded, "Cin * kh * kw", bound)


def integer_depthwise_eligibility(wrapper, input_quantizer, lut: bool = False) -> Tuple[bool, str]:
    """(True, '') when `wrapper` can run in integer convolution mode as a depthwise convolution (mctq_packed_dwconv2d_i8):
    the layer, wrapper and input-quantizer conditions of integer_conv_eligibility, with groups == in_channels > 1 (any
    channel multiplier) instead of groups 1, a contiguous or channels_last [Cout, 1, kh, kw] weight, kh * kw at most
    33025 (the int32 bound of the centred sum: each factor has magnitude <= 255), and a dilated window that the kernel can
    stage in shared memory (mctq_packed_dwconv2d_i8_plan).  `lut=True` also accepts LUT weights that meet
    _lut_code_eligibility.  Host-only."""
    r = _conv_eligibility(wrapper, input_quantizer, lut, depthwise=True)
    if not r[0]:
        return r
    _, _, e, shape, is_lut = r
    if is_lut:
        ok, reason = _lut_code_eligibility(e)
        if not ok:
            return ok, reason
    kh, kw = shape[2], shape[3]
    K = kh * kw
    if K > 33025:
        return False, f"kh * kw = {K} exceeds 33025, the largest window whose int32 sum of code products cannot overflow"
    # the planner fails for every input size exactly when its smallest tile (one output of one channel) does not fit: ask
    # it for the one output of an input as large as the dilated window
    dh, dw = (int(d) for d in wrapper.layer.dilation)
    ih, iw = (kh - 1) * dh + 1, (kw - 1) * dw + 1
    if ops.dwconv_plan(1, 1, ih, iw, 1, (kh, kw), (1, 1), (dh, dw), (0, 0, 0, 0)) is None:
        return False, (f"the dilated {kh} x {kw} window ({ih} x {iw} input pixels) does not fit the depthwise kernel's "
                       f"shared memory")
    return True, ""


_SHAPE_METHODS = ("flatten", "reshape", "view", "contiguous")
_SHAPE_FUNCS = (torch.flatten, torch.reshape)


def integer_linear_edges(model: torch.nn.Module) -> Tuple[Dict[str, Tuple[str, object]], Dict[str, str], str]:
    """Trace `model` with torch.fx (holders and quantization wrappers as leaves) and find the holder -> wrapper edges of
    integer linear mode: ({wrapper name: (holder name, holder quantizer)}, {wrapper name: why its input does not qualify},
    '') -- or ({}, {}, why the model cannot be traced).  An edge may pass through flatten / reshape / view / contiguous."""
    from mct_quantizers_b200.pytorch.activation_quantization_holder import PytorchActivationQuantizationHolder
    from mct_quantizers_b200.pytorch.fused_activation_holder import _LeafTracer
    from mct_quantizers_b200.pytorch.quantize_wrapper import PytorchQuantizationWrapper
    try:
        graph = _LeafTracer().trace(model)
    except Exception as err:                                     # noqa: BLE001 - any tracing failure switches nothing
        return {}, {}, f"the model cannot be traced with torch.fx ({type(err).__name__}: {err})"
    modules = dict(model.named_modules())
    edges, why = {}, {}
    for node in graph.nodes:
        if node.op != "call_module" or not isinstance(modules.get(node.target), PytorchQuantizationWrapper):
            continue
        if len(node.args) != 1 or node.kwargs:
            why[node.target] = "the wrapper is called with more than one input"
            continue
        src = node.args[0]
        while isinstance(src, torch.fx.Node) and src.args and (
                (src.op == "call_method" and src.target in _SHAPE_METHODS) or
                (src.op == "call_function" and src.target in _SHAPE_FUNCS)):
            src = src.args[0]
        holder = modules.get(src.target) if isinstance(src, torch.fx.Node) and src.op == "call_module" else None
        if not isinstance(holder, PytorchActivationQuantizationHolder):
            why[node.target] = "the input is not the output of an activation quantization holder"
        elif getattr(holder, "quantization_bypass", False):
            why[node.target] = f"the input holder {src.target} bypasses quantization"
        elif node.target in edges and edges[node.target][0] != src.target:
            why[node.target] = "the wrapper is called on the outputs of different holders"
        else:
            edges[node.target] = (src.target, holder.activation_holder_quantizer)
    return edges, why, ""


class PackedState:
    """Per-wrapper packed state (the wrapper's `_packed` attribute): its PackedWeight entries, whether the wrapper runs in
    fused linear mode (and batched linear mode), and the launch state of its forward (the unpack plan / the fused-linear descriptor, built on first use
    and rebuilt when the codes move; not pickled)."""
    fused = False
    batched = False             # class default: states pickled before batched mode existed load with it off
    integer = False             # integer linear mode (and its input quantizer): off for states pickled before it existed
    input_quantizer = None

    def __init__(self, entries: List[PackedWeight]):
        self.entries = entries
        self.fused = False
        self.batched = False
        self.integer, self.input_quantizer = False, None
        self._plan, self._sig, self._lin, self._ilin = None, None, None, None

    def __getstate__(self):
        return {'entries': self.entries, 'fused': self.fused, 'batched': self.batched, 'integer': self.integer,
                'input_quantizer': self.input_quantizer, '_plan': None, '_sig': None, '_lin': None, '_ilin': None}

    def bind(self, wrapper):
        """Point the entries at `wrapper` (after a copy or unpickling they point nowhere)."""
        for e in self.entries:
            if e._owner is None or e._owner() is not wrapper:
                e._owner = weakref.ref(wrapper)

    def weight_vars(self, wrapper):
        self.bind(wrapper)
        return [(e.name, e, e.quantizer) for e in self.entries]

    def _signature(self):
        return [e.codes.data_ptr() for e in self.entries]

    def rebuild(self, wrapper) -> List[torch.Tensor]:
        """All packed weights of the wrapper, freshly allocated, in ONE unpack launch (per kernel variant)."""
        self.bind(wrapper)
        sig = self._signature()
        if self._plan is None or sig != self._sig:
            self._plan = ops.UnpackPlan([e.plan_item() for e in self.entries], fresh=True)
            self._sig = sig
        return self._plan.run()

    def fused_forward(self, wrapper, x):
        """x @ W^T + b from the codes (mctq_packed_linear), or None when this call must take the exact packed path: x is not
        a plain CUDA tensor on the codes' device with the rebuilt weight's dtype (and the bias's), autograd would record the
        call, the layer has forward hooks, a compiler is tracing, or x has more than FUSED_LINEAR_MAX_ROWS rows (batched
        mode: more than FUSED_BATCHED_MAX_ROWS rows; rows above FUSED_LINEAR_MAX_ROWS take mctq_packed_linear_batched)."""
        e = self.entries[0]
        if e._owner is None or e._owner() is not wrapper:
            self.bind(wrapper)
        if type(x) not in ops._PLAIN_TENSOR_TYPES or not x.is_cuda or x.dtype != e.dtype_out or x.dim() == 0:
            return None
        layer = wrapper.__dict__['_modules'][LAYER]
        in_f = layer.in_features
        limit = (FUSED_BATCHED_MAX_ROWS if self.__dict__.get('batched', False) else FUSED_LINEAR_MAX_ROWS).get(x.dtype, 0)
        if x.shape[-1] != in_f or x.numel() > limit * in_f:
            return None
        bias = layer.bias
        if bias is not None and (bias.dtype != x.dtype or bias.device != x.device):
            return None
        if torch.is_grad_enabled() and (x.requires_grad or (bias is not None and bias.requires_grad)):
            return None
        if layer._forward_hooks or layer._forward_pre_hooks or _nn_module._global_forward_hooks or \
                _nn_module._global_forward_pre_hooks or torch.compiler.is_compiling():
            return None
        codes = e.codes
        if x.device != codes.device:
            return None
        lin = self.__dict__.get('_lin')
        if lin is None or lin[0] != codes.data_ptr():
            item = e.plan_item()
            lin = (codes.data_ptr(), ops.PackedLinear(codes, e.kind, e.is_signed, e.dtype_out, layer.out_features, in_f,
                                                      item[8], item[9], item[10]))
            self._lin = lin
        if x.numel() > FUSED_LINEAR_MAX_ROWS.get(x.dtype, 0) * in_f:
            return lin[1].batched(x, bias)
        return lin[1](x, bias)

    def integer_forward(self, wrapper, x):
        """layer(Q(x)) in integer arithmetic (ops.IntegerLinear, or ops.IntegerConv2d / ops.IntegerDepthwiseConv2d for a
        Conv2d layer), or None when this
        call must take the packed path of the wrapper's other modes: the conditions of fused_forward, without its row limit;
        a Conv2d layer also needs a 4-D x."""
        e = self.entries[0]
        if e._owner is None or e._owner() is not wrapper:
            self.bind(wrapper)
        if type(x) not in ops._PLAIN_TENSOR_TYPES or not x.is_cuda or x.dtype != e.dtype_out or x.dim() == 0:
            return None
        layer = wrapper.__dict__['_modules'][LAYER]
        bias = layer.bias
        conv = type(layer) is torch.nn.Conv2d
        if conv:
            if x.dim() != 4 or x.shape[1] != layer.in_channels:
                return None
        elif x.shape[-1] != layer.in_features:
            return None
        if bias is not None and (bias.dtype != x.dtype or bias.device != x.device):
            return None
        if torch.is_grad_enabled() and (x.requires_grad or (bias is not None and bias.requires_grad)):
            return None
        if layer._forward_hooks or layer._forward_pre_hooks or _nn_module._global_forward_hooks or \
                _nn_module._global_forward_pre_hooks or torch.compiler.is_compiling():
            return None
        codes = e.codes
        if x.device != codes.device:
            return None
        lin = self.__dict__.get('_ilin')
        if lin is None or lin[0] != codes.data_ptr():
            q = self.input_quantizer
            from mct_quantizers_b200.pytorch.fused_activation_holder import affine_scalar_params
            scale, zp, _, _ = affine_scalar_params(q)
            x_scale, x_zp, qmin, qmax = q._validated_launch_args(scale, zp)[1]      # what the holder's kernel receives
            item = e.plan_item()
            scale, zps, lut = item[8], item[9], None
            if e.kind in _native.PACK_LUT_KINDS:         # codes lut_k, scale thr * 2^-(bw-1) (exact: _lut_eligibility)
                wq = e.quantizer
                scale, lut = scale * 2.0 ** -(int(wq.lut_values_bitwidth) - 1), wq._lut_values_np
            if conv and layer.groups > 1:              # switched by integer_depthwise_eligibility
                launch = ops.IntegerDepthwiseConv2d(codes, e.kind, e.is_signed, e.dtype_out, layer.out_channels,
                                                    layer.in_channels, layer.kernel_size, e.stride_out, layer.stride,
                                                    layer.dilation, ops.conv_padding(layer), scale, zps, x_scale, x_zp, qmin,
                                                    qmax, lut)
            elif conv:
                launch = ops.IntegerConv2d(codes, e.kind, e.is_signed, e.dtype_out, layer.out_channels, layer.in_channels,
                                           layer.kernel_size, e.stride_out, layer.stride, layer.dilation,
                                           ops.conv_padding(layer), scale, zps, x_scale, x_zp, qmin, qmax, lut, pad=True)
            else:
                launch = ops.IntegerLinear(codes, e.kind, e.is_signed, e.dtype_out, layer.out_features, layer.in_features,
                                           scale, zps, x_scale, x_zp, qmin, qmax, lut, pad=True)
            lin = (codes.data_ptr(), launch)
            self._ilin = lin
        return lin[1](x, bias)

    def forward(self, wrapper, args, kwargs):
        if torch.jit.is_tracing():
            raise RuntimeError("this PytorchQuantizationWrapper holds packed weights (pack_weights / pack_model_weights): "
                               "they cannot be traced or exported to ONNX, which needs the float weights; export the "
                               "model before packing it")
        if self.__dict__.get('integer', False) and len(args) == 1 and not kwargs:
            y = self.integer_forward(wrapper, args[0])
            if y is not None:
                return y
        if self.fused and len(args) == 1 and not kwargs:
            y = self.fused_forward(wrapper, args[0])
            if y is not None:
                return y
        d = wrapper.__dict__
        if d.get('_prequantized', False):              # a ModelWeightPlan has installed this forward's weights
            return wrapper._run_layer(args, kwargs)
        weights = dict(zip((e.name for e in self.entries), self.rebuild(wrapper)))
        for (name, w, q), wants_training in zip(wrapper._weights_vars, wrapper._training_flags()):
            weights[name] = q(w, d['training']) if wants_training else q(w)
        wrapper.set_quantize_weights(weights)
        try:
            return wrapper._run_layer(args, kwargs)
        finally:
            wrapper.set_quantize_weights({})               # drop the rebuilt weights: only the codes stay resident


def pack_wrapper_weights(wrapper, fused_linear: bool = False, batched_linear: bool = False, integer_linear: bool = False,
                         input_quantizer=None, integer_conv: bool = False, integer_lut: bool = False,
                         integer_depthwise: bool = False, integer_pad: bool = False) -> Dict:
    """Pack every weight of `wrapper` that can be packed (see the module docstring).  Returns
    {name: {'packed': bool, 'kind': str | None, 'reason': str, 'code_bytes': int, 'float_bytes': int}}.
    `fused_linear=True` also switches the wrapper to fused linear mode when fused_linear_eligibility allows it (on a wrapper
    packed earlier it only switches the mode), and every report entry gains 'fused': bool and 'fused_reason': str.
    `batched_linear=True` (needs fused_linear=True) also switches it to batched linear mode when batched_linear_eligibility
    allows it, and every report entry gains 'batched': bool and 'batched_reason': str.
    `integer_linear=True` (needs `input_quantizer`, the quantizer of the activation holder whose output the wrapper reads)
    also switches it to integer linear mode when integer_linear_eligibility allows it, and every report entry gains
    'integer': bool, 'integer_reason': str and 'input_holder' (the holder's module name for pack_model_weights, else None).
    `integer_conv=True` (needs `input_quantizer` too) does the same for integer convolution mode (integer_conv_eligibility),
    and every report entry gains 'integer_conv': bool, 'integer_conv_reason': str and 'input_holder'.
    `integer_lut=True` (needs integer_linear=True and / or integer_conv=True) extends those modes to LUT weights.
    `integer_depthwise=True` (needs integer_conv=True) extends integer convolution mode to depthwise Conv2d layers
    (integer_depthwise_eligibility); their report entries keep the keys 'integer_conv' and 'integer_conv_reason'.
    `integer_pad=True` (needs integer_linear=True and / or integer_conv=True) lifts the row-length and channel-count rules
    of those modes: the codes of such Linear and groups-1 Conv2d layers are padded (DESIGN §7f)."""
    if batched_linear and not fused_linear:
        raise ValueError("batched_linear=True needs fused_linear=True (batched mode extends the fused mode)")
    _check_integer_lut(integer_lut, integer_linear, integer_conv)
    _check_integer_depthwise(integer_depthwise, integer_conv)
    _check_integer_pad(integer_pad, integer_linear, integer_conv)
    if integer_linear and input_quantizer is None:
        raise ValueError("integer_linear=True needs the input_quantizer of the activation holder that feeds the wrapper")
    if integer_conv and input_quantizer is None:
        raise ValueError("integer_conv=True needs the input_quantizer of the activation holder that feeds the wrapper")
    report = {}
    state = wrapper.__dict__.get('_packed')
    entries = list(state.entries) if state is not None else []
    keep, new = [], []
    for name, w, q in wrapper.get_weights_vars():
        kind, reason = packing_kind(q, w)
        if kind is None:
            keep.append((name, w, q))
            report[name] = dict(packed=False, kind=None, reason=reason, code_bytes=0,
                                float_bytes=w.numel() * w.element_size() if isinstance(w, torch.Tensor) else 0)
            continue
        y_ref = q(w)                                    # layout and values the rebuilt weight must reproduce
        codes, is_signed, C, inner = _emit_codes(q, w, kind)
        e = PackedWeight(wrapper, name, q, kind, is_signed, y_ref.dtype, y_ref.shape, y_ref.stride(), C, inner)
        wrapper.register_buffer(e.codes_name, codes)
        if kind in _native.PACK_LUT_KINDS:
            wrapper.register_buffer(e.quot_name, _lut_quotients_host(q).to(w.device).view(torch.int32))
        rebuilt = ops.UnpackPlan([e.plan_item()]).run()[0]
        if rebuilt.stride() != y_ref.stride() or not torch.equal(_bits(rebuilt), _bits(y_ref)):
            raise RuntimeError(f"packing weight {name!r}: the rebuilt weight differs from quantizer(weight)")
        new.append((e, w))
        report[name] = dict(packed=True, kind=_KIND_NAMES[kind], reason="", code_bytes=codes.numel() * codes.element_size(),
                            float_bytes=w.numel() * w.element_size())
    if new:
        _drop_float_weights(wrapper, new, entries, keep)
    if fused_linear:
        _switch_to_fused(wrapper, report)
    if batched_linear:
        _switch_to_batched(wrapper, report)
    if integer_linear:
        _switch_to_integer(wrapper, report, input_quantizer, None, lut=integer_lut, pad=integer_pad)
    if integer_conv:
        _switch_to_integer(wrapper, report, input_quantizer, None, conv=True, lut=integer_lut, depthwise=integer_depthwise,
                           pad=integer_pad)
    return report


def _check_integer_lut(integer_lut, integer_linear, integer_conv):
    if integer_lut and not (integer_linear or integer_conv):
        raise ValueError("integer_lut=True needs integer_linear=True and / or integer_conv=True (it extends those modes to "
                         "LUT weights)")


def _check_integer_depthwise(integer_depthwise, integer_conv):
    if integer_depthwise and not integer_conv:
        raise ValueError("integer_depthwise=True needs integer_conv=True (it extends integer convolution mode to depthwise "
                         "Conv2d layers)")


def _check_integer_pad(integer_pad, integer_linear, integer_conv):
    if integer_pad and not (integer_linear or integer_conv):
        raise ValueError("integer_pad=True needs integer_linear=True and / or integer_conv=True (it extends those modes to "
                         "row lengths and channel counts off the GEMM's granule)")


def _drop_float_weights(wrapper, new, entries, keep):
    # drop every reference to the float weights: the wrapper's parameter, the layer attribute (or the positional constant)
    for e, w in new:
        if wrapper.is_str_attr:
            delattr(wrapper, e.name)
            setattr(wrapper.layer, e.name, None)
        else:
            delattr(wrapper, f'{POSITIONAL_WEIGHT}_{e.name}')
            setattr(wrapper, f'{QUANTIZED_POSITIONAL_WEIGHT}_{e.name}', None)
            wrapper.weight_values[e.name] = None
        entries.append(e)
        e.quantizer.__dict__.pop('_direct_cache', None)      # launch constants of the float weight's path (pin its tables)
    wrapper._weights_vars = keep
    wrapper._training_arg = None
    state = wrapper.__dict__.get('_packed')
    wrapper._packed = PackedState(entries)
    wrapper._packed.fused = state is not None and state.fused
    wrapper._packed.batched = state is not None and state.batched
    if state is not None and state.__dict__.get('integer', False):
        wrapper._packed.integer, wrapper._packed.input_quantizer = True, state.input_quantizer


def _switch_to_fused(wrapper, report):
    ok, reason = fused_linear_eligibility(wrapper)
    state = wrapper.__dict__.get('_packed')
    if ok:
        state.fused, state._lin = True, None
    _report_packed_entries(wrapper, report)
    for r in report.values():
        r['fused'], r['fused_reason'] = ok, reason


def _switch_to_batched(wrapper, report):
    ok, reason = batched_linear_eligibility(wrapper)
    state = wrapper.__dict__.get('_packed')
    if ok:
        state.batched, state._lin = True, None
    for r in report.values():
        r['batched'], r['batched_reason'] = ok, reason


def _switch_to_integer(wrapper, report, input_quantizer, holder_name, reason=None, conv=False, lut=False, depthwise=False,
                       pad=False):
    eligibility = functools.partial(integer_conv_eligibility if conv else integer_linear_eligibility, pad=pad)
    layer = wrapper.__dict__['_modules'].get(LAYER)
    if conv and depthwise and type(layer) is torch.nn.Conv2d and layer.groups > 1:
        eligibility = integer_depthwise_eligibility
    ok, why = (False, reason) if reason else eligibility(wrapper, input_quantizer, lut=lut)
    state = wrapper.__dict__.get('_packed')
    if ok:
        state.integer, state.input_quantizer, state._ilin = True, input_quantizer, None
    _report_packed_entries(wrapper, report)
    flag, flag_reason = ('integer_conv', 'integer_conv_reason') if conv else ('integer', 'integer_reason')
    for r in report.values():
        r[flag], r[flag_reason], r['input_holder'] = ok, why, holder_name


def _report_packed_entries(wrapper, report):
    state = wrapper.__dict__.get('_packed')
    for e in (state.entries if state is not None else []):
        if e.name not in report:                      # packed by an earlier call
            report[e.name] = dict(packed=True, kind=_KIND_NAMES[e.kind], reason="already packed",
                                  code_bytes=e.codes.numel() * e.codes.element_size(), float_bytes=0)


def _bits(t):
    return t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int16)


def pack_model_weights(model: torch.nn.Module, fused_linear: bool = False, batched_linear: bool = False,
                       integer_linear: bool = False, integer_conv: bool = False, integer_lut: bool = False,
                       integer_depthwise: bool = False, integer_pad: bool = False) -> Dict[str, Dict]:
    """pack_weights(fused_linear, batched_linear) on every PytorchQuantizationWrapper of `model`: {wrapper module name:
    {weight name: report entry}}.  `integer_linear=True` then switches, in place, every eligible wrapper whose input is the
    output of an activation quantization holder (integer_linear_edges) to integer linear mode; every report entry gains
    'integer', 'integer_reason' and 'input_holder'.  `integer_conv=True` does the same for integer convolution mode on the
    same edges; every report entry gains 'integer_conv', 'integer_conv_reason' and 'input_holder'.  `integer_lut=True` extends
    both to LUT weights, and `integer_depthwise=True` extends integer convolution mode to depthwise Conv2d layers.
    `integer_pad=True` lifts the row-length and channel-count rules of both (padded codes, DESIGN §7f).  When the
    model cannot be traced nothing is switched and the reason is reported."""
    if batched_linear and not fused_linear:
        raise ValueError("batched_linear=True needs fused_linear=True (batched mode extends the fused mode)")
    _check_integer_lut(integer_lut, integer_linear, integer_conv)
    _check_integer_depthwise(integer_depthwise, integer_conv)
    _check_integer_pad(integer_pad, integer_linear, integer_conv)
    from mct_quantizers_b200.pytorch.quantize_wrapper import PytorchQuantizationWrapper
    wrappers = {mod_name: mod for mod_name, mod in model.named_modules()
                if isinstance(mod, PytorchQuantizationWrapper) and mod.is_weights_quantization}
    reports = {name: pack_wrapper_weights(mod, fused_linear, batched_linear) for name, mod in wrappers.items()}
    if integer_linear or integer_conv:
        edges, why, failure = integer_linear_edges(model)
        for name, mod in wrappers.items():
            holder, q = edges.get(name, (None, None)) if name not in why else (None, None)
            reason = failure or why.get(name) or ("" if holder else "the wrapper is not called in the traced forward")
            for conv in (False, True) if integer_linear and integer_conv else (integer_conv,):
                _switch_to_integer(mod, reports[name], q, holder, None if holder else reason, conv=conv, lut=integer_lut,
                                   depthwise=integer_depthwise, pad=integer_pad)
    return reports
