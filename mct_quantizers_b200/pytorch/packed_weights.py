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

Packing is one-way and for inference only:
  * the rebuild dtype is the weight's dtype at packing time; `.half()` does not change it (the codes are integer buffers);
  * the packed state travels with the module: `state_dict` / `load_state_dict` between packed models of the same structure,
    `.to(device)`, `torch.save` + `pytorch_load_quantized_model`;
  * a packed wrapper cannot be traced (ONNX export needs the float weights, which are gone) and cannot be trained.
"""
import weakref
from typing import Dict, List, Optional, Tuple

import torch

from mct_quantizers_b200 import _native, ops
from mct_quantizers_b200.common.constants import POSITIONAL_WEIGHT, QUANTIZED_POSITIONAL_WEIGHT

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
        if self.kind in (_native.PACK_LUT_U8, _native.PACK_LUT_I4):
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
    if kind in (_native.PACK_LUT_U8, _native.PACK_LUT_I4):
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


class PackedState:
    """Per-wrapper packed state (the wrapper's `_packed` attribute): its PackedWeight entries and the unpack plan of its
    forward (built on first use, rebuilt when the codes move; not pickled)."""

    def __init__(self, entries: List[PackedWeight]):
        self.entries = entries
        self._plan, self._sig = None, None

    def __getstate__(self):
        return {'entries': self.entries, '_plan': None, '_sig': None}

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

    def forward(self, wrapper, args, kwargs):
        if torch.jit.is_tracing():
            raise RuntimeError("this PytorchQuantizationWrapper holds packed weights (pack_weights / pack_model_weights): "
                               "they cannot be traced or exported to ONNX, which needs the float weights; export the "
                               "model before packing it")
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


def pack_wrapper_weights(wrapper) -> Dict:
    """Pack every weight of `wrapper` that can be packed (see the module docstring).  Returns
    {name: {'packed': bool, 'kind': str | None, 'reason': str, 'code_bytes': int, 'float_bytes': int}}."""
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
        if kind in (_native.PACK_LUT_U8, _native.PACK_LUT_I4):
            quot = ops.lut_quotients(q._lut_values_torch, q.lut_values_bitwidth, True).to(w.device)
            wrapper.register_buffer(e.quot_name, quot.view(torch.int32))
        rebuilt = ops.UnpackPlan([e.plan_item()]).run()[0]
        if rebuilt.stride() != y_ref.stride() or not torch.equal(_bits(rebuilt), _bits(y_ref)):
            raise RuntimeError(f"packing weight {name!r}: the rebuilt weight differs from quantizer(weight)")
        new.append((e, w))
        report[name] = dict(packed=True, kind=_KIND_NAMES[kind], reason="", code_bytes=codes.numel() * codes.element_size(),
                            float_bytes=w.numel() * w.element_size())
    if not new:
        return report
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
    wrapper._packed = PackedState(entries)
    return report


def _bits(t):
    return t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int16)


def pack_model_weights(model: torch.nn.Module) -> Dict[str, Dict]:
    """pack_weights() on every PytorchQuantizationWrapper of `model`: {wrapper module name: {weight name: report entry}}."""
    from mct_quantizers_b200.pytorch.quantize_wrapper import PytorchQuantizationWrapper
    return {mod_name: pack_wrapper_weights(mod) for mod_name, mod in model.named_modules()
            if isinstance(mod, PytorchQuantizationWrapper) and mod.is_weights_quantization}
