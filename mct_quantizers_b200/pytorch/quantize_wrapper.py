"""PytorchQuantizationWrapper: owns a layer's float weights and hands the layer their fake-quantized version
on every forward.  Reference: mct_quantizers/pytorch/quantize_wrapper.py:29-270.

Differences that do not change results:
  * whether a quantizer's __call__ takes a `training` argument is looked up once per quantizer instead of
    calling inspect.signature on every forward (17 us per weight in the reference);
  * `quantize_weights_batched()` / the module-level `quantize_model_weights()` run all affine weight quantizers
    of a wrapper / a whole model in ONE kernel launch (mctq_fq_affine_multi).
"""
import inspect
from typing import List, Union, Any, Dict, Tuple, Callable

import torch
import torch.nn as nn

from mct_quantizers_b200.common.base_inferable_quantizer import BaseInferableQuantizer
from mct_quantizers_b200.common.constants import LAYER, TRAINING, POSITIONAL_WEIGHT, QUANTIZED_POSITIONAL_WEIGHT
from mct_quantizers_b200.logger import Logger


def _takes_training(quantizer) -> bool:
    return TRAINING in inspect.signature(quantizer.__call__).parameters


class PytorchQuantizationWrapper(nn.Module):
    def __init__(self,
                 module: Union[nn.Module, Callable],
                 weights_quantizers: Dict[Union[int, str], BaseInferableQuantizer],
                 weight_values: Dict[int, torch.Tensor] = None,
                 op_call_args: List = None,
                 op_call_kwargs: Dict[str, Any] = None,
                 is_inputs_as_list: bool = False):
        """
        Args:
            module: an nn.Module or a functional op (torch.sub, torch.cat ...).
            weights_quantizers: weight attribute name (str) or positional index (int) -> quantizer.
            weight_values: positional index -> constant tensor, for functional ops with constant inputs.
            op_call_args / op_call_kwargs: extra call arguments of a functional op.
            is_inputs_as_list: the op takes its tensor inputs as one list (torch.cat).
        """
        super().__init__()
        if isinstance(module, nn.Module):
            self.add_module(LAYER, module)
        else:
            setattr(self, LAYER, module)        # functional op

        self.weights_quantizers = weights_quantizers
        self.weight_values = weight_values if weight_values is not None else dict()
        for pos, weight_val in self.weight_values.items():
            if not isinstance(weight_val, torch.Tensor):
                Logger.error(f'Positional weight at position {pos} should be a torch.Tensor, '
                             f'but type is {type(weight_val)}.')

        self.op_call_args = [] if op_call_args is None else op_call_args
        self.op_call_kwargs = {} if op_call_kwargs is None else op_call_kwargs
        self.is_inputs_as_list = is_inputs_as_list

        # either all weights are named attributes of the layer (str keys) or all are positional constants
        # (int keys matching weight_values); mixing is not supported
        if len(self.weight_values) == 0:
            if not all(isinstance(w, str) for w in self.weights_quantizers):
                Logger.error('"weights_quantizers" keys should be all strings')
            self.is_str_attr = True
        else:
            if not all(isinstance(w, int) for w in self.weight_values):
                Logger.error('All "weight_values" keys should be integers')
            if not all(a == b for a, b in zip(weights_quantizers, weight_values)):
                Logger.error('Mismatch between "weights_quantizers" and "weight_values" keys')
            self.is_str_attr = False

        self._set_weights_vars(True)

    @property
    def is_weights_quantization(self) -> bool:
        return self.num_weights_quantizers > 0

    @property
    def num_weights_quantizers(self) -> int:
        return len(self.weights_quantizers)

    def convert_to_inferable_quantizers(self):
        """Replace trainable quantizers (objects exposing convert2inferable) by their inferable twins."""
        if self.is_weights_quantization:
            inferable = {}
            for name, quantizer in self.weights_quantizers.items():
                if hasattr(quantizer, 'convert2inferable') and callable(quantizer.convert2inferable):
                    inferable.update({name: quantizer.convert2inferable()})
            self.weights_quantizers = inferable
            self._set_weights_vars(False)

    def _set_weights_vars(self, is_training: bool = True):
        """Move the float weights out of the layer into parameters of the wrapper and bind each to its quantizer."""
        self._weights_vars = []
        self._training_arg = []
        for name, quantizer in self.weights_quantizers.items():
            if self.is_str_attr:
                source = self.layer if is_training else self
                weight = getattr(source, name).detach()
                delattr(self.layer, name)
                setattr(self.layer, name, weight)
                if is_training:
                    self.register_parameter(name, torch.nn.Parameter(weight, requires_grad=True))
                weight_var = getattr(self, name)
            else:
                weight = self.weight_values[name]
                self.register_parameter(f'{POSITIONAL_WEIGHT}_{name}', torch.nn.Parameter(weight, requires_grad=False))
                setattr(self, f'{QUANTIZED_POSITIONAL_WEIGHT}_{name}', weight)
                weight_var = getattr(self, f'{POSITIONAL_WEIGHT}_{name}')
            quantizer.initialize_quantization(weight.shape, name, self)
            self._weights_vars.append((name, weight_var, quantizer))
            self._training_arg.append(_takes_training(quantizer))

    def set_quantize_weights(self, quantized_weights: dict):
        """Install quantized weights into the layer (named) or the wrapper's positional slots."""
        for weight_attr in self.weights_quantizers:
            weight = quantized_weights.get(weight_attr)
            if self.is_str_attr:
                setattr(self.layer, weight_attr, weight)
            else:
                setattr(self, f'{QUANTIZED_POSITIONAL_WEIGHT}_{weight_attr}', weight)

    def get_weights_vars(self) -> List[Tuple[str, Any, BaseInferableQuantizer]]:
        return self._weights_vars

    def _training_flags(self):
        flags = getattr(self, '_training_arg', None)
        if flags is None or len(flags) != len(self._weights_vars):    # e.g. unpickled from an older object
            flags = [_takes_training(q) for _, _, q in self._weights_vars]
            self._training_arg = flags
        return flags

    def forward(self, *args: List[Any], **kwargs: Dict[str, Any]) -> Union[torch.Tensor, List[torch.Tensor]]:
        d = self.__dict__
        packed = d.get('_packed')
        if packed is not None:              # packed weights (pack_weights): rebuilt from their codes, see packed_weights.py
            return packed.forward(self, args, kwargs)
        # Lean path for the usual case -- an nn.Module layer with named weights and no extra call arguments: same effects as
        # the general path below (every weight quantized, the result installed as the layer's attribute, the layer called)
        # without nn.Module's __getattr__ / __setattr__ detours, which cost more than the launch of a small weight
        # (13 -> 7 us of Python per wrapped layer and forward).
        layer = d['_modules'].get(LAYER)
        if layer is not None and d['is_str_attr'] and not d['op_call_args'] and not d['op_call_kwargs'] \
                and not d['is_inputs_as_list'] and type(self).set_quantize_weights is PytorchQuantizationWrapper.set_quantize_weights:
            if not d.get('_prequantized', False):
                wv = d['_weights_vars']
                flags = d.get('_training_arg')
                if flags is None or len(flags) != len(wv):
                    flags = self._training_flags()
                ld = layer.__dict__
                for (name, weight, quantizer), wants_training in zip(wv, flags):
                    qw = quantizer(weight, d['training']) if wants_training else quantizer(weight)
                    if name in ld:
                        ld[name] = qw               # a plain attribute since _set_weights_vars: what setattr would do
                    else:
                        setattr(layer, name, qw)
            return layer(*args, **kwargs)

        # (a ModelWeightPlan that is active has already installed this forward's quantized weights: model_quantization.py)
        if self.is_weights_quantization and not self.__dict__.get('_prequantized', False):
            quantized_weights = {}
            for (name, unquantized_weight, quantizer), wants_training in zip(self._weights_vars, self._training_flags()):
                if wants_training:
                    quantized_weights[name] = quantizer(unquantized_weight, self.training)
                else:
                    quantized_weights[name] = quantizer(unquantized_weight)
            self.set_quantize_weights(quantized_weights)
        return self._run_layer(args, kwargs)

    def _run_layer(self, args, kwargs):
        """Call the layer on the installed (quantized) weights."""
        if not self.is_str_attr:
            # splice the (quantized) constants back into the positional inputs at their recorded positions
            args = list(args)
            for pos in sorted(self.weights_quantizers):
                args.insert(pos, getattr(self, f'{QUANTIZED_POSITIONAL_WEIGHT}_{pos}'))

        _kwargs = {**self.op_call_kwargs, **kwargs}
        if self.is_inputs_as_list:
            return self.layer(args, *self.op_call_args, **_kwargs)
        return self.layer(*args, *self.op_call_args, **_kwargs)

    def get_quantized_weights(self) -> Dict[str, torch.Tensor]:
        """weight name / position -> quantized weight (the quantizers run; the layer does not).  Packed weights are rebuilt
        from their codes."""
        out = {name: quantizer(w) for name, w, quantizer in self.get_weights_vars()}
        packed = self.__dict__.get('_packed')
        if packed is not None:
            out.update(zip((e.name for e in packed.entries), packed.rebuild(self)))
        return out

    def pack_weights(self, fused_linear: bool = False, batched_linear: bool = False, integer_linear: bool = False,
                     input_quantizer=None, integer_conv: bool = False, integer_lut: bool = False,
                     integer_depthwise: bool = False, integer_pad: bool = False) -> Dict[str, Dict]:
        """Keep the weights of this wrapper as int8 / int4 codes or LUT indices instead of floats (inference only, one-way;
        see mct_quantizers_b200.pytorch.packed_weights).  Returns, per weight, whether it was packed and why not.
        `fused_linear=True`: a packed nn.Linear wrapper computes small-batch products straight from its codes (opt-in: not
        bit-identical to the float layer; the report says per weight whether the mode applies).  `batched_linear=True`
        (with fused_linear): batched inputs too, on the tensor cores.  `integer_linear=True` with `input_quantizer` (the
        quantizer of the activation holder whose output this wrapper reads): layer(Q(x)) as an exact integer product of
        8-bit codes on the tensor cores (see packed_weights).  `integer_conv=True` with `input_quantizer`: the same for a
        Conv2d layer, as an implicit GEMM of the codes.  `integer_lut=True` (with either): LUT weights too, their indices
        looked up as int8 codes in the GEMM.  `integer_depthwise=True` (with integer_conv): depthwise Conv2d layers too,
        as an exact int32 window sum of the codes.  `integer_pad=True` (with integer_linear / integer_conv): row lengths and
        channel counts off the GEMM's granule too, their codes padded with Q's zero-point code."""
        from mct_quantizers_b200.pytorch.packed_weights import pack_wrapper_weights
        return pack_wrapper_weights(self, fused_linear, batched_linear, integer_linear, input_quantizer, integer_conv,
                                    integer_lut, integer_depthwise, integer_pad)

    def quantize_weights_batched(self) -> Dict[str, torch.Tensor]:
        """get_quantized_weights() with every affine weight quantizer of this wrapper fused into one launch."""
        from mct_quantizers_b200.pytorch.model_quantization import quantize_weight_vars
        return quantize_weight_vars(self.get_weights_vars())
