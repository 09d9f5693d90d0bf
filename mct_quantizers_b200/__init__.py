"""mct_quantizers_b200 -- B200-native fake-quant path behind the mct_quantizers (1.6.0) PyTorch API.

Same public names as the reference's mct_quantizers/__init__.py:16-34 for the PyTorch side (the Keras twin and the
ONNX-runtime session helpers are out of scope, see DESIGN.md)."""
__version__ = "1.6.0"

from mct_quantizers_b200.common.base_inferable_quantizer import QuantizationTarget, BaseInferableQuantizer, \
    mark_quantizer, QuantizerID
from mct_quantizers_b200.common.quant_info import QuantizationMethod
from mct_quantizers_b200.common import constants
from mct_quantizers_b200.common.get_quantizers import get_inferable_quantizer_class
from mct_quantizers_b200.pytorch.activation_quantization_holder import PytorchActivationQuantizationHolder
from mct_quantizers_b200.pytorch.fln_activation_quantization_holder import PytorchFLNActivationQuantizationHolder
from mct_quantizers_b200.pytorch.preserving_activation_quantization_holder import \
    PytorchPreservingActivationQuantizationHolder
from mct_quantizers_b200.pytorch.load_model import pytorch_load_quantized_model
from mct_quantizers_b200.pytorch.quantize_wrapper import PytorchQuantizationWrapper
from mct_quantizers_b200.pytorch.model_quantization import quantize_model_weights, plan_model_weights, ModelWeightPlan, \
    ActivationPlan, quantize_activations
from mct_quantizers_b200.pytorch.packed_weights import pack_model_weights
from mct_quantizers_b200.pytorch import quantizers as pytorch_quantizers
from mct_quantizers_b200.pytorch.fused_activation_holder import PytorchFusedActivationQuantizationHolder, \
    fuse_activation_producers
from mct_quantizers_b200.ops import host_pipeline, private_stream
from mct_quantizers_b200.pytorch.quantizer_utils import reference_arithmetic
