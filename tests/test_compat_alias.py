"""`mct_quantizers_b200.compat`: `import mct_quantizers` resolves to this package, and modules pickled by the UNMODIFIED
reference (tests/golden/ref_pickles/, made by tests/golden/make_ref_pickles.py) load as B200 objects that reproduce the
reference's results."""
import glob
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PICKLES = os.path.join(ROOT, "tests", "golden", "ref_pickles")
NAMES = sorted(os.path.basename(p)[:-3] for p in glob.glob(os.path.join(PICKLES, "*.pt")))


def test_alias_serves_the_reference_module_paths(tmp_path):
    """Run in a fresh interpreter, from an empty directory, so that the alias cannot collide with anything already
    imported or lying in the working directory."""
    code = r'''
import sys
sys.path.insert(0, %r)
import mct_quantizers_b200.compat
import mct_quantizers, mct_quantizers_b200
assert mct_quantizers is mct_quantizers_b200 and mct_quantizers.__version__ == "1.6.0"
from mct_quantizers.pytorch.quantizers.weights_inferable_quantizers.weights_symmetric_inferable_quantizer import WeightsSymmetricInferableQuantizer as A
from mct_quantizers.pytorch.quantizers.activation_inferable_quantizers.activation_lut_pot_inferable_quantizer import ActivationLutPOTInferableQuantizer
from mct_quantizers.pytorch.quantizers import WeightsSymmetricInferableQuantizer as B
from mct_quantizers_b200.pytorch.quantizers import WeightsSymmetricInferableQuantizer as C
assert A is B is C
from mct_quantizers.pytorch.quantizer_utils import get_working_device, to_torch_tensor
from mct_quantizers.common.constants import POSITIONAL_WEIGHT, QUANTIZED_POSITIONAL_WEIGHT
from mct_quantizers.common.get_quantizers import get_inferable_quantizer_class
from mct_quantizers.common.base_inferable_quantizer import QuantizationTarget, mark_quantizer, BaseInferableQuantizer
from mct_quantizers.common.quant_info import QuantizationMethod
from mct_quantizers.pytorch.quantizers.base_pytorch_inferable_quantizer import BasePyTorchInferableQuantizer
from mct_quantizers.pytorch.metadata import add_metadata, get_metadata
from mct_quantizers.pytorch.load_model import pytorch_load_quantized_model
from mct_quantizers import PytorchQuantizationWrapper, PytorchActivationQuantizationHolder, pytorch_quantizers
assert get_inferable_quantizer_class(QuantizationTarget.Weights, QuantizationMethod.SYMMETRIC, BasePyTorchInferableQuantizer) is A
for missing in ("mct_quantizers.keras", "mct_quantizers.pytorch.onnxruntime_session_options"):
    try:
        __import__(missing)
    except ModuleNotFoundError:
        pass
    else:
        raise AssertionError(missing + " should not resolve")
print("ok")
''' % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]


def _load(name):
    import mct_quantizers_b200.compat  # noqa: F401
    from mct_quantizers_b200 import pytorch_load_quantized_model
    return pytorch_load_quantized_model(os.path.join(PICKLES, name + ".pt"))


@pytest.mark.parametrize("name", NAMES)
def test_reference_pickles_load_as_b200_objects(name):
    import mct_quantizers_b200 as mctq
    m = _load(name)
    assert type(m).__module__.startswith("mct_quantizers_b200.")
    if name.startswith("holder"):
        assert isinstance(m, mctq.PytorchActivationQuantizationHolder.__mro__[0]) or hasattr(m, "activation_holder_quantizer")
        assert type(m.activation_holder_quantizer).__module__.startswith("mct_quantizers_b200.")
    else:
        assert isinstance(m, mctq.PytorchQuantizationWrapper)
        assert all(type(q).__module__.startswith("mct_quantizers_b200.") for q in m.weights_quantizers.values())


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_reference_pickles_reproduce_reference_results(name):
    exp = np.load(os.path.join(PICKLES, "expected.npz"))
    dev = torch.device("cuda:0")
    m = _load(name).to(dev)
    x = torch.from_numpy(exp[name + "/x"]).to(dev)
    with torch.no_grad():
        y = m(x)
    want = exp[name + "/y"]
    if name.startswith("holder"):
        assert np.array_equal(y.cpu().numpy().view(np.uint32), want.view(np.uint32)), name        # bit-exact
    else:
        qw = m.get_quantized_weights()
        for key in [k for k in exp.files if k.startswith(name + "/qw/")]:
            got = qw[key.split("/qw/")[1]].cpu().numpy()
            assert np.array_equal(got.view(np.uint32), exp[key].view(np.uint32)), key             # quantized weights: bit-exact
        # the wrapped conv / linear itself runs in cuDNN / cuBLAS (TF32 off by default for convs? allow float tolerance)
        assert np.allclose(y.cpu().numpy(), want, rtol=1e-3, atol=1e-3), name
