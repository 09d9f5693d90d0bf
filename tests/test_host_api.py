"""Host-side contract of the replacement package (no GPU): constructor-derived parameters vs the fixtures
generated from the reference, validation messages, registry, wrapper / holder plumbing with fake quantizers,
pickling and fx tracing, C-ABI symbol export, and the loud failure when no CUDA device is present."""
import ctypes
import io
import os
import pickle
import re
import warnings

import numpy as np
import pytest
import torch

import golden_util as G
import mct_quantizers_b200 as mctq
from mct_quantizers_b200 import _native
from mct_quantizers_b200.pytorch import quantizers as Q

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = G.case_names()
HAS_GPU = torch.cuda.is_available()


def _np(v):
    return v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)


@pytest.mark.parametrize("name", CASES)
def test_constructor_parameters_match_reference(name):
    """scales / zero points / fixed ranges / integer domain of the replacement == the reference's attributes."""
    case = G.get_case(name)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        q = getattr(Q, case["cls"])(**case["args"])
    for attr, meta in case["params"].items():
        got = getattr(q, attr)
        if meta["kind"] == "tensor":
            assert isinstance(got, torch.Tensor) and str(got.dtype) == "torch." + meta["dtype"], attr
            assert G.bits_equal(_np(got), case["p"][attr]), attr
        elif meta["kind"] == "ndarray":
            assert isinstance(got, (np.ndarray, np.generic)), attr
            assert np.array_equal(np.asarray(got), case["p"][attr]), attr
        else:
            assert type(got).__name__ == meta["kind"], (attr, type(got))
            assert got == meta["value"], attr


def test_attribute_types():
    w = Q.WeightsPOTInferableQuantizer(4, [2.0, 0.5], True, 1)
    assert isinstance(w.threshold_np, np.ndarray) and w.threshold == [2.0, 0.5]
    assert w.scales.dtype == torch.float32 and w.zero_points.dtype == torch.int32 and w.zero_points.shape == (2,)
    a = Q.ActivationPOTInferableQuantizer(8, [4.0], False)
    assert isinstance(a.scales, float) and a.zero_points == 0 and isinstance(a.threshold_np, np.generic)
    assert (a.min_quantized_domain, a.max_quantized_domain) == (0, 255)
    u = Q.ActivationUniformInferableQuantizer(8, [-1.0], [2.3])
    assert isinstance(u.scale, float) and isinstance(u.zero_point, int) and isinstance(u.min_range, float)
    wu = Q.WeightsUniformInferableQuantizer(8, [-1.0, 0.5], [2.0, 3.0], True, 0)
    assert isinstance(wu.adjusted_min_range_np, np.ndarray) and wu.zero_points.dtype == torch.int32
    assert float(wu.min_range[1]) == 0.0                                   # strictly positive range is re-anchored at 0
    lw = Q.WeightsLUTSymmetricInferableQuantizer(3, [-4.0, 0.0, 3.0], [1.0], False)
    assert lw.lut_values == [-4.0, 0.0, 3.0] and lw._lut_values_torch.dtype == torch.float32 and lw.eps == 1e-8
    la = Q.ActivationLutPOTInferableQuantizer(3, [0.0, 3.0, 200.0], [2.0], False)
    assert isinstance(la.threshold, float) and isinstance(la.lut_values, torch.Tensor)
    for q in (w, a, u, wu, lw, la):
        assert (q.reuse, q.enable_reuse, q.quantizer_first_run, q.resue_outputs, q._use_custom_impl) == (False, False, True, None, False)
    w.enable_reuse_quantizer()
    assert w.enable_reuse and w.quantizer_first_run
    w.disable_reuse_quantizer()
    assert not w.enable_reuse
    w.enable_custom_impl()
    assert w._use_custom_impl


ERRORS = [
    (lambda: Q.WeightsSymmetricInferableQuantizer(8, [1.0], True), 'Channel axis is missing in per channel quantization'),
    (lambda: Q.WeightsSymmetricInferableQuantizer(8, [1.0, 2.0], False), 'In per-tensor quantization threshold should be of length 1 but is 2'),
    (lambda: Q.WeightsPOTInferableQuantizer(8, [3.0], False), 'Expected threshold to be power of 2 but is [3.0]'),
    (lambda: Q.WeightsSymmetricInferableQuantizer(8, np.array([1.0]), False), "Threshold is expected to be a list, but is of type <class 'numpy.ndarray'>"),
    (lambda: Q.WeightsUniformInferableQuantizer(8, [1.0], [0.5], False), 'Max range must be greater than min value but min is 1.0 and max is 0.5'),
    (lambda: Q.WeightsUniformInferableQuantizer(8, [0.0], [1.0], True), 'Channel axis is missing in per channel quantization'),
    (lambda: Q.WeightsUniformInferableQuantizer(8, [0.0, 0.1], [1.0, 2.0], False), 'In per-tensor quantization min_range should be of length 1 but is 2'),
    (lambda: Q.ActivationSymmetricInferableQuantizer(8, [1.0, 2.0], True),
     'For activation, only per-tensor quantization is supported. Thus, threshold should be of length 1 but is 2'),
    (lambda: Q.ActivationPOTInferableQuantizer(8, [3.0], True), 'Expected threshold to be power of 2 but is [3.0]'),
    (lambda: Q.ActivationUniformInferableQuantizer(8, [0.0, 0.0], [1.0, 1.0]),
     'For activation, only per-tensor quantization is supported. Thus, min_range should be of length 1 but is 2'),
    (lambda: Q.WeightsLUTSymmetricInferableQuantizer(2, [-1.5, 0.0, 1.0], [1.0], False), 'Expected lut values to be integers'),
    (lambda: Q.WeightsLUTSymmetricInferableQuantizer(1, [-1.0, 0.0, 1.0], [1.0], False), 'Expected num of lut values to be less or equal than 2 but got 3'),
    (lambda: Q.WeightsLUTSymmetricInferableQuantizer(3, [-200.0, 0.0, 1.0], [1.0], False), 'Expected lut values in the quantization range'),
    (lambda: Q.ActivationLutPOTInferableQuantizer(3, [-1.0, 0.0, 1.0], [1.0], False), 'Expected unsigned lut values in unsigned activation quantization'),
    (lambda: Q.WeightsLUTSymmetricInferableQuantizer(9, [-1.0, 0.0, 1.0], [1.0], False), 'Look-Up-Table bit configuration has 9 bits. It must be less then 8'),
    (lambda: Q.ActivationLutPOTInferableQuantizer(3, [0.0, 1.0], [1.0, 2.0], True),
     'For activation, quantization per channel is not supported and threshold should be of length 1 but is 2'),
    (lambda: Q.WeightsLUTSymmetricInferableQuantizer(3, [0.0, 1.0], [1.0, 2.0], True, None, 2), 'Channel axis is missing in per channel quantization'),
    (lambda: Q.WeightsLUTSymmetricInferableQuantizer(3, [0.0, 1.0], [1.0, 2.0], True, 0), 'input_rank is missing in per channel quantization'),
    (lambda: Q.WeightsLUTPOTInferableQuantizer(3, [0.0, 1.0], [3.0], False), 'Expected threshold to be power of 2 but is [3.0]'),
    (lambda: Q.WeightsLUTSymmetricInferableQuantizer(3, (0.0, 1.0), [1.0], False), "lut_values is expected to be a list, but is of type <class 'tuple'>"),
]


@pytest.mark.parametrize("k", range(len(ERRORS)))
def test_validation_messages(k):
    fn, msg = ERRORS[k]
    with pytest.raises(AssertionError) as e:
        fn()
    assert str(e.value) == msg


def test_lut_bitwidth_warning():
    with pytest.warns(UserWarning, match="Num of bits equal to multiplier n bits"):
        Q.WeightsLUTSymmetricInferableQuantizer(8, [0.0, 1.0], [1.0], False)


def test_registry_finds_exactly_one_class():
    T, M = mctq.QuantizationTarget, mctq.QuantizationMethod
    base = Q.BasePyTorchInferableQuantizer
    expect = {(T.Weights, M.POWER_OF_TWO): Q.WeightsPOTInferableQuantizer, (T.Weights, M.SYMMETRIC): Q.WeightsSymmetricInferableQuantizer,
              (T.Weights, M.UNIFORM): Q.WeightsUniformInferableQuantizer, (T.Weights, M.LUT_SYM_QUANTIZER): Q.WeightsLUTSymmetricInferableQuantizer,
              (T.Weights, M.LUT_POT_QUANTIZER): Q.WeightsLUTPOTInferableQuantizer, (T.Activation, M.POWER_OF_TWO): Q.ActivationPOTInferableQuantizer,
              (T.Activation, M.SYMMETRIC): Q.ActivationSymmetricInferableQuantizer, (T.Activation, M.UNIFORM): Q.ActivationUniformInferableQuantizer,
              (T.Activation, M.LUT_POT_QUANTIZER): Q.ActivationLutPOTInferableQuantizer}
    for (t, m), cls in expect.items():
        assert mctq.get_inferable_quantizer_class(t, m, base) is cls
        assert cls.identifier is mctq.QuantizerID.INFERABLE and m in cls.quantization_method and cls.quantization_target == t
    with pytest.raises(Exception, match="Found 0 quantizer for target Activation"):
        mctq.get_inferable_quantizer_class(T.Activation, M.LUT_SYM_QUANTIZER, base)

    @mctq.mark_quantizer(quantization_target=T.Weights, quantization_method=[M.UNIFORM], identifier=mctq.QuantizerID.INFERABLE)
    class Duplicate(Q.BasePyTorchInferableQuantizer):
        def __call__(self, x):
            return x
    try:
        with pytest.raises(Exception, match="Found 2 quantizer"):
            mctq.get_inferable_quantizer_class(T.Weights, M.UNIFORM, base)
    finally:
        Duplicate.quantization_method = None
        assert mctq.get_inferable_quantizer_class(T.Weights, M.UNIFORM, base) is Q.WeightsUniformInferableQuantizer


# -------------------------------------------------------------------------------------------- wrapper / holders
class ZeroWeights(mctq.BaseInferableQuantizer):
    """Fake quantizer with a `training` argument (the wrapper must pass self.training)."""

    def __init__(self):
        super().__init__()
        self.seen_training = []

    def __call__(self, inputs, training):
        self.seen_training.append(training)
        return inputs * 0


class AddOne(mctq.BaseInferableQuantizer):
    def __call__(self, inputs):
        return inputs + 1


def test_wrapper_named_weights_with_fake_quantizer():
    conv = torch.nn.Conv2d(3, 4, 3)
    w0 = conv.weight.detach().clone()
    zq = ZeroWeights()
    wrapper = mctq.PytorchQuantizationWrapper(conv, {'weight': zq})
    assert wrapper.is_weights_quantization and wrapper.num_weights_quantizers == 1
    assert sorted(wrapper.state_dict().keys()) == ['layer.bias', 'weight']
    (name, w, q), = wrapper.get_weights_vars()
    assert name == 'weight' and q is zq and torch.equal(w.detach(), w0) and isinstance(w, torch.nn.Parameter)
    wrapper.eval()
    y = wrapper(torch.ones(1, 3, 8, 8))
    assert zq.seen_training == [False]
    assert torch.equal(wrapper.layer.weight, torch.zeros_like(w0))
    assert torch.allclose(y, conv.bias.detach().reshape(1, 4, 1, 1).expand_as(y))
    wrapper.train()
    wrapper(torch.ones(1, 3, 8, 8))
    assert zq.seen_training == [False, True]
    assert set(wrapper.weights_quantizers) == {'weight'}


def test_wrapper_positional_weights():
    sub = mctq.PytorchQuantizationWrapper(torch.sub, {0: AddOne()}, {0: torch.tensor([1.0, 2.0, 3.0])})
    assert torch.equal(sub(torch.tensor([1.0, 1.0, 1.0])), torch.tensor([1.0, 2.0, 3.0]))       # (c + 1) - x
    assert 'positional_weight_0' in dict(sub.named_parameters())
    cat = mctq.PytorchQuantizationWrapper(torch.cat, {0: AddOne(), 2: AddOne()},
                                          {0: torch.zeros(1, 2), 2: torch.ones(1, 2)}, op_call_kwargs={'dim': 0},
                                          is_inputs_as_list=True)
    out = cat(torch.full((1, 2), 5.0))
    assert torch.equal(out, torch.tensor([[1.0, 1.0], [5.0, 5.0], [2.0, 2.0]]))
    assert cat.get_quantized_weights().keys() == {0, 2}


def test_wrapper_validation_raises_through_logger():
    with pytest.raises(Exception, match='"weights_quantizers" keys should be all strings'):
        mctq.PytorchQuantizationWrapper(torch.nn.Linear(2, 2), {0: AddOne()})
    with pytest.raises(Exception, match='should be a torch.Tensor'):
        mctq.PytorchQuantizationWrapper(torch.sub, {0: AddOne()}, {0: [1.0]})
    with pytest.raises(Exception, match='Mismatch between "weights_quantizers" and "weight_values" keys'):
        mctq.PytorchQuantizationWrapper(torch.sub, {1: AddOne()}, {0: torch.ones(1)})
    with pytest.raises(Exception, match='All "weight_values" keys should be integers'):
        mctq.PytorchQuantizationWrapper(torch.sub, {'a': AddOne()}, {'a': torch.ones(1)})


def test_holders_and_bypass():
    h = mctq.PytorchActivationQuantizationHolder(AddOne())
    assert torch.equal(h(torch.zeros(3)), torch.ones(3))
    for cls in (mctq.PytorchFLNActivationQuantizationHolder, mctq.PytorchPreservingActivationQuantizationHolder):
        x = torch.zeros(3)
        assert torch.equal(cls(AddOne())(x), torch.ones(3))
        assert cls(AddOne(), quantization_bypass=True)(x) is x
        assert cls(AddOne(), True).quantization_bypass is True
    real = mctq.PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(7, [-4.0], [4.0]))
    q = real.activation_holder_quantizer
    assert np.isclose(q.min_range, -4.03149606299213) and np.isclose(q.max_range, 3.96850393700787)
    assert np.isclose(q.scale, 0.062992125984252) and q.zero_point == 64


def test_pickle_roundtrip_of_modules():
    """Quantizer objects carry numpy / torch state only (no ctypes handles), so wrappers and holders pickle."""
    conv = torch.nn.Conv2d(3, 4, 3)
    thr = [float(v) for v in conv.weight.detach().abs().flatten(1).amax(1)]
    model = torch.nn.Sequential(
        mctq.PytorchQuantizationWrapper(conv, {'weight': Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)}),
        mctq.PytorchActivationQuantizationHolder(Q.ActivationLutPOTInferableQuantizer(2, [0.0, 10.0, 100.0], [2.0], False)),
        mctq.PytorchFLNActivationQuantizationHolder(Q.ActivationPOTInferableQuantizer(8, [4.0], True), True))
    buf = io.BytesIO()
    torch.save(model, buf)
    buf.seek(0)
    loaded = torch.load(buf, weights_only=False)
    q0, q1 = model[0].weights_quantizers['weight'], loaded[0].weights_quantizers['weight']
    assert torch.equal(q0.scales, q1.scales) and q1.channel_axis == 0 and q1._per_device == {}
    assert loaded[2].quantization_bypass is True
    assert pickle.loads(pickle.dumps(Q.WeightsLUTPOTInferableQuantizer(2, [-8.0, 0.0, 4.0], [0.5], False))).lut_values == [-8.0, 0.0, 4.0]


def test_fx_trace_records_the_custom_op():
    holder = mctq.PytorchActivationQuantizationHolder(Q.ActivationSymmetricInferableQuantizer(8, [3.7], True))
    gm = torch.fx.symbolic_trace(torch.nn.Sequential(torch.nn.ReLU(), holder))
    targets = [n.target for n in gm.graph.nodes if n.op == 'call_function']
    assert torch.ops.mctq.fq_affine_scalar in targets or any('fq_affine_scalar' in str(t) for t in targets)
    node = [n for n in gm.graph.nodes if 'fq_affine_scalar' in str(n.target)][0]
    assert node.args[1:] == (3.7 / 128, 0, -128, 127)
    buf = io.BytesIO()
    torch.save(gm, buf)
    buf.seek(0)
    torch.load(buf, weights_only=False)


def test_meta_kernels_give_shapes_and_dtypes():
    x = torch.empty(4, 6, 5, dtype=torch.bfloat16, device='meta')
    assert torch.ops.mctq.fq_affine_scalar(x, 0.1, 0, -128, 127).dtype == torch.bfloat16
    s, z = torch.empty(6, device='meta'), torch.empty(6, dtype=torch.int32, device='meta')
    assert torch.ops.mctq.fq_affine_channel(x, s, z, 1, 0, 255).shape == x.shape
    tab = torch.empty(128, dtype=torch.uint8, device='meta')
    assert torch.ops.mctq.fq_lut_scalar(x, tab, 4, 1.0, 1.0, True).dtype == torch.float32
    codes, vals = torch.ops.mctq.quantize_affine_channel(x, s, z, 1, 0, 15, 2, False)
    assert codes.shape == (60,) and codes.dtype == torch.uint8 and vals.numel() == 0


# -------------------------------------------------------------------------------------------- native boundary
def test_shared_library_exports_every_declared_symbol():
    """Every function include/mctq.h declares is exported by libmctq_sm100.so and bound in _native.SIGNATURES."""
    header = open(os.path.join(ROOT, "include", "mctq.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(mctq_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_native.SIGNATURES), declared ^ set(_native.SIGNATURES)
    lib = _native.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.mctq_abi_version() == 1
    assert b"sm_100a" in lib.mctq_build_info()
    assert lib.mctq_lut_table_bytes(16) % 16 == 0 and lib.mctq_lut_table_bytes(0) == 0 and lib.mctq_lut_table_bytes(257) == 0
    assert ctypes.sizeof(_native.MctqTensorDesc) == 80
    # the cubin inside is sm_100a only
    assert os.path.getsize(_native.LIB_PATH) > 100000


def test_tuning_keys_and_staging_size():
    """mctq_set_tuning keeps key 3 (dependent-launch order) and key 9 (NVTX ranges) and rejects every other key; the
    host-buffer staging size is fixed: three slots of a 32 MiB input and a 64 MiB output chunk, plus 16 MiB of parameters."""
    lib = _native.load()
    for key in (-1, 0, 1, 2, 4, 5, 6, 7, 8, 10, 11, 12, 13):
        for value in (0, 1, 2, 3):
            assert lib.mctq_set_tuning(key, value) == -1, (key, value)          # MCTQ_E_BADARG
    prev = lib.mctq_set_tuning(3, 2)
    assert prev in (0, 1, 2, 3)
    assert lib.mctq_set_tuning(3, 3) == 2
    assert lib.mctq_set_tuning(3, 4) == -1
    assert lib.mctq_set_tuning(3, prev) == 3
    prev = lib.mctq_set_tuning(9, 1)
    assert prev in (0, 1)
    assert lib.mctq_set_tuning(9, prev) == 1
    assert lib.mctq_host_staging_min_bytes() == 3 * (32 + 64) * 2 ** 20 + 16 * 2 ** 20


def test_multi_plan_host_helper():
    lib = _native.load()
    descs = (_native.MctqTensorDesc * 3)()
    tile = lib.mctq_multi_tile_elems()
    for d, n in zip(descs, (1, tile, 3 * tile + 1)):
        d.n = n
    starts = (ctypes.c_int32 * 4)()
    total = lib.mctq_multi_plan(ctypes.cast(descs, ctypes.c_void_p), 3, ctypes.cast(starts, ctypes.c_void_p))
    assert total == 6 and list(starts) == [0, 1, 2, 6]


def test_lut_multi_plan_host_compiler():
    """mctq_lut_multi_plan is host-only code: descriptor validation, variant selection per tensor, tile counts, the grouping by
    kernel variant and the 64-tensors-per-launch chunking can be checked without a GPU (device pointers are never
    dereferenced here)."""
    lib = _native.load()
    assert ctypes.sizeof(_native.MctqLutTensorDesc) == 64

    def desc(n, C, inner, dtype=0, x=0x7f0000000000, y=0x7f1000000000, blob=0x7f2000000000, K=16, bw=8):
        d = _native.MctqLutTensorDesc()
        d.x, d.y, d.prepared_dev, d.n, d.C, d.inner = x, y, blob, n, C, inner
        d.dtype, d.K, d.lut_values_bitwidth, d.is_signed = dtype, K, bw, 1
        return d

    def plan(ds):
        arr = (_native.MctqLutTensorDesc * len(ds))(*ds)
        nb = lib.mctq_lut_multi_plan_bytes(ctypes.cast(arr, ctypes.c_void_p), len(ds))
        if nb == 0:
            return 0, lib.mctq_lut_multi_plan(ctypes.cast(arr, ctypes.c_void_p), len(ds), None, 0), None
        buf = (ctypes.c_uint8 * nb)()
        return nb, lib.mctq_lut_multi_plan(ctypes.cast(arr, ctypes.c_void_p), len(ds), ctypes.cast(buf, ctypes.c_void_p), nb), buf

    tile_f32 = 256 * 4 * 4                # threads x unroll x 4-element vectors, one tile per CTA
    tile_bf16_wide = 256 * 4 * 8          # 2-byte inputs, rows a multiple of 8: 8-element vectors
    nb, total, buf = plan([desc(tile_f32 * 3 + 1, 128, 4096), desc(5, 1, 1), desc(tile_bf16_wide * 2, 64, 4096, dtype=1),
                           desc(tile_f32 + 1, 64, 36, dtype=1)])       # rows of 36: not a multiple of 8 -> 4-element vectors
    assert total == 4 + 1 + 2 + 2 and nb > 64
    hdr = np.frombuffer(bytes(buf)[:32], dtype=np.int32)
    assert hdr[1] == 4 and hdr[2] == 4 and hdr[3] == 1                 # n_desc, four kernel variants = four launches, 1 tile per CTA
    # tensors of one variant share a launch
    _, total1, buf1 = plan([desc(tile_f32 * 2, 16, 4096), desc(tile_f32 * 5, 16, 8192), desc(tile_f32, 16, 4096)])
    assert total1 == 8 and np.frombuffer(bytes(buf1)[:32], dtype=np.int32)[2] == 1
    # more than 64 tensors of one variant: several launches, every one with its own tile numbering
    nb2, total2, buf2 = plan([desc(1000 + k, 8, 128) for k in range(400)])
    assert total2 == 400 and np.frombuffer(bytes(buf2)[:32], dtype=np.int32)[2] == 7
    assert nb2 > nb
    # tensors the prepared path cannot run are refused (the caller keeps them on their own call)
    assert plan([desc(100, 4, 25, x=0x7f0000000004)])[1] == -1         # misaligned x
    assert plan([desc(100, 4, 25, bw=14)])[1] == 1                     # grids of more than 10 bits: coarse cell table (prepare decides)
    assert plan([desc(100, 4, 25, bw=17)])[1] == -4                    # not a valid lut_values_bitwidth
    assert plan([desc(0, 1, 1)])[1] == -1                              # empty tensor
    assert plan([desc(100, 1, 1, dtype=5)])[1] == -2
    assert lib.mctq_fq_lut_prepared_multi(None, None) == -1


@pytest.mark.skipif(HAS_GPU, reason="checks the no-GPU failure mode")
def test_fails_loudly_without_a_gpu():
    """No CPU arithmetic path: a call on a machine without CUDA raises instead of silently computing elsewhere."""
    q = Q.ActivationSymmetricInferableQuantizer(8, [4.0], True)
    with pytest.raises(_native.MctqError, match="no CUDA device"):
        q(torch.randn(8))
    with pytest.raises(_native.MctqError):
        Q.WeightsLUTSymmetricInferableQuantizer(2, [0.0, 1.0], [1.0], False)(torch.randn(8))
    import mct_quantizers_b200 as mctq
    with pytest.raises(_native.MctqError, match="no CUDA device"):
        with mctq.host_pipeline():
            pass
    # whole-model plans never take host tensors into a launch: they stay on the per-layer call, which raises as above
    from mct_quantizers_b200.pytorch.model_quantization import WeightPlan
    plan = WeightPlan([("w", torch.randn(4, 8), Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 4, True, 0))])
    assert plan.plan is None and plan.lut_plan is None and len(plan.other) == 1
    with pytest.raises(_native.MctqError):
        plan.run()


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "mct_quantizers_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", src, flags=re.M), os.path.join(dirpath, f)


def test_reference_arithmetic_flavours():
    """`tensor / python_number` is a true division in libtorch's CPU kernel and a multiplication by the f32 reciprocal in its
    CUDA kernel, so the unmodified reference derives (slightly) different scales -- and now and then a different zero
    point -- on a CUDA machine.  Known answers: the 'cuda' column was printed by the unmodified reference running on a
    B200 (tools/differential_fuzz.py found the difference), the 'cpu' column by the same reference in the build container."""
    cases = [  # bits, min, max, (cuda scale, cuda zp), (cpu scale, cpu zp)
        (6, -1.4895310758373934, 4.583981513977051, (0.09640496969223022, 14), (0.09640496224164963, 15)),
        (3, -3.3297648164422617, 10.17188549041748, (1.928807258605957, 2), (1.9288071393966675, 2)),
        (4, -3.388154673240042, 6.393187046051025, (0.6520894765853882, 5), (0.6520894169807434, 5)),
        (4, -2.6913525735410344, 4.400905132293701, (0.47281718254089355, 6), (0.47281715273857117, 6)),
        (7, -1.866444401955146, 8.238741874694824, (0.07956839352846146, 23), (0.07956840097904205, 23)),
        (3, -2.1926928017257845, 3.288418769836426, (0.7830159664154053, 3), (0.7830159068107605, 3)),
    ]
    assert mctq.reference_arithmetic() == "cpu"
    try:
        for mode, col in (("cuda", 3), ("cpu", 4)):
            mctq.reference_arithmetic(mode)
            for c in cases:
                q = Q.WeightsUniformInferableQuantizer(c[0], [c[1]], [c[2]], False)
                assert np.float32(q.scales.cpu().item()) == np.float32(c[col][0]), (mode, c)
                assert int(q.zero_points.cpu().item()) == c[col][1], (mode, c)
        with pytest.raises(ValueError):
            mctq.reference_arithmetic("gpu")
    finally:
        mctq.reference_arithmetic("cpu")
