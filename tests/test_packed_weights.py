"""Packed weight storage: int8 / int4 affine codes and LUT indices rebuilt bit-exactly (csrc/mctq_unpack.cu,
ops.UnpackPlan / mctq::dequantize_lut, pytorch/packed_weights.py)."""
import copy
import ctypes
import os
import warnings

import numpy as np
import pytest
import torch

import golden_util as G
import mct_quantizers_b200 as mctq
from mct_quantizers_b200 import _native, ops
from mct_quantizers_b200.pytorch import quantizers as Q
from mct_quantizers_b200.pytorch.packed_weights import code_kind, packing_kind, pack_model_weights

LUT_CASES = [n for n in G.case_names() if G.get_case(n)["cls"].startswith("WeightsLUT")]


# --------------------------------------------------------------------------------------------- CPU
def dequant_lut_reference(idx, lut, thr, C, inner, bw, signed):
    """LUT indices (into the original centroid list) -> values, the last two lines of the reference's lut_quantizer restated
    in numpy f32 (IEEE division and multiplication, no contraction): y = (lut[idx] / 2^(bw - signed)) * thr[c]."""
    idx = np.ascontiguousarray(idx).reshape(-1).astype(np.int64)
    q = np.asarray(lut, dtype=np.float32).reshape(-1) / np.float32(2.0 ** (bw - int(bool(signed))))
    thr = np.asarray(thr, dtype=np.float32).reshape(-1)
    assert thr.size == C and idx.min(initial=0) >= 0 and idx.max(initial=0) < q.size
    c = (np.arange(idx.size, dtype=np.int64) // inner) % C
    return (q[idx] * thr[c]).astype(np.float32)


@pytest.mark.parametrize("name", LUT_CASES)
def test_lut_indices_dequantise_to_y(name):
    """The LUT analogue of test_codes_dequantise_to_y: oracle indices -> dequant_lut_reference == the reference's y, bitwise."""
    case = G.get_case(name)
    out = G.oracle_run(case)
    p = out["p"]
    y = dequant_lut_reference(out["idx"], p["lut"], p["thr"], p["C"], p["inner"], p["bw"], p["signed"]).reshape(case["y"].shape)
    assert G.bits_equal(y, case["y"]), G.mismatch_report(y, case["y"])
    assert out["idx"].min() >= 0 and out["idx"].max() < p["lut"].size


@pytest.mark.parametrize("bw,signed", [(8, True), (4, True), (12, True), (8, False)])
def test_lut_quotients_are_the_reference_division(bw, signed):
    lut = torch.tensor([-(2 ** (bw - 1)), -3.0, 0.0, 1.0, 5.0, 2 ** (bw - 1) - 1]) if signed else torch.tensor([0.0, 3.0, 2.0 ** bw - 1])
    want = lut.to(torch.float32) / 2 ** (bw - int(signed))
    got = ops.lut_quotients(lut, bw, signed)
    assert got.dtype == torch.float32 and got.device.type == "cpu"
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))


def _desc(n, C, inner, kind=_native.PACK_AFFINE_I8, dtype=_native.F32, codes=0x7f0000000000, y=0x7f1000000000, K=16):
    d = _native.MctqPackedDesc()
    d.codes, d.y, d.n, d.C, d.inner = codes, y, n, C, inner
    d.kind, d.is_signed, d.y_dtype, d.K = kind, 1, dtype, K
    d.scale = 0x7f2000000000
    lut = kind in (_native.PACK_LUT_U8, _native.PACK_LUT_I4)
    d.zp, d.lut_quotients = (None, 0x7f4000000000) if lut else (0x7f3000000000, None)
    return d


def _plan(ds):
    lib = _native.load()
    arr = (_native.MctqPackedDesc * len(ds))(*ds)
    p = ctypes.cast(arr, ctypes.c_void_p)
    nb = lib.mctq_unpack_plan_bytes(p, len(ds))
    if nb == 0:
        return lib.mctq_unpack_plan(p, len(ds), None, 0), None
    buf = (ctypes.c_uint8 * nb)()
    total = lib.mctq_unpack_plan(p, len(ds), ctypes.cast(buf, ctypes.c_void_p), nb)
    return total, ctypes.c_int32.from_buffer(buf, 8).value        # (total tiles, launches)


def test_unpack_plan_host_compiler():
    """mctq_unpack_plan is host-only code (device pointers are never dereferenced): validation, variant selection, tile
    counts, grouping by variant and at most 64 tensors per launch."""
    assert ctypes.sizeof(_native.MctqPackedDesc) == 80
    tile4, tile8 = 256 * 4 * 4, 256 * 4 * 8
    assert _plan([_desc(tile4 * 3, 64, 192)]) == (3, 1)                                   # int8 codes, f32 rows of 192: V = 4
    assert _plan([_desc(tile8 * 2, 64, 256, kind=_native.PACK_AFFINE_I4)]) == (2, 1)      # int4 per channel, rows % 8: V = 8
    assert _plan([_desc(tile8 * 2, 64, 256, dtype=_native.BF16)]) == (2, 1)               # 2-byte outputs: V = 8
    assert _plan([_desc(tile4 + 1, 1, 1)]) == (2, 1)                                      # ragged tail, odd n
    # four kinds (and an output dtype) = five variants = five launches
    total, launches = _plan([_desc(tile4, 16, 256), _desc(tile8, 1, 1, kind=_native.PACK_LUT_U8, K=200),
                             _desc(tile8, 16, 512, kind=_native.PACK_LUT_I4), _desc(tile8, 16, 512, kind=_native.PACK_AFFINE_I4),
                             _desc(tile8, 16, 512, dtype=_native.F16)])
    assert launches == 5 and total == 1 + 2 + 1 + 1 + 1                   # per-tensor f32 LUT_U8: 4-element vectors
    # one variant: tensors share launches of <= 64
    for count, want in ((64, 1), (65, 2), (130, 3)):
        assert _plan([_desc(960, 8, 120) for _ in range(count)]) == (count, want)
    # empty tensors are accepted and skipped
    assert _plan([_desc(0, 1, 1, codes=0, y=0), _desc(100, 1, 1)]) == (1, 1)
    assert _plan([_desc(0, 1, 1, codes=0, y=0)]) == (0, 0)
    # malformed descriptors
    assert _plan([_desc(100, 1, 1, kind=5)]) == (-1, None)
    assert _plan([_desc(100, 1, 1, dtype=3)]) == (-2, None)
    assert _plan([_desc(100, 1, 1, kind=_native.PACK_LUT_U8, dtype=_native.BF16)]) == (-2, None)   # LUT outputs are f32
    assert _plan([_desc(100, 1, 1, kind=_native.PACK_LUT_I4, K=17)]) == (-4, None)
    assert _plan([_desc(100, 1, 1, kind=_native.PACK_LUT_U8, K=257)]) == (-4, None)
    assert _plan([_desc(100, 1, 1, kind=_native.PACK_LUT_U8, K=0)]) == (-4, None)
    assert _plan([_desc(100, 3, 1)]) == (-1, None)                                        # n is not outer * C * inner
    assert _plan([_desc(-1, 1, 1)]) == (-1, None)
    assert _plan([_desc(100, 1, 1, codes=0x7f0000000004)]) == (-1, None)                  # misaligned codes
    assert _plan([_desc(100, 1, 1, y=0x7f1000000008)]) == (-1, None)                      # misaligned output
    assert _plan([_desc(100, 1, 1, codes=0)]) == (-1, None)
    d = _desc(100, 1, 1)
    d.zp = None
    assert _plan([d]) == (-1, None)                                                       # affine needs zero points
    assert _plan([_desc(100, 1, 1), _desc(100, 1, 1, kind=0)]) == (-1, None)              # one bad tensor fails the plan
    # several faults in one descriptor: kind -> dtype -> LUT dtype -> n / C / inner -> empty -> pointers -> parameters
    assert _plan([_desc(100, 3, 1, kind=5, dtype=3)]) == (-1, None)
    assert _plan([_desc(100, 3, 1, dtype=3)]) == (-2, None)
    assert _plan([_desc(100, 1, 1, kind=_native.PACK_LUT_I4, dtype=_native.BF16, K=17)]) == (-2, None)
    assert _plan([_desc(100, 3, 1, kind=_native.PACK_LUT_I4, K=17)]) == (-1, None)
    assert _plan([_desc(100, 1, 1, kind=_native.PACK_LUT_I4, K=17, codes=0x7f0000000004)]) == (-1, None)
    d = _desc(0, 1, 1, kind=_native.PACK_LUT_I4, K=17, codes=0, y=0)
    d.lut_quotients = None
    assert _plan([d]) == (0, 0)                                                           # empty: parameters unchecked
    d = _desc(0, 1, 1, codes=0, y=0)
    d.zp = None
    assert _plan([d, _desc(100, 1, 1)]) == (1, 1)
    lib = _native.load()
    assert lib.mctq_unpack_plan(None, 1, None, 0) == -1 and lib.mctq_unpack_multi(None, None) == -1


def _lut_q(K, per_channel=True, axis=0, C=4, rank=2, bw=8, num_bits=None, pot=False):
    half = 2 ** (bw - 1)
    rng = np.random.default_rng(K)
    lut = sorted(rng.choice(np.arange(-half, half), size=K, replace=False).tolist())
    thr = [2.0 ** int(rng.integers(-2, 2)) if pot else float(rng.uniform(0.5, 2.0)) for _ in range(C if per_channel else 1)]
    cls = Q.WeightsLUTPOTInferableQuantizer if pot else Q.WeightsLUTSymmetricInferableQuantizer
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return cls(num_bits=num_bits or max(1, int(np.ceil(np.log2(K)))), lut_values=[float(v) for v in lut], threshold=thr,
                   per_channel=per_channel, channel_axis=axis if per_channel else None, input_rank=rank if per_channel else None,
                   lut_values_bitwidth=bw)


class _UserQ:
    """A user-defined weight quantizer (not one of the built-in classes: the registry must not see it)."""

    def __init__(self, *args):
        pass

    def initialize_quantization(self, *args):
        pass

    def __call__(self, inputs):
        return inputs * 0.5


def test_packing_decisions():
    w = torch.zeros(4, 6)
    sym8 = Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 4, True, 0)
    assert code_kind(sym8, w) == (_native.PACK_AFFINE_I8, "")
    assert code_kind(Q.WeightsSymmetricInferableQuantizer(4, [1.0], False), w) == (_native.PACK_AFFINE_I4, "")
    assert code_kind(Q.WeightsPOTInferableQuantizer(3, [1.0] * 4, True, 0), w) == (_native.PACK_AFFINE_I4, "")
    assert code_kind(Q.WeightsUniformInferableQuantizer(8, [-1.0] * 4, [1.0] * 4, True, 0), w) == (_native.PACK_AFFINE_I8, "")
    assert code_kind(Q.WeightsUniformInferableQuantizer(4, [-1.0], [1.0], False), w) == (_native.PACK_AFFINE_I4, "")
    assert code_kind(_lut_q(16), w) == (_native.PACK_LUT_I4, "")
    assert code_kind(_lut_q(17), w) == (_native.PACK_LUT_U8, "")
    assert code_kind(_lut_q(256, num_bits=8), w) == (_native.PACK_LUT_U8, "")
    assert code_kind(_lut_q(2, pot=True), w) == (_native.PACK_LUT_I4, "")
    # what keeps its float weight, and why
    assert "built-in" in code_kind(_UserQ(8, [1.0] * 4, True, 0), w)[1]
    assert "wider" not in code_kind(Q.WeightsSymmetricInferableQuantizer(9, [1.0], False), w)[1]
    assert code_kind(Q.WeightsSymmetricInferableQuantizer(9, [1.0], False), w)[0] is None
    assert "8-bit codes" in code_kind(Q.WeightsUniformInferableQuantizer(12, [-1.0], [1.0], False), w)[1]
    reuse = Q.WeightsSymmetricInferableQuantizer(8, [1.0], False)
    reuse.enable_reuse_quantizer()
    assert "enable_reuse" in code_kind(reuse, w)[1]
    custom = Q.WeightsSymmetricInferableQuantizer(8, [1.0], False)
    custom.enable_custom_impl()
    assert "_use_custom_impl" in code_kind(custom, w)[1]
    bad_zp = Q.WeightsUniformInferableQuantizer(8, [-1.0] * 4, [1.0] * 4, True, 0)
    bad_zp._zero_point_out_of_range = True                 # what the constructor records when ATen would refuse the zero point
    assert "zero point" in code_kind(bad_zp, w)[1]
    assert "input_rank" in code_kind(_lut_q(16, rank=4), w)[1]
    assert "dtype" in code_kind(sym8, w.double())[1]
    assert packing_kind(sym8, w) == (None, "the weight is not on a CUDA device")


# --------------------------------------------------------------------------------------------- GPU
class _Holder(torch.nn.Module):
    def __init__(self, w):
        super().__init__()
        self.weight = torch.nn.Parameter(w)

    def forward(self, x):
        return x


def _bits(t):
    t = t.detach().contiguous()
    return t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int16)


def _check_rebuilt(q, w, want_kind):
    y_ref = q(w.clone())
    wrapper = mctq.PytorchQuantizationWrapper(_Holder(w), {"weight": q})
    report = wrapper.pack_weights()
    assert report["weight"]["packed"], report
    assert report["weight"]["kind"] == want_kind
    assert "weight" not in dict(wrapper.named_parameters())
    got = wrapper.get_quantized_weights()["weight"]
    assert got.dtype == y_ref.dtype and got.shape == y_ref.shape and got.stride() == y_ref.stride()
    assert torch.equal(_bits(got), _bits(y_ref))
    # and through the forward: the layer sees the rebuilt weight, which is dropped afterwards
    seen = {}
    wrapper.layer.forward = lambda x: seen.setdefault("w", wrapper.layer.weight.clone())
    wrapper(torch.zeros(1, device=w.device))
    assert torch.equal(_bits(seen["w"]), _bits(y_ref)) and wrapper.layer.weight is None


AFFINE_SHAPES = [((64, 40), 0), ((33, 5), 1), ((6, 7, 3), -1), ((16, 8, 3, 3), 0), ((7,), 0), ((1,), 0), ((0, 4), 1), ((5, 24), 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("qname", ["sym8", "sym4", "pot4", "uni8", "uni4"])
@pytest.mark.parametrize("per_channel", [True, False])
def test_affine_rebuilt_equals_quantizer(dtype, qname, per_channel):
    g = torch.Generator().manual_seed(7)
    for shape, axis in AFFINE_SHAPES:
        w = (torch.randn(shape, generator=g) * 2).to("cuda", dtype)
        C = shape[axis] if per_channel else 1
        bits = int(qname[-1])
        thr = [float(2 ** int(v)) for v in torch.randint(-1, 2, (C,), generator=g)]
        if qname.startswith("sym"):
            q = Q.WeightsSymmetricInferableQuantizer(bits, thr, per_channel, axis if per_channel else None)
        elif qname.startswith("pot"):
            q = Q.WeightsPOTInferableQuantizer(bits, thr, per_channel, axis if per_channel else None)
        else:
            q = Q.WeightsUniformInferableQuantizer(bits, [-t for t in thr], [t * 0.75 for t in thr], per_channel,
                                                   axis if per_channel else None)
        _check_rebuilt(q, w, "affine_i4" if bits == 4 else "affine_i8")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_channels_last_conv_weights(dtype):
    w = torch.randn(32, 16, 3, 3).to("cuda", dtype).to(memory_format=torch.channels_last)
    for axis in (0, 1):
        q = Q.WeightsSymmetricInferableQuantizer(8, [0.5 + 0.01 * c for c in range(w.shape[axis])], True, axis)
        _check_rebuilt(q, w.clone(memory_format=torch.channels_last), "affine_i8")
    q = Q.WeightsUniformInferableQuantizer(4, [-1.0], [1.0], False)
    _check_rebuilt(q, w.clone(memory_format=torch.channels_last), "affine_i4")


LUT_SHAPES = [((64, 40), 0), ((33, 5), 1), ((6, 7, 3), -1), ((7,), 0), ((1,), 0), ((0, 4), 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("K", [2, 16, 17, 256])
@pytest.mark.parametrize("per_channel", [True, False])
def test_lut_rebuilt_equals_quantizer(dtype, K, per_channel):
    g = torch.Generator().manual_seed(K)
    for shape, axis in LUT_SHAPES:
        w = (torch.randn(shape, generator=g) * 1.5).to("cuda", dtype)
        q = _lut_q(K, per_channel, axis, C=shape[axis], rank=len(shape), num_bits=8 if K > 128 else None, pot=K == 2)
        _check_rebuilt(q, w, "lut_i4" if K <= 16 else "lut_u8")
    if not per_channel:                                            # 0-dim weights come back 1-D, like the reference
        _check_rebuilt(_lut_q(K, False, num_bits=8 if K > 128 else None), torch.tensor(0.3, device="cuda", dtype=dtype),
                       "lut_i4" if K <= 16 else "lut_u8")


@pytest.mark.gpu
@pytest.mark.parametrize("device", ["cuda", "cpu"])
@pytest.mark.parametrize("K,idx_mode", [(16, 2), (16, 1), (100, 1)])
def test_dequantize_lut_inverts_lut_indices(device, K, idx_mode):
    q = _lut_q(K, True, 1, C=24, rank=3)
    x = torch.randn(5, 24, 33, device=device)
    table = mctq.pytorch.quantizer_utils.lut_search_table(q._lut_values_np, q.lut_values_bitwidth, True)
    thr = q._threshold_torch.to(device).reshape(-1)
    want = torch.ops.mctq.fq_lut_tensor(x, table, K, thr, True, 1, float(q.eps))
    idx = torch.ops.mctq.lut_indices(x, table, K, thr, True, 1, float(q.eps), idx_mode)
    got = torch.ops.mctq.dequantize_lut(idx, idx_mode, list(x.shape), q._lut_values_torch.to(device), q.lut_values_bitwidth,
                                        True, thr, True, 1)
    assert got.device.type == device and got.shape == want.shape and torch.equal(_bits(got), _bits(want))
    # per tensor, 0-dim
    x0 = torch.tensor(-0.7, device=device)
    thr0 = thr[:1].clone()
    want0 = torch.ops.mctq.fq_lut_tensor(x0, table, K, thr0, False, 0, float(q.eps))
    idx0 = torch.ops.mctq.lut_indices(x0, table, K, thr0, False, 0, float(q.eps), idx_mode)
    got0 = torch.ops.mctq.dequantize_lut(idx0, idx_mode, [], q._lut_values_torch.to(device), q.lut_values_bitwidth, True, thr0,
                                         False, 0)
    assert got0.shape == (1,) and torch.equal(_bits(got0), _bits(want0.reshape(1)))


@pytest.mark.gpu
def test_one_launch_of_many_tensors_of_all_kinds():
    """> 64 tensors mixing the four kinds in one plan: bitwise results and the expected number of launches."""
    g = torch.Generator().manual_seed(3)
    wrappers, refs = [], []
    for k in range(80):
        kind = k % 4
        rows = 40 + 8 * (k % 3)
        w = torch.randn(rows, 96, generator=g).cuda()
        if kind == 0:
            q = Q.WeightsSymmetricInferableQuantizer(8, [1.0 + 0.01 * r for r in range(rows)], True, 0)
        elif kind == 1:
            q = Q.WeightsUniformInferableQuantizer(4, [-2.0] * rows, [1.5] * rows, True, 0)
        elif kind == 2:
            q = _lut_q(40, True, 0, C=rows)
        else:
            q = _lut_q(16, True, 0, C=rows)
        refs.append(q(w.clone()))
        wrappers.append(mctq.PytorchQuantizationWrapper(torch.nn.Linear(96, rows, bias=False).cuda(), {"weight": q}))
        wrappers[-1]._weights_vars[0][1].data.copy_(w)
    model = torch.nn.ModuleList(wrappers)
    pack_model_weights(model)
    x = torch.randn(2, 96, device="cuda")
    # per wrapper: one launch per forward
    before = _native.launch_count()
    for m, ref in zip(wrappers, refs):
        assert torch.equal(_bits(m(x)), _bits(torch.nn.functional.linear(x, ref)))
    torch.cuda.synchronize()
    assert _native.launch_count() - before == len(wrappers)
    # under the plan: one launch per variant group (4 kinds, 20 tensors each) for all 80 tensors
    plan = mctq.plan_model_weights(model)
    (idx, unpack), = plan.plan._unpack_plans
    assert len(idx) == 80 and unpack.n_launches == 4
    before = _native.launch_count()
    plan.refresh()
    torch.cuda.synchronize()
    assert _native.launch_count() - before == 4
    for m, ref in zip(wrappers, refs):
        assert torch.equal(_bits(m.layer.weight), _bits(ref))
    # 130 tensors of one variant: three launches
    items = [m._packed.entries[0].plan_item() for m in wrappers if m._packed.entries[0].kind == _native.PACK_AFFINE_I8] * 7
    big = ops.UnpackPlan(items[:130])
    before = _native.launch_count()
    outs = big.run()
    torch.cuda.synchronize()
    assert big.n_launches == 3 and _native.launch_count() - before == 3
    i8_refs = [r for k, r in enumerate(refs) if k % 4 == 0] * 7
    assert all(torch.equal(_bits(o), _bits(r)) for o, r in zip(outs, i8_refs[:130]))


def _tv_model(name, dtype=torch.float32):
    import torchvision
    import importlib.util
    spec = importlib.util.spec_from_file_location("mfb", os.path.join(os.path.dirname(__file__), "..", "tools", "model_forward_bench.py"))
    mfb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mfb)
    torch.manual_seed(0)
    m = getattr(torchvision.models, name)(weights=None).eval()
    return mfb.quantize_model(m, mctq, Q).to("cuda", dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mobilenet_v2", "resnet18"])
def test_torchvision_logits_bit_equal(name):
    model = _tv_model(name)
    x = torch.randn(4, 3, 224, 224, device="cuda")
    with torch.no_grad():
        want = model(x)
        packed = copy.deepcopy(model)
        report = pack_model_weights(packed)
        assert all(r["packed"] for rep in report.values() for r in rep.values())
        assert torch.equal(packed(x), want)                                       # eager
        with mctq.plan_model_weights(packed):
            assert torch.equal(packed(x), want)                                   # whole-model unpack launch
        fused = mctq.fuse_activation_producers(copy.deepcopy(packed))
        assert torch.equal(fused(x), want)                                        # producers fused into the holders
        static_x = x.clone()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                packed(static_x)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_y = packed(static_x)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_y, want)                                        # replayed from a CUDA graph


def _lut_linear_model(dtype, n_layers=2, out_f=11008, in_f=4096):
    torch.manual_seed(0)
    layers = []
    for _ in range(n_layers):
        lin = torch.nn.Linear(in_f, out_f, bias=False, device="cuda", dtype=dtype)
        layers.append(mctq.PytorchQuantizationWrapper(lin, {"weight": _lut_q(16, True, 0, C=out_f, rank=2)}))
        in_f, out_f = out_f, in_f
    return torch.nn.Sequential(*layers)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,limit", [(torch.float32, 0.135), (torch.bfloat16, 0.26)])
def test_packed_memory(dtype, limit):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    model = _lut_linear_model(dtype)
    before = torch.cuda.memory_allocated() - base
    x = torch.randn(4, 4096, device="cuda")                  # LUT weights rebuild as f32, whatever the storage dtype
    with torch.no_grad():
        want = model(x)
        for m in model:
            m.layer.weight = None                 # drop the fake-quantized copies the float forward leaves behind
        pack_model_weights(model)
        ops.clear_lut_caches()                    # the quantizers' prepared tables (built by the float path) are not weights
        torch.cuda.synchronize()
        after = torch.cuda.memory_allocated() - base
        assert after <= limit * before, (after, before)
        torch.cuda.reset_peak_memory_stats()
        resident = torch.cuda.memory_allocated()
        got = model(x)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - resident
        largest_rebuilt = 4096 * 11008 * 4                                    # LUT weights rebuild as f32
        activations = 2 * 4 * 11008 * x.element_size() + (1 << 20)
        assert peak <= largest_rebuilt + activations, (peak, largest_rebuilt)
    assert torch.equal(got, want)


def _small_packed(seed):
    torch.manual_seed(seed)
    m = torch.nn.Sequential(torch.nn.Conv2d(3, 16, 3, bias=False), torch.nn.ReLU(), torch.nn.Flatten(),
                            torch.nn.Linear(16 * 6 * 6, 10, bias=False)).cuda()
    m[0] = mctq.PytorchQuantizationWrapper(m[0], {"weight": Q.WeightsSymmetricInferableQuantizer(8, [0.3] * 16, True, 0)})
    m[3] = mctq.PytorchQuantizationWrapper(m[3], {"weight": _lut_q(16, True, 0, C=10, rank=2)})
    pack_model_weights(m)
    return m


@pytest.mark.gpu
def test_round_trips(tmp_path):
    x = torch.randn(2, 3, 8, 8, device="cuda")
    a, b = _small_packed(0), _small_packed(1)
    with torch.no_grad():
        want = a(x)
        assert not torch.equal(b(x), want)
        b.load_state_dict(a.state_dict())
        assert torch.equal(b(x), want)                                            # state_dict between packed models
        path = os.path.join(tmp_path, "packed.pt")
        torch.save(a, path)
        c = mctq.pytorch_load_quantized_model(path)
        assert torch.equal(c(x), want)                                            # torch.save / load
        assert torch.equal(a.half()(x), want)                                     # the rebuild dtype stays the packing-time dtype
        import mct_quantizers_b200.compat  # noqa: F401
        import mct_quantizers
        assert isinstance(c[0], mct_quantizers.PytorchQuantizationWrapper)
        if torch.cuda.device_count() > 1:
            d = copy.deepcopy(c).to("cuda:1")
            assert torch.equal(d(x.to("cuda:1")).cpu(), want.cpu())               # .to(device)


@pytest.mark.gpu
def test_errors_and_fallbacks():
    x = torch.randn(2, 8, device="cuda")
    # ONNX-export tracing of a packed wrapper
    m = mctq.PytorchQuantizationWrapper(torch.nn.Linear(8, 4).cuda(), {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 4, True, 0)})
    m.pack_weights()
    m._packed.entries[0].quantizer.enable_custom_impl()
    with pytest.raises(RuntimeError, match="packed weights"):
        torch.jit.trace(m, x)
    # fallbacks keep their float weight and today's behaviour
    reuse = Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 4, True, 0)
    reuse.enable_reuse_quantizer()
    cases = {
        "user": _UserQ(8, [1.0] * 4, True, 0),
        "reuse": reuse,
        "wide": Q.WeightsUniformInferableQuantizer(12, [-1.0], [1.0], False),
        "zp": Q.WeightsUniformInferableQuantizer(8, [-1.0] * 4, [1.0] * 4, True, 0),
    }
    cases["zp"]._zero_point_out_of_range = True
    for key, q in cases.items():
        lin = torch.nn.Linear(8, 4).cuda()
        ref = copy.deepcopy(lin)
        w = mctq.PytorchQuantizationWrapper(lin, {"weight": q})
        report = w.pack_weights()
        assert not report["weight"]["packed"] and report["weight"]["reason"]
        assert "weight" in dict(w.named_parameters()) and w.__dict__.get("_packed") is None
        if key == "zp":
            with pytest.raises(RuntimeError, match="zero_point"):
                w(x)
        elif key != "reuse":
            assert torch.equal(w(x), torch.nn.functional.linear(x, q(ref.weight.detach()), ref.bias))
    cpu = mctq.PytorchQuantizationWrapper(torch.nn.Linear(8, 4), {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 4, True, 0)})
    assert cpu.pack_weights()["weight"]["reason"] == "the weight is not on a CUDA device"
