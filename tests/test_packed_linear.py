"""Fused packed linear (csrc/mctq_packed_linear.cu, torch.ops.mctq.packed_linear, fused linear mode of packed wrappers)."""
import copy
import ctypes
import os
import warnings

import numpy as np
import pytest
import torch

import mct_quantizers_b200 as mctq
from mct_quantizers_b200 import _native, ops
from mct_quantizers_b200.pytorch import quantizers as Q
from mct_quantizers_b200.pytorch.packed_weights import (FUSED_LINEAR_MAX_ROWS, PackedState, PackedWeight,
                                                        fused_linear_eligibility, pack_model_weights)
from test_packed_variants import decoded_f64

LUT_KINDS = (_native.PACK_LUT_U8, _native.PACK_LUT_I4)
U_OUT = {torch.float32: 2.0 ** -24, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}


def _lut_q(K, C, per_channel=True, axis=0, rank=2):
    rng = np.random.default_rng(K)
    lut = sorted(rng.choice(np.arange(-128, 128), size=K, replace=False).tolist())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return Q.WeightsLUTSymmetricInferableQuantizer(
            num_bits=max(1, int(np.ceil(np.log2(K)))), lut_values=[float(v) for v in lut],
            threshold=[float(rng.uniform(0.5, 2.0)) for _ in range(C if per_channel else 1)], per_channel=per_channel,
            channel_axis=axis if per_channel else None, input_rank=rank if per_channel else None, lut_values_bitwidth=8)


# --------------------------------------------------------------------------------------------- CPU
def _fake_packed(wrapper, name="weight", C=None, inner=None, shape=None, stride=None):
    """A PackedState built on the host (no codes buffer): what pack_weights leaves behind, for the eligibility rules."""
    layer = wrapper.layer
    shape = shape or tuple(layer.weight.shape)
    stride = stride or (shape[1], 1)
    e = PackedWeight(wrapper, name, wrapper.weights_quantizers[name], _native.PACK_AFFINE_I8, True, torch.float32, shape,
                     stride, C if C is not None else shape[0], inner if inner is not None else shape[1])
    wrapper._packed = PackedState([e])
    return wrapper


def test_fused_eligibility():
    sym = lambda C, axis=0: Q.WeightsSymmetricInferableQuantizer(8, [1.0] * C, True, axis)   # noqa: E731
    lin = mctq.PytorchQuantizationWrapper(torch.nn.Linear(6, 4), {"weight": sym(4)})
    assert fused_linear_eligibility(lin) == (False, "the weight is not packed")
    assert fused_linear_eligibility(_fake_packed(lin)) == (True, "")
    per_tensor = mctq.PytorchQuantizationWrapper(torch.nn.Linear(6, 4), {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0], False)})
    assert fused_linear_eligibility(_fake_packed(per_tensor, C=1, inner=1)) == (True, "")
    # channel_axis 1: per input channel
    ax1 = mctq.PytorchQuantizationWrapper(torch.nn.Linear(6, 4), {"weight": sym(6, 1)})
    ok, why = fused_linear_eligibility(_fake_packed(ax1, C=6, inner=1))
    assert not ok and "channel_axis 0" in why
    sq = mctq.PytorchQuantizationWrapper(torch.nn.Linear(4, 4), {"weight": sym(4, 1)})       # C == out, but inner == 1
    assert not fused_linear_eligibility(_fake_packed(sq, C=4, inner=1))[0]
    # conv, Linear subclass
    conv = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(3, 4, 1), {"weight": sym(4)})
    ok, why = fused_linear_eligibility(_fake_packed(conv, shape=(4, 3), stride=(3, 1), C=4, inner=3))
    assert not ok and "Conv2d" in why

    class MyLinear(torch.nn.Linear):
        pass
    sub = mctq.PytorchQuantizationWrapper(MyLinear(6, 4), {"weight": sym(4)})
    ok, why = fused_linear_eligibility(_fake_packed(sub))
    assert not ok and "MyLinear" in why
    # a second quantized weight
    two = mctq.PytorchQuantizationWrapper(torch.nn.Linear(6, 4), {"weight": sym(4), "bias": Q.WeightsSymmetricInferableQuantizer(8, [1.0], False)})
    ok, why = fused_linear_eligibility(_fake_packed(two))
    assert not ok and "other than 'weight'" in why
    # positional weights of a functional op
    pos = mctq.PytorchQuantizationWrapper(torch.nn.functional.linear, {1: sym(4)}, weight_values={1: torch.zeros(4, 6)})
    ok, why = fused_linear_eligibility(pos)
    assert not ok and "positional" in why
    # extra call arguments
    kw = mctq.PytorchQuantizationWrapper(torch.nn.Linear(6, 4), {"weight": sym(4)}, op_call_kwargs={"x": 1})
    assert not fused_linear_eligibility(_fake_packed(kw))[0]
    # a transposed rebuilt layout
    assert not fused_linear_eligibility(_fake_packed(copy.deepcopy(lin), stride=(1, 4)))[0]


def _lin_desc(out_f=10, in_f=33, kind=_native.PACK_AFFINE_I8, dtype=_native.F32, C=None, inner=None, K=16):
    d = _native.MctqPackedDesc()
    d.codes, d.y, d.n = 0x7f0000000000, None, out_f * in_f
    d.C = out_f if C is None else C
    d.inner = in_f if inner is None else inner
    d.kind, d.is_signed, d.y_dtype, d.K = kind, 1, dtype, K
    d.scale = 0x7f2000000000
    lut = kind in LUT_KINDS
    d.zp, d.lut_quotients = (None, 0x7f4000000000) if lut else (0x7f3000000000, None)
    return d


def _call(d, out_f=10, in_f=33, x=0x7f5000000000, dtype=None, M=1, y=0x7f6000000000):
    lib = _native.load()
    p = ctypes.addressof(d) if d is not None else None
    return lib.mctq_packed_linear(p, out_f, in_f, x, d.y_dtype if dtype is None and d is not None else (dtype or 0), M, None, y, None)


def test_c_abi_rejections():
    """Every argument check runs before any CUDA call (device pointers are never touched): no GPU needed."""
    assert _call(_lin_desc(), M=0) == 0                                                       # nothing to do
    assert _call(None) == -1
    assert _call(_lin_desc(kind=0)) == -1 and _call(_lin_desc(kind=5)) == -1                  # bad kind
    assert _call(_lin_desc(), x=None) == -1 and _call(_lin_desc(), y=None) == -1              # null pointers
    d = _lin_desc()
    d.codes = None
    assert _call(d) == -1
    d = _lin_desc()
    d.scale = None
    assert _call(d) == -1
    d = _lin_desc()
    d.zp = None
    assert _call(d) == -1                                                                     # affine needs zero points
    d = _lin_desc(kind=_native.PACK_LUT_I4)
    d.lut_quotients = None
    assert _call(d) == -4
    assert _call(_lin_desc(), in_f=34) == -1                                                  # n != out * in
    assert _call(_lin_desc(C=33, inner=1)) == -1                                              # per input channel
    assert _call(_lin_desc(C=5, inner=33)) == -1                                              # C not in {1, out}
    assert _call(_lin_desc(C=10, inner=1)) == -1                                              # C == out, but not rows
    assert _call(_lin_desc(), dtype=3) == -2                                                  # bad dtype
    assert _call(_lin_desc(dtype=_native.BF16), dtype=_native.F32) == -2                      # x is not the weight's dtype
    assert _call(_lin_desc(kind=_native.PACK_LUT_U8, dtype=_native.BF16)) == -2               # LUT weights are f32
    assert _call(_lin_desc(kind=_native.PACK_LUT_I4, K=17)) == -4                             # K out of range
    assert _call(_lin_desc(kind=_native.PACK_LUT_U8, K=257)) == -4
    assert _call(_lin_desc(kind=_native.PACK_LUT_U8, K=0)) == -4
    assert _call(_lin_desc(), M=-1) == -1
    assert _call(_lin_desc(out_f=0, in_f=33), out_f=0) == -1
    # several faults: null w -> kind -> dtype -> shape -> pointers -> parameters -> M == 0
    assert _call(_lin_desc(kind=5, dtype=3)) == -1
    assert _call(_lin_desc(dtype=3), in_f=34) == -2
    assert _call(_lin_desc(kind=_native.PACK_LUT_I4, dtype=_native.BF16, K=17)) == -2
    assert _call(_lin_desc(kind=_native.PACK_LUT_I4, K=17), in_f=34) == -1
    assert _call(_lin_desc(kind=_native.PACK_LUT_I4, K=17), M=-1) == -1
    assert _call(_lin_desc(kind=_native.PACK_LUT_I4, K=17), x=None) == -1
    assert _call(_lin_desc(kind=_native.PACK_LUT_I4, K=17), M=0) == -4
    d = _lin_desc()
    d.zp = None
    assert _call(d, M=0) == -1


# --------------------------------------------------------------------------------------------- GPU
def _exact_items(kind, dtype, out_f, in_f, per_channel, seed):
    """Codes and parameters whose products and partial sums are all exact: power-of-two scales / thresholds, small zero
    points, LUT values on the 8-bit grid.  Returns (codes, is_signed, scale, zp, quotients)."""
    g = torch.Generator().manual_seed(seed)
    n = out_f * in_f
    lut = kind in LUT_KINDS
    nb = n if kind in (_native.PACK_AFFINE_I8, _native.PACK_LUT_U8) else (n + 1) // 2
    C = out_f if per_channel else 1
    scale = 2.0 ** torch.randint(-2, 2, (C,), generator=g).float()
    if kind == _native.PACK_LUT_U8:
        K = 200
        codes = torch.randint(0, K, (nb,), generator=g).to(torch.uint8)
    else:
        K = 16
        codes = torch.randint(0, 256, (nb,), generator=g).to(torch.uint8)
    is_signed = not lut and seed % 2 == 0
    zp = None if lut else torch.randint(-2, 3, (C,), generator=g).int() + (0 if is_signed else 2)
    quot = ops.lut_quotients(torch.randint(-128, 128, (K,), generator=g).float(), 8, True) if lut else None
    return codes.cuda(), is_signed, scale.cuda(), (zp.cuda() if zp is not None else None), quot


def _rebuilt(codes, kind, is_signed, dtype, out_f, in_f, scale, zp, quot):
    """The weight as the host decoder of the wire format rebuilds it (test_packed_variants.decoded_f64): a reference that
    shares no decode code with the kernel under test."""
    C = scale.numel()
    host = lambda t: None if t is None else t.cpu().numpy()                     # noqa: E731
    w = decoded_f64(host(codes), kind, is_signed, dtype, C, in_f if C > 1 else 1, host(scale), host(zp), host(quot),
                    count=out_f * in_f)
    return torch.from_numpy(w.reshape(out_f, in_f)).to(dtype)


def _reference(x, w, bias):
    """f64 product of x and the rebuilt weight (numpy), and sum_k |x_k w_k| + |b|."""
    x64 = x.detach().double().cpu().numpy().reshape(-1, x.shape[-1])
    w64 = w.double().cpu().numpy()
    y = x64 @ w64.T
    mag = np.abs(x64) @ np.abs(w64).T
    if bias is not None:
        b = bias.double().cpu().numpy()
        y, mag = y + b, mag + np.abs(b)
    return y, mag


CROSS = {dt: FUSED_LINEAR_MAX_ROWS[dt] for dt in (torch.float32, torch.bfloat16, torch.float16)}
EXACT_SHAPES = [(1, 1, (1,)), (10, 33, (3,)), (4096, 4095, (2,)), (10, 4096, ("X",)), (1, 4095, (5,)), (4096, 64, (2, 3)),
                (10, 33, ("X",)), (10, 1, (4,)), (4096, 33, (1,)), (17, 1040, (9,)), (7, 16, (2, 5))]
KIND_DTYPES = [(k, dt) for k in (_native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4) for dt in (torch.float32, torch.bfloat16, torch.float16)] \
    + [(k, torch.float32) for k in LUT_KINDS]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", KIND_DTYPES)
@pytest.mark.parametrize("per_channel", [True, False])
@pytest.mark.parametrize("with_bias", [True, False])
def test_exact_on_representable_data(kind, dtype, per_channel, with_bias):
    """Every product and partial sum is exact in f32, so the fused output must equal the f64 product rounded once to the
    output dtype, whatever the reduction order: wrong channels, nibbles or tails cannot hide."""
    g = torch.Generator().manual_seed(kind)
    for seed, (out_f, in_f, lead) in enumerate(EXACT_SHAPES):
        lead = tuple(CROSS[dtype] if v == "X" else v for v in lead)
        codes, is_signed, scale, zp, quot = _exact_items(kind, dtype, out_f, in_f, per_channel, seed)
        x = (torch.randint(-2, 3, lead + (in_f,), generator=g).float() * 0.25).to("cuda", dtype)
        bias = (torch.randint(-8, 9, (out_f,), generator=g).float() * 0.25).to("cuda", dtype) if with_bias else None
        w = _rebuilt(codes, kind, is_signed, dtype, out_f, in_f, scale, zp, quot)
        y = torch.ops.mctq.packed_linear(x, codes, kind, is_signed, out_f, scale, zp, quot, bias)
        want, _ = _reference(x, w, bias)
        want = torch.from_numpy(want).to(dtype).reshape(lead + (out_f,))
        assert y.shape == want.shape and y.dtype == dtype and y.is_contiguous()
        assert torch.equal(y.cpu().view(torch.int16 if dtype != torch.float32 else torch.int32),
                           want.view(torch.int16 if dtype != torch.float32 else torch.int32)), (out_f, in_f, lead)
    # a transposed (non-contiguous) x and an empty one
    codes, is_signed, scale, zp, quot = _exact_items(kind, dtype, 10, 33, per_channel, 1)
    xt = (torch.randint(-2, 3, (33, 3), generator=g).float() * 0.25).to("cuda", dtype).t()
    y = torch.ops.mctq.packed_linear(xt, codes, kind, is_signed, 10, scale, zp, quot, None)
    w = _rebuilt(codes, kind, is_signed, dtype, 10, 33, scale, zp, quot)
    assert torch.equal(y.cpu(), torch.from_numpy(_reference(xt, w, None)[0]).to(dtype))
    assert torch.ops.mctq.packed_linear(xt[:0], codes, kind, is_signed, 10, scale, zp, quot, None).shape == (0, 10)


def _bound_ok(y, x, w, bias):
    want, mag = _reference(x, w, bias)
    K = x.shape[-1]
    got = y.double().cpu().numpy().reshape(want.shape)
    lim = (K + 3) * 2.0 ** -24 * mag * 1.01 + U_OUT[y.dtype] * np.abs(want)
    return bool(np.all(np.abs(got - want) <= lim)), float(np.max(np.abs(got - want) - lim))


def _wrapped_linear(out_f, in_f, qname, dtype, bias=True, seed=0):
    torch.manual_seed(seed)
    lin = torch.nn.Linear(in_f, out_f, bias=bias, device="cuda", dtype=dtype)
    w = lin.weight.detach()
    thr = [float(t) for t in w.float().abs().amax(1).clamp_min(1e-6)]
    if qname == "lut16":
        q = _lut_q(16, out_f)
    elif qname == "lut100":
        q = _lut_q(100, out_f)
    elif qname == "sym4":
        q = Q.WeightsSymmetricInferableQuantizer(4, thr, True, 0)
    elif qname == "uni8":
        q = Q.WeightsUniformInferableQuantizer(8, [-t for t in thr], [t * 0.6 for t in thr], True, 0)
    else:
        q = Q.WeightsSymmetricInferableQuantizer(8, [max(thr)], False)
    return mctq.PytorchQuantizationWrapper(lin, {"weight": q})


BOUND_FORMATS = [("lut16", torch.float32), ("lut100", torch.float32), ("sym4", torch.bfloat16), ("sym4", torch.float16),
                 ("uni8", torch.float32), ("uni8", torch.bfloat16), ("sym8t", torch.float16)]


@pytest.mark.gpu
@pytest.mark.parametrize("qname,dtype", BOUND_FORMATS)
def test_error_bound_on_random_data(qname, dtype):
    shapes = [(11008, 4096), (4096, 11008), (10, 33), (1, 4095)] if qname in ("lut16", "sym4") else [(10, 33), (4096, 4095)]
    for out_f, in_f in shapes:
        m = _wrapped_linear(out_f, in_f, qname, dtype if not qname.startswith("lut") else torch.float32)
        xdt = torch.float32 if qname.startswith("lut") else dtype
        report = m.pack_weights(fused_linear=True)
        assert report["weight"]["fused"], report
        w = m.get_quantized_weights()["weight"]
        bias = m.layer.bias.detach()
        for M in (1, 3, FUSED_LINEAR_MAX_ROWS[xdt]):
            x = torch.randn(M, in_f, device="cuda").to(xdt)
            with torch.no_grad():
                y = m(x)
                ok, worst = _bound_ok(y, x, w, bias)
                assert ok, (out_f, in_f, M, worst)
                if xdt == torch.float32:          # the f32 exact path meets the same bound (a check of the formula)
                    ok, worst = _bound_ok(torch.nn.functional.linear(x, w, bias), x, w, bias)
                    assert ok, ("exact path", worst)
        del m, w
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_deterministic_and_graph_replay():
    m = _wrapped_linear(4096, 11008, "lut16", torch.float32)
    m.pack_weights(fused_linear=True)
    x = torch.randn(2, 11008, device="cuda")
    with torch.no_grad():
        a, b = m(x), m(x)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            m(x)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            y = m(x)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(y.view(torch.int32), a.view(torch.int32))


def _exact_path(m, *args):
    """The wrapper's output on the exact packed path (fused mode switched off for the call)."""
    st = m._packed
    st.fused = False
    try:
        return m(*args)
    finally:
        st.fused = True


@pytest.mark.gpu
def test_fallbacks_equal_the_exact_path():
    m = _wrapped_linear(64, 96, "sym4", torch.bfloat16)
    m.pack_weights(fused_linear=True)
    calls = []
    before = _native.launch_count()
    x = torch.randn(3, 96, device="cuda", dtype=torch.bfloat16)
    with torch.no_grad():
        m(x)
    torch.cuda.synchronize()
    assert _native.launch_count() - before == 1                                   # fused: one launch, no unpack
    big = torch.randn(FUSED_LINEAR_MAX_ROWS[torch.bfloat16] + 1, 96, device="cuda", dtype=torch.bfloat16)
    with torch.no_grad():
        assert torch.equal(m(big), _exact_path(m, big))                           # above the crossover
        with pytest.raises(RuntimeError) as fused_err:
            m(x.float())                                                           # dtype mismatch: F.linear's error
        with pytest.raises(RuntimeError) as exact_err:
            _exact_path(m, x.float())
        assert str(fused_err.value) == str(exact_err.value)
    # autograd needed: exact path, with a graph
    xg = x.clone().requires_grad_(True)
    y = m(xg)
    assert y.grad_fn is not None and torch.equal(y.detach(), _exact_path(m, xg).detach())
    # a forward hook on the layer: exact path, and the hook runs
    h = m.layer.register_forward_hook(lambda mod, i, o: calls.append(1))
    with torch.no_grad():
        assert torch.equal(m(x), _exact_path(m, x)) and calls
    h.remove()
    # x on another device: the host-tensor path of F.linear raises like the exact path
    with torch.no_grad(), pytest.raises(RuntimeError):
        m(x.cpu())


@pytest.mark.gpu
def test_memory_of_a_fused_forward():
    torch.cuda.synchronize()
    torch.manual_seed(0)
    layers, in_f, out_f = [], 4096, 11008
    for _ in range(2):
        lin = torch.nn.Linear(in_f, out_f, bias=False, device="cuda")
        layers.append(mctq.PytorchQuantizationWrapper(lin, {"weight": _lut_q(16, out_f)}))
        in_f, out_f = out_f, in_f
    model = torch.nn.Sequential(*layers)
    x = torch.randn(1, 4096, device="cuda")
    with torch.no_grad():
        report = pack_model_weights(model, fused_linear=True)
        assert all(r["fused"] for rep in report.values() for r in rep.values())
        ops.clear_lut_caches()
        model(x)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        resident = torch.cuda.memory_allocated()
        model(x)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - resident
    activations = (4096 + 11008 + 4096) * 4
    assert peak <= activations + (1 << 20), peak


def _small(seed, fused=True):
    torch.manual_seed(seed)
    m = torch.nn.Sequential(torch.nn.Conv2d(3, 16, 3, bias=False), torch.nn.ReLU(), torch.nn.Flatten(),
                            torch.nn.Linear(16 * 6 * 6, 10), torch.nn.Linear(10, 10)).cuda()
    m[0] = mctq.PytorchQuantizationWrapper(m[0], {"weight": Q.WeightsSymmetricInferableQuantizer(8, [0.3] * 16, True, 0)})
    m[3] = mctq.PytorchQuantizationWrapper(m[3], {"weight": _lut_q(16, 10)})
    m[4] = mctq.PytorchQuantizationWrapper(m[4], {"weight": Q.WeightsSymmetricInferableQuantizer(8, [0.5] * 10, True, 0)})
    report = pack_model_weights(m, fused_linear=fused)
    return m, report


@pytest.mark.gpu
def test_reports_round_trips_and_model_plan(tmp_path):
    x = torch.randn(2, 3, 8, 8, device="cuda")
    a, report = _small(0)
    assert report["0"]["weight"]["fused"] is False and "Conv2d" in report["0"]["weight"]["fused_reason"]
    assert report["3"]["weight"]["fused"] and report["4"]["weight"]["fused"]
    assert "fused" not in _small(0, fused=False)[1]["3"]["weight"]                   # the default report is unchanged
    b, _ = _small(1)
    with torch.no_grad():
        want = a(x)
        b.load_state_dict(a.state_dict())
        assert b[3]._packed.fused and torch.equal(b(x), want)                       # state_dict
        path = os.path.join(tmp_path, "fused.pt")
        torch.save(a, path)
        c = mctq.pytorch_load_quantized_model(path)
        assert c[3]._packed.fused and torch.equal(c(x), want)                       # torch.save / load
        d = copy.deepcopy(c).cpu().cuda()
        assert d[3]._packed.fused and torch.equal(d(x), want)                       # .to()
        # switching an already packed model only switches the mode
        e, _ = _small(0, fused=False)
        assert not e[3]._packed.fused
        rep = pack_model_weights(e, fused_linear=True)
        assert e[3]._packed.fused and rep["3"]["weight"]["reason"] == "already packed"
        assert torch.equal(e(x), want)
        # ModelWeightPlan leaves the fused wrappers alone; the others stay bit-equal to today's path
        plain, _ = _small(0, fused=False)
        want_plain = plain(x)
        del want_plain
        with mctq.plan_model_weights(a) as plan:
            assert [w for w in plan.wrappers] == [a[0]]
            assert a[3].layer.weight is None and not a[3].__dict__.get("_prequantized", False)
            assert torch.equal(a(x), want)
            assert torch.equal(a[0](x), plain[0](x))
        q = mctq.quantize_model_weights(a)
        assert torch.equal(q["3"]["weight"], plain[3].get_quantized_weights()["weight"])


@pytest.mark.gpu
def test_opcheck():
    codes, is_signed, scale, zp, quot = _exact_items(_native.PACK_AFFINE_I4, torch.float32, 10, 33, True, 0)
    x = torch.randn(3, 33, device="cuda")
    torch.library.opcheck(torch.ops.mctq.packed_linear.default,
                          (x, codes, _native.PACK_AFFINE_I4, is_signed, 10, scale, zp, None, torch.randn(10, device="cuda")))
    # the host-tensor implementation goes through the device and matches
    y = torch.ops.mctq.packed_linear(x.cpu(), codes.cpu(), _native.PACK_AFFINE_I4, is_signed, 10, scale.cpu(), zp.cpu(), None, None)
    assert y.device.type == "cpu" and torch.equal(y, torch.ops.mctq.packed_linear(x, codes, _native.PACK_AFFINE_I4, is_signed, 10,
                                                                                 scale, zp, None, None).cpu())


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
def test_torchvision_in_situ(name):
    model = _tv_model(name)
    fused = copy.deepcopy(model)
    report = pack_model_weights(fused, fused_linear=True)
    linears = [k for k, rep in report.items() if rep["weight"]["fused"]]
    assert len(linears) == 1                                                          # the classifier
    clf = fused.get_submodule(linears[0])
    w = clf.get_quantized_weights()["weight"]
    with torch.no_grad():
        x1 = torch.randn(1, 3, 224, 224, device="cuda")
        want1 = model(x1)
        seen = {}
        h = clf.register_forward_pre_hook(lambda mod, args: seen.setdefault("x", args[0].clone()))
        got1 = fused(x1)
        h.remove()
        # a hook on the wrapper (not on the inner Linear) keeps the fused path: the launch descriptor exists only there
        assert clf._packed._lin is not None
        ok, worst = _bound_ok(got1, seen["x"], w, clf.layer.bias.detach())
        assert ok, worst
        assert torch.equal(got1.argmax(1), want1.argmax(1))
        clf._packed._lin = None
        x256 = torch.randn(256, 3, 224, 224, device="cuda")
        assert torch.equal(fused(x256), model(x256))                                  # above the crossover: bit-equal
        assert clf._packed._lin is None
