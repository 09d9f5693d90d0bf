"""Integer convolution mode: mctq_quantize_nhwc_i8 + mctq_packed_conv2d_i8 (csrc/mctq_packed_igemm.cu) and the packed-wrapper
mode built on them (pytorch/packed_weights.py).  Every GPU result is checked bit for bit against an exact integer reference
of the formula in include/mctq.h."""
import contextlib
import copy
import ctypes
import io
import pickle

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import mct_quantizers_b200 as mctq
from mct_quantizers_b200 import _native, ops
from mct_quantizers_b200.pytorch import packed_weights as PW
from mct_quantizers_b200.pytorch import quantizers as Q
from mct_quantizers_b200.pytorch.activation_quantization_holder import PytorchActivationQuantizationHolder
from mct_quantizers_b200.pytorch.packed_weights import PackedState, PackedWeight, integer_conv_eligibility

from test_packed_linear import _lin_desc

I8, I4, LU8 = _native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4, _native.PACK_LUT_U8
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
E_BADARG, E_DTYPE, E_RANGE = -1, -2, -3


# ------------------------------------------------------------------------------------------------ integer reference
def conv_reference(qx, zx, qw, zw, f, bias, stride, dilation, padding, out_dtype):
    """The formula of include/mctq.h: qx [N, Cin, H, W] codes, qw [Cout, Cin, kh, kw] codes, padding (pt, pb, pl, pr).
    The window is gathered with Tensor.unfold from Q(x)'s codes padded with zx; the sums run in float64, which is exact
    for these sizes (|sum| < 2^53), then c is converted to int64 and rounded once to f32."""
    (sh, sw), (dh, dw), (pt, pb, pl, pr) = stride, dilation, padding
    Cout, Cin, kh, kw = qw.shape
    p = F.pad(qx.to(torch.float64), (pl, pr, pt, pb), value=float(zx))
    X = p.unfold(2, dh * (kh - 1) + 1, sh).unfold(3, dw * (kw - 1) + 1, sw)[..., ::dh, ::dw]   # [N, Cin, Ho, Wo, kh, kw]
    W = qw.to(torch.float64)
    K = Cin * kh * kw
    zw = zw.reshape(-1).to(torch.float64).expand(Cout)
    acc = torch.einsum("nchwrs,ocrs->nohw", X, W)
    sx = X.sum(dim=(1, 4, 5))[:, None]
    sw_ = W.sum(dim=(1, 2, 3))[None, :, None, None]
    zw4 = zw[None, :, None, None]
    c = acc - zw4 * sx - zx * sw_ + K * zx * zw4
    y = c.to(torch.int64).to(torch.float32) * f.reshape(-1).to(torch.float32).expand(Cout)[None, :, None, None]
    if bias is not None:
        y = y + bias.to(torch.float32)[None, :, None, None]
    return y.to(out_dtype)


def test_reference_hand_worked():
    # one pixel of code 5, zx = 2, a 3x3 kernel of ones with padding 1: 8 padded taps hold zx = 2
    qx = torch.full((1, 1, 1, 1), 5)
    qw = torch.ones((1, 1, 3, 3), dtype=torch.int64)
    args = ((1, 1), (1, 1), (1, 1, 1, 1), torch.float32)
    # acc = 5 + 8 * 2 = 21, Sw = 9  ->  c = 21 - 2 * 9 = 3 = (5 - 2) * 1: the padded taps contribute 0
    y = conv_reference(qx, 2, qw, torch.zeros(1), torch.tensor([0.5]), torch.tensor([1.0]), *args)
    assert y.item() == 2.5
    # zw = 1: every (qw - zw) is 0, Sx = 21 counts the padded taps as zx  ->  c = 21 - 21 - 18 + 9 * 2 = 0
    y = conv_reference(qx, 2, qw, torch.ones(1), torch.tensor([0.5]), None, *args)
    assert y.item() == 0.0
    # c = 16777217 is not an f32: it rounds to 16777216 before the scaling
    y = conv_reference(torch.ones((1, 1, 1, 1)), 0, torch.ones((1, 1, 1, 1)), torch.tensor([-16777216]), torch.tensor([1.0]),
                       None, (1, 1), (1, 1), (0, 0, 0, 0), torch.float32)
    assert y.item() == 16777216.0
    # stride 2, dilation 2 on a 5 x 5 ramp: output (0, 0) reads rows / columns 0, 2, 4
    qx = torch.arange(25).reshape(1, 1, 5, 5)
    y = conv_reference(qx, 0, torch.ones((1, 1, 3, 3), dtype=torch.int64), torch.zeros(1), torch.ones(1), None, (2, 2),
                       (2, 2), (0, 0, 0, 0), torch.float32)
    assert y.shape == (1, 1, 1, 1) and y.item() == sum(5 * r + s for r in (0, 2, 4) for s in (0, 2, 4))


@pytest.mark.parametrize("padding,kernel,stride,dilation", [
    (0, 3, 1, 1), (1, 3, 2, 1), ((2, 1), (5, 3), (1, 2), 1), ("valid", 3, 2, 2), ("same", (4, 3), 1, (1, 2)),
    ("same", 2, 1, 1), (3, 7, 2, 1), ((0, 2), 1, (2, 1), 1)])
def test_geometry_matches_conv2d(padding, kernel, stride, dilation):
    layer = torch.nn.Conv2d(16, 4, kernel, stride=stride, padding=padding, dilation=dilation)
    pad = ops.conv_padding(layer)
    for H, W in ((9, 11), (16, 16), (13, 8)):
        ref = layer(torch.randn(2, 16, H, W)).shape
        assert ops.conv_output_hw(H, W, layer.kernel_size, layer.stride, layer.dilation, pad) == tuple(ref[2:])
        qx = torch.randint(-3, 4, (2, 16, H, W))
        y = conv_reference(qx, 0, torch.ones((4, 16) + layer.kernel_size, dtype=torch.int64), torch.zeros(1), torch.ones(1),
                           None, layer.stride, layer.dilation, pad, torch.float32)
        assert y.shape == ref


def test_reference_matches_float_conv():
    """With zx = zw = 0 and f = 1 the formula is the float convolution of the codes (exact in f64)."""
    g = torch.Generator().manual_seed(0)
    layer = torch.nn.Conv2d(16, 8, (3, 2), stride=(2, 1), padding=(1, 0), dilation=(1, 2), bias=False)
    qx = torch.randint(-20, 20, (2, 16, 7, 9), generator=g)
    qw = torch.randint(-5, 5, (8, 16, 3, 2), generator=g)
    ref = F.conv2d(qx.double(), qw.double(), stride=layer.stride, padding=layer.padding, dilation=layer.dilation)
    y = conv_reference(qx, 0, qw, torch.zeros(1), torch.ones(1), None, layer.stride, layer.dilation,
                       ops.conv_padding(layer), torch.float64)
    assert torch.equal(y, ref.float().double())


@pytest.mark.parametrize("kind", [I8, I4])
@pytest.mark.parametrize("signed", [True, False])
def test_code_reorder(kind, signed):
    g = torch.Generator().manual_seed(kind * 2 + signed)
    lo, hi = ((-8, 7) if signed else (0, 15)) if kind == I4 else ((-128, 127) if signed else (0, 255))
    qw = torch.randint(lo, hi + 1, (6, 32, 3, 3), generator=g, dtype=torch.int32)
    codes = ops.pack_weight_codes(qw, kind, signed)
    assert torch.equal(ops.weight_code_values(codes, kind, signed, 6, 288), qw.reshape(6, 288))
    rsc = ops.conv_codes_rsc(codes, kind, signed, 6, 32, 3, 3)
    assert rsc.numel() == codes.numel()
    assert torch.equal(ops.weight_code_values(rsc, kind, signed, 6, 288), qw.permute(0, 2, 3, 1).reshape(6, 288))


def test_window_sums_on_the_host():
    g = torch.Generator().manual_seed(1)
    P = torch.randint(-100, 100, (2 * 6 * 7,), generator=g, dtype=torch.int32)
    sx = ops.conv_window_sums(P, 2, 6, 7, 16, (3, 3), (2, 1), (1, 2), (1, 0, 2, 1), 3)
    # the window of each output pixel gathered as in conv_reference, padded taps counting Cin * zx = 48
    p = F.pad(P.reshape(2, 6, 7).to(torch.int64), (2, 1, 1, 0), value=48)
    ref = p.unfold(1, 3, 2).unfold(2, 5, 1)[..., ::1, ::2].sum(dim=(3, 4))
    assert sx.shape == (2 * 3 * 6,) and torch.equal(sx.to(torch.int64), ref.reshape(-1))


# ------------------------------------------------------------------------------------------------ C-ABI rejections
def _geom(**k):
    g = dict(N=2, H=8, W=8, Cin=16, Ho=8, Wo=8, kh=3, kw=3, sh=1, sw=1, dh=1, dw=1, pt=1, pb=1, pl=1, pr=1)
    g.update(k)
    return _native.MctqConv2dGeom(*(g[f] for f, _ in _native.MctqConv2dGeom._fields_))


def _conv_call(d, g=None, Cout=10, xq=0x7f5000000000, x_signed=1, zx=0, w_rowsum=0x7f6100000000, factor=0x7f6200000000,
               y_dtype=_native.F32, y=0x7f6000000000, nchw=1):
    lib = _native.load()
    g = g if g is not None else _geom()
    return lib.mctq_packed_conv2d_i8(ctypes.byref(d) if d is not None else None, ctypes.byref(g) if g is not False else None,
                                     Cout, xq, x_signed, zx, None, w_rowsum, factor, None, y_dtype, y, nchw, None)


def test_c_abi_rejections():
    K = 16 * 9
    ok = lambda **k: _lin_desc(out_f=10, in_f=K, **k)                             # noqa: E731
    assert _conv_call(None) == E_BADARG
    assert _conv_call(ok(), g=False) == E_BADARG
    assert _conv_call(_lin_desc(out_f=10, in_f=K, kind=LU8)) == E_BADARG                # LUT kinds
    assert _conv_call(ok(dtype=_native.BF16)) == E_DTYPE                             # y dtype != rebuilt dtype
    assert _conv_call(ok(), y_dtype=7) == E_DTYPE
    for field in ("H", "W", "Cin", "Ho", "Wo", "kh", "kw", "sh", "sw", "dh", "dw"):
        assert _conv_call(ok(), g=_geom(**{field: 0})) == E_BADARG, field               # non-positive geometry
    assert _conv_call(ok(), g=_geom(N=-1)) == E_BADARG
    assert _conv_call(ok(), g=_geom(pt=-1)) == E_BADARG and _conv_call(ok(), g=_geom(pr=-1)) == E_BADARG
    assert _conv_call(ok(), nchw=2) == E_BADARG
    assert _conv_call(_lin_desc(out_f=10, in_f=8 * 9), g=_geom(Cin=8)) == E_BADARG   # Cin % 16
    assert _conv_call(_lin_desc(out_f=10, in_f=16, kind=I4), g=_geom(kh=1, kw=1)) == E_BADARG   # int4: K % 32
    assert _conv_call(ok(), Cout=11) == E_BADARG                                     # descriptor of another shape
    assert _conv_call(ok(), xq=0x7f5000000008) == E_BADARG                           # misaligned x codes
    d = ok()
    d.codes = 0x7f0000000004
    assert _conv_call(d) == E_BADARG                                                 # misaligned weight codes
    assert _conv_call(ok(), xq=None) == E_BADARG
    assert _conv_call(ok(), y=None) == E_BADARG
    assert _conv_call(ok(), factor=None) == E_BADARG
    assert _conv_call(ok(), zx=3, w_rowsum=None) == E_BADARG                         # zx != 0 needs Sw
    assert _conv_call(ok(), g=_geom(N=2 ** 30, Ho=2, Wo=1)) == E_BADARG               # M = N * Ho * Wo >= 2^31
    assert _conv_call(ok(), x_signed=1, zx=128) == E_RANGE                           # zx outside the x codes' range
    assert _conv_call(ok(), x_signed=0, zx=-1) == E_RANGE
    # K = Cin * kh * kw over the int32 bound of the (weight, x) signedness pair; at the bound: accepted (M = 0: no-op)
    for ws, xs, k in ((1, 1, 131071), (0, 1, 65793), (1, 0, 65793), (0, 0, 33025)):
        cin = k // 16 * 16
        d = _lin_desc(out_f=2, in_f=cin + 16)
        d.is_signed = ws
        assert _conv_call(d, g=_geom(Cin=cin + 16, kh=1, kw=1), Cout=2, x_signed=xs) == E_RANGE
        d = _lin_desc(out_f=2, in_f=cin)
        d.is_signed = ws
        assert _conv_call(d, g=_geom(Cin=cin, kh=1, kw=1, N=0), Cout=2, x_signed=xs) == 0
    assert _conv_call(ok(), g=_geom(N=0)) == 0
    lib = _native.load()
    q = lambda **k: lib.mctq_quantize_nhwc_i8(k.get("x", 0x7f5000000000), k.get("dt", _native.F32), k.get("N", 1),   # noqa: E731
                                               k.get("C", 16), k.get("H", 4), k.get("W", 4), 1.0, 0, k.get("qmin", -128),
                                               k.get("qmax", 127), k.get("codes", 0x7f6000000000), None, None)
    assert q(x=None) == E_BADARG and q(codes=None) == E_BADARG and q(N=-1) == E_BADARG
    assert q(C=0) == E_BADARG and q(H=0) == E_BADARG and q(W=0) == E_BADARG
    assert q(dt=5) == E_DTYPE
    assert q(qmin=1, qmax=0) == E_RANGE and q(qmin=-129) == E_RANGE and q(qmin=0, qmax=256) == E_RANGE
    assert q(N=0) == 0


# ------------------------------------------------------------------------------------------------ eligibility and reports
def _act(kind="sym", bits=8, signed=True):
    if kind == "sym":
        return Q.ActivationSymmetricInferableQuantizer(bits, [4.0], signed)
    if kind == "uniform":
        return Q.ActivationUniformInferableQuantizer(bits, [-1.5], [3.0])
    return Q.ActivationLutPOTInferableQuantizer(bits, [-2.0, 0.0, 1.0, 3.0], [4.0], signed)


def _conv_wrapper(cin=32, cout=8, k=3, **kw):
    w = Q.WeightsSymmetricInferableQuantizer(8, [1.0] * cout, True, 0)
    return mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(cin, cout, k, **kw), {"weight": w})


def _fake_packed_conv(wrapper, kind=I8, channels_last=False, C=None):
    """A PackedState built on the host (no codes buffer): what pack_weights leaves behind, for the eligibility rules."""
    shape = tuple(wrapper.layer.weight.shape)
    t = torch.empty(shape, device="meta")
    stride = (t.to(memory_format=torch.channels_last) if channels_last else t).stride()
    K = shape[1] * shape[2] * shape[3]
    e = PackedWeight(wrapper, "weight", wrapper.weights_quantizers["weight"], kind, True, torch.float32, shape, stride,
                     shape[0] if C is None else C, K if C is None else 1)
    wrapper._packed = PackedState([e])
    return wrapper


def test_eligibility():
    q = _act()
    assert integer_conv_eligibility(_fake_packed_conv(_conv_wrapper()), q) == (True, "")
    assert integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(), channels_last=True), q) == (True, "")
    assert integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(), C=1), q) == (True, "")
    assert integer_conv_eligibility(_conv_wrapper(), q) == (False, "the weight is not packed")
    lin = mctq.PytorchQuantizationWrapper(torch.nn.Linear(32, 8), {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 8, True, 0)})
    assert integer_conv_eligibility(lin, q) == (False, "the layer is Linear, not torch.nn.Conv2d")
    ok, why = integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(groups=2)), q)
    assert not ok and "groups = 2" in why
    ok, why = integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(cin=32, cout=32, groups=32)), q)
    assert not ok and "depthwise" in why
    ok, why = integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(padding=1, padding_mode="reflect")), q)
    assert not ok and "padding_mode" in why
    lut = _fake_packed_conv(_conv_wrapper(), kind=LU8)
    ok, why = integer_conv_eligibility(lut, q)
    assert not ok and "lut_u8" in why
    ok, why = integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(cin=24)), q)
    assert not ok and "in_channels = 24 is not a multiple of 16" in why
    ok, why = integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(cin=16, k=1), kind=I4), q)
    assert not ok and "multiple of 32" in why
    assert integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(cin=16, k=2), kind=I4), q)[0]
    ok, why = integer_conv_eligibility(_fake_packed_conv(_conv_wrapper()), _act("lut"))
    assert not ok and "per-tensor affine" in why
    ok, why = integer_conv_eligibility(_fake_packed_conv(_conv_wrapper()), _act(bits=16))
    assert not ok and "8-bit codes" in why
    # a rebuilt weight of another layout, parameters along another axis
    w = _fake_packed_conv(_conv_wrapper())
    w._packed.entries[0].stride_out = (1, 72, 24, 8)
    ok, why = integer_conv_eligibility(w, q)
    assert not ok and "contiguous or channels_last" in why
    w = _fake_packed_conv(_conv_wrapper())
    w._packed.entries[0].C, w._packed.entries[0].inner = 32, 9
    ok, why = integer_conv_eligibility(w, q)
    assert not ok and "channel_axis 0" in why
    # K over the bound: u8 x u8
    big = _fake_packed_conv(_conv_wrapper(cin=3680, cout=1, k=3))
    big._packed.entries[0].is_signed = False
    ok, why = integer_conv_eligibility(big, _act(signed=False))
    assert not ok and "33025" in why


def test_shared_input_quantizer_reasons_are_unchanged():
    """integer_linear_eligibility's input-quantizer reasons, word for word."""
    from test_integer_linear import _wrapper
    from test_packed_linear import _fake_packed
    cases = {"lut": "the input quantizer ActivationLutPOTInferableQuantizer is not a per-tensor affine activation quantizer "
                    "(ActivationSymmetric / POT / Uniform)",
             16: "the input quantization range [-32768, 32767] does not fit 8-bit codes"}
    assert PW.integer_linear_eligibility(_fake_packed(_wrapper()), _act("lut")) == (False, cases["lut"])
    assert PW.integer_linear_eligibility(_fake_packed(_wrapper()), _act(bits=16)) == (False, cases[16])
    assert integer_conv_eligibility(_fake_packed_conv(_conv_wrapper()), _act("lut")) == (False, cases["lut"])
    reuse = _act()
    reuse.enable_reuse = True
    assert PW.integer_linear_eligibility(_fake_packed(_wrapper()), reuse) == \
        (False, "the input quantizer reuses its outputs (enable_reuse)")
    assert integer_conv_eligibility(_fake_packed_conv(_conv_wrapper()), reuse) == \
        (False, "the input quantizer reuses its outputs (enable_reuse)")


class _Net(torch.nn.Module):
    def __init__(self, holders, wrappers, body):
        super().__init__()
        self.h = torch.nn.ModuleList(holders)
        self.w = torch.nn.ModuleList(wrappers)
        self.body = body

    def forward(self, x):
        return self.body(self, x)


def _lin_wrapper():
    return mctq.PytorchQuantizationWrapper(torch.nn.Linear(32, 8), {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 8, True, 0)})


def _fake_lin():
    from test_packed_linear import _fake_packed
    return _fake_packed(_lin_wrapper())


def test_model_reports_without_a_gpu():
    H = lambda: PytorchActivationQuantizationHolder(_act())                      # noqa: E731
    body = lambda m, x: m.w[2](m.h[1](m.w[1](torch.relu(m.w[0](m.h[0](x)))).mean((2, 3))))   # noqa: E731
    mk = lambda: _Net([H(), H()], [_fake_packed_conv(_conv_wrapper()), _fake_packed_conv(_conv_wrapper(cin=8)), _fake_lin()],  # noqa: E731
                      body)
    net = mk()
    reports = PW.pack_model_weights(net, integer_conv=True)
    on, relu_in, lin = (reports[f"w.{i}"]["weight"] for i in range(3))
    assert (on["integer_conv"], on["integer_conv_reason"], on["input_holder"]) == (True, "", "h.0")
    assert "integer" not in on
    assert relu_in["integer_conv"] is False and "not the output of an activation quantization holder" in relu_in["integer_conv_reason"]
    assert lin["integer_conv"] is False and lin["integer_conv_reason"] == "the layer is Linear, not torch.nn.Conv2d"
    assert net.w[0]._packed.integer and net.w[0]._packed.input_quantizer is net.h[0].activation_holder_quantizer
    assert not net.w[1]._packed.integer and not net.w[2]._packed.integer
    # integer_linear=True alone: exactly today's report for the conv wrappers, and the Linear switches
    net = mk()
    reports = PW.pack_model_weights(net, integer_linear=True)
    r = reports["w.0"]["weight"]
    assert (r["integer"], r["integer_reason"], r["input_holder"]) == (False, "the layer is Conv2d, not torch.nn.Linear", "h.0")
    assert "integer_conv" not in r and not net.w[0]._packed.integer
    assert reports["w.2"]["weight"]["integer"] and net.w[2]._packed.integer
    # both flags: both sets of keys, each wrapper switched by its own mode
    net = mk()
    reports = PW.pack_model_weights(net, integer_linear=True, integer_conv=True)
    r0, r2 = reports["w.0"]["weight"], reports["w.2"]["weight"]
    assert r0["integer"] is False and r0["integer_conv"] is True and r0["input_holder"] == "h.0"
    assert r2["integer"] is True and r2["integer_conv"] is False and r2["input_holder"] == "h.1"
    assert net.w[0]._packed.integer and net.w[2]._packed.integer and not net.w[1]._packed.integer
    # an untraceable model
    def untraceable(m, x):
        if x.sum() > 0:
            return m.w[0](m.h[0](x))
        return x
    net = _Net([H()], [_fake_packed_conv(_conv_wrapper())], untraceable)
    r = PW.pack_model_weights(net, integer_conv=True)["w.0"]["weight"]
    assert r["integer_conv"] is False and "cannot be traced" in r["integer_conv_reason"] and r["input_holder"] is None
    with pytest.raises(ValueError, match="input_quantizer"):
        PW.pack_wrapper_weights(_conv_wrapper(), integer_conv=True)


def _torchvision_models():
    tv = pytest.importorskip("torchvision")
    import sys
    import os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    try:
        from model_forward_bench import quantize_model
    finally:
        sys.path.pop(0)
    return {"resnet18": lambda: quantize_model(tv.models.resnet18(), mctq, Q),
            "mobilenet_v2": lambda: quantize_model(tv.models.mobilenet_v2(), mctq, Q)}


def _fake_pack_model(model):
    from mct_quantizers_b200.pytorch.quantize_wrapper import PytorchQuantizationWrapper
    from test_packed_linear import _fake_packed
    for m in model.modules():
        if isinstance(m, PytorchQuantizationWrapper):
            _fake_packed_conv(m) if isinstance(m.layer, torch.nn.Conv2d) else _fake_packed(m)
    return model


@pytest.mark.parametrize("name", ["resnet18", "mobilenet_v2"])
def test_benchmark_model_reports(name):
    model = _fake_pack_model(_torchvision_models()[name]())
    reports = PW.pack_model_weights(model, integer_conv=True)
    switched = {n for n, r in reports.items() if r["weight"]["integer_conv"]}
    reasons = {n: r["weight"]["integer_conv_reason"] for n, r in reports.items() if not r["weight"]["integer_conv"]}
    if name == "resnet18":
        # every block conv and downsample conv reads a ReLU holder, except the stem and layer1.0.conv1 (after max-pool)
        assert len(switched) == 18 and "layer2.0.downsample.0" in switched and "layer1.0.conv2" in switched
        for n in ("conv1", "layer1.0.conv1", "fc"):
            assert "not the output of an activation quantization holder" in reasons[n]
    else:
        assert "groups = 32" in reasons["features.1.conv.0.0"]                  # depthwise
        assert "not the output of an activation quantization holder" in reasons["features.2.conv.0.0"]
        # the projection convs read the depthwise conv's ReLU6 holder; the expansion convs read the previous block's output
        assert switched == {"features.1.conv.1"} | {f"features.{i}.conv.2" for i in range(2, 18)}
    assert all(model.get_submodule(n)._packed.integer for n in switched)


# ------------------------------------------------------------------------------------------------ GPU: NHWC quantizer
def _launch_args(q):
    from mct_quantizers_b200.pytorch.fused_activation_holder import affine_scalar_params
    s, z, _, _ = affine_scalar_params(q)
    return q._validated_launch_args(s, z)[1]


def _scalar_codes(x, scale, zp, qmin, qmax):
    """Codes of mctq_fq_affine_scalar with code_mode INT8, in x's logical NCHW order."""
    lib = _native.load()
    xd = x.contiguous()
    y = torch.empty_like(xd)
    codes = torch.empty(xd.shape, dtype=torch.int8 if qmin < 0 else torch.uint8, device=x.device)
    tag = {torch.float32: _native.F32, torch.bfloat16: _native.BF16, torch.float16: _native.F16}[x.dtype]
    rc = lib.mctq_fq_affine_scalar(xd.data_ptr(), y.data_ptr(), codes.data_ptr(), xd.numel(), tag, float(np.float32(scale)),
                                   zp, qmin, qmax, _native.CODES_INT8, torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "mctq_fq_affine_scalar")
    return codes


def _special_x(shape, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g) * 3
    flat = x.view(-1)
    flat[::97] = float("nan")
    flat[5::89] = float("inf")
    flat[7::83] = -float("inf")
    flat[11::79] = 1e6
    return x.to(dtype).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", [(1, 16, 1, 1), (3, 5, 7, 9), (2, 64, 56, 56), (1, 200, 3, 33), (5, 17, 13, 1)])
@pytest.mark.parametrize("qname", ["s8", "u8", "uniform"])
def test_nhwc_codes_and_sums(dtype, shape, qname):
    q = {"s8": _act(), "u8": _act(signed=False), "uniform": Q.ActivationUniformInferableQuantizer(8, [-1.3], [2.9])}[qname]
    s, z, qmin, qmax = _launch_args(q)
    x = _special_x(shape, dtype, sum(shape))
    ref = _scalar_codes(x, s, z, qmin, qmax).permute(0, 2, 3, 1)
    for xin in (x, x.to(memory_format=torch.channels_last), x[..., :].transpose(2, 3).contiguous().transpose(2, 3)):
        codes, P = ops.quantize_nhwc_i8(xin, s, z, qmin, qmax, True)
        assert codes.shape == ref.shape and codes.is_contiguous() and torch.equal(codes, ref)
        assert torch.equal(P.cpu().to(torch.int64), ref.cpu().to(torch.int64).sum(-1).reshape(-1))
    c2, p2 = torch.ops.mctq.quantize_nhwc_i8(x, s, z, qmin, qmax, False)
    assert torch.equal(c2, ref) and p2.numel() == 0


# ------------------------------------------------------------------------------------------------ GPU: the GEMM
def _conv_case(N, Cin, H, W, Cout, k, stride, dilation, padding, kind, w_signed, per_channel, zw_nonzero, x_signed, zx,
               dtype, with_bias, channels_last, seed):
    """One packed_conv2d_i8 call against the reference; the output sits inside a NaN-filled buffer that must stay NaN."""
    g = torch.Generator().manual_seed(seed)
    kh, kw = k
    lo, hi = ((-8, 7) if w_signed else (0, 15)) if kind == I4 else ((-128, 127) if w_signed else (0, 255))
    qw = torch.randint(lo, hi + 1, (Cout, Cin, kh, kw), generator=g, dtype=torch.int32)
    C = Cout if per_channel else 1
    zw = torch.randint(lo, hi + 1, (C,), generator=g, dtype=torch.int32) if zw_nonzero else torch.zeros(C, dtype=torch.int32)
    scale = (torch.rand(C, generator=g) * 0.02 + 0.001).to(torch.float32)
    xlo, xhi = (-128, 127) if x_signed else (0, 255)
    qx = torch.randint(xlo, xhi + 1, (N, Cin, H, W), generator=g, dtype=torch.int32)
    x_scale = 0.0371
    f = (torch.tensor(np.float32(x_scale)) * scale).to(torch.float32)
    bias = (torch.randn(Cout, generator=g) * 3).to(dtype).cuda() if with_bias else None
    codes = ops.pack_weight_codes(qw.permute(0, 2, 3, 1).contiguous(), kind, w_signed).cuda()
    conv = ops.IntegerConv2d.from_parts(codes, kind, w_signed, dtype, Cout, Cin, k, stride, dilation, padding, f.cuda(),
                                        zw.cuda(), None, zx)
    xq = qx.permute(0, 2, 3, 1).contiguous().to(torch.int8 if x_signed else torch.uint8).cuda()
    P = qx.sum(1).to(torch.int32).reshape(-1).cuda()
    sx = ops.conv_window_sums(P, N, H, W, Cin, k, stride, dilation, padding, zx)
    Ho, Wo = conv.output_hw(H, W)
    ref = conv_reference(qx.cuda(), zx, qw.cuda(), zw.cuda(), f.cuda(), bias, stride, dilation, padding, dtype)
    assert ref.shape == (N, Cout, Ho, Wo)
    y = conv.gemm(xq, sx, bias, channels_last=channels_last)
    assert y.shape == ref.shape
    assert y.is_contiguous(memory_format=torch.channels_last if channels_last else torch.contiguous_format)
    bits = lambda t: t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)    # noqa: E731
    assert torch.equal(bits(y), bits(ref)), f"{(y.float() - ref.float()).abs().max()}"
    # canary: write into the middle of a NaN buffer through the same kernel
    M = N * Ho * Wo
    canary = torch.full((M * Cout + 64,), float("nan"), dtype=dtype, device="cuda")
    g_ = _native.MctqConv2dGeom(N, H, W, Cin, Ho, Wo, kh, kw, *stride, *dilation, *padding)
    lib = _native.load()
    out = canary[32:32 + M * Cout]
    rc = lib.mctq_packed_conv2d_i8(conv._w._desc_ptr, ctypes.addressof(g_), Cout, xq.data_ptr(), int(x_signed), zx,
                                   sx.data_ptr() if conv.needs_x_rowsum else None, conv.w_rowsum.data_ptr(),
                                   conv.factor.data_ptr(), bias.data_ptr() if bias is not None else None,
                                   {torch.float32: _native.F32, torch.bfloat16: _native.BF16, torch.float16: _native.F16}[dtype],
                                   out.data_ptr(), 0 if channels_last else 1, torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "mctq_packed_conv2d_i8")
    assert torch.isnan(canary[:32]).all() and torch.isnan(canary[32 + M * Cout:]).all()
    assert torch.equal(bits(out), bits(y.permute(0, 2, 3, 1) if channels_last else y).reshape(-1))
    return conv


# (N, Cin, H, W, Cout, kernel, stride, dilation, padding (pt, pb, pl, pr))
_SHAPES = [
    (1, 16, 5, 5, 8, (1, 1), (1, 1), (1, 1), (0, 0, 0, 0)),
    (2, 32, 9, 7, 130, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1)),
    (3, 16, 11, 13, 64, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1)),
    (1, 48, 12, 10, 40, (5, 5), (1, 2), (2, 1), (4, 3, 2, 1)),                  # asymmetric, dilated
    (2, 16, 15, 15, 96, (7, 7), (2, 2), (1, 1), (3, 3, 3, 3)),
    (1, 32, 10, 9, 33, (3, 2), (1, 1), (2, 2), (2, 0, 0, 2)),
    (5, 64, 14, 14, 128, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1)),                   # M = 980: several row tiles
    (1, 256, 7, 7, 512, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1)),
    (64, 64, 8, 8, 64, (1, 1), (2, 2), (1, 1), (0, 0, 0, 0)),                     # strided 1x1 (downsample)
]
_CONFIGS = [(kind, ws, xs, zx) for kind in (I8, I4) for ws in (True, False) for xs, zx in ((True, 0), (True, -7), (False, 0),
                                                                                            (False, 128))]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ci", range(len(_CONFIGS)))
def test_conv_bit_exact(ci, dtype):
    kind, ws, xs, zx = _CONFIGS[ci]
    for si in range(ci % 3, len(_SHAPES), 3):
        N, Cin, H, W, Cout, k, st, dil, pad = _SHAPES[si]
        if kind == I4 and (Cin * k[0] * k[1]) % 32:
            Cin = 32
        _conv_case(N, Cin, H, W, Cout, k, st, dil, pad, kind, ws, per_channel=(si + ci) % 2 == 0,
                   zw_nonzero=(si + ci) % 3 != 0, x_signed=xs, zx=zx, dtype=dtype, with_bias=si % 2 == 1,
                   channels_last=(si + ci) % 4 < 2, seed=1000 * ci + si)


@pytest.mark.gpu
def test_split_k_of_1_and_8_and_large_m():
    # Cout = 128, M = 16, K = 256 * 9 runs as clusters of 8 CTAs; M = 64 * 56 * 56 as many single-CTA row tiles
    _conv_case(1, 256, 4, 4, 128, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), I8, True, True, True, True, 3, torch.float32, True,
               False, 11)
    _conv_case(64, 64, 56, 56, 64, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), I8, True, True, True, False, 5, torch.bfloat16, True,
               True, 12)
    _conv_case(8, 32, 33, 31, 200, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1), I4, False, False, True, False, 200, torch.float16,
               False, False, 13)


@pytest.mark.gpu
def test_torch_ops_match_integer_conv():
    g = torch.Generator().manual_seed(3)
    layer = torch.nn.Conv2d(32, 24, 3, padding=1)
    qw = torch.randint(-8, 8, (24, 32, 3, 3), generator=g, dtype=torch.int32)
    codes = ops.pack_weight_codes(qw, I4, True).cuda()
    zw = torch.randint(-8, 8, (24,), generator=g, dtype=torch.int32).cuda()
    scale = (torch.rand(24, generator=g) * 0.01 + 0.001).cuda()
    conv = ops.IntegerConv2d(codes, I4, True, torch.bfloat16, 24, 32, (3, 3), (288, 9, 3, 1), (1, 1), (1, 1),
                             ops.conv_padding(layer), scale, zw, 0.05, 2, -128, 127)
    x = torch.randn(2, 32, 6, 6, device="cuda").to(torch.bfloat16)
    qx, P = torch.ops.mctq.quantize_nhwc_i8(x, 0.05, 2, -128, 127, True)
    sx = ops.conv_window_sums(P, 2, 6, 6, 32, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), 2)
    rsc = ops.conv_codes_rsc(codes, I4, True, 24, 32, 3, 3)
    args = (2, sx, rsc, I4, True, 24, [3, 3], [1, 1], [1, 1], [1, 1, 1, 1], zw, conv.w_rowsum, conv.factor, None,
            torch.bfloat16, False)
    y = torch.ops.mctq.packed_conv2d_i8(qx, *args)
    assert torch.equal(y.view(torch.int16), conv(x).view(torch.int16))
    y_cpu = torch.ops.mctq.packed_conv2d_i8(qx.cpu(), *[a.cpu() if isinstance(a, torch.Tensor) else a for a in args])
    assert torch.equal(y_cpu.view(torch.int16), y.cpu().view(torch.int16))
    with pytest.raises(RuntimeError, match="window code sums"):
        torch.ops.mctq.packed_conv2d_i8(qx, 2, None, *args[2:])
    with pytest.raises(ValueError, match="zero points"):
        torch.ops.mctq.packed_conv2d_i8(qx, 2, sx, rsc, I4, True, 24, [3, 3], [1, 1], [1, 1], [1, 1, 1, 1], zw[:1],
                                        conv.w_rowsum, conv.factor, None, torch.bfloat16, False)


# ------------------------------------------------------------------------------------------------ GPU: module level
@contextlib.contextmanager
def _no_tf32():
    """The packed path's F.conv2d in full f32: with TF32 (cuDNN's default) it is further from the exact sum than the
    tolerance of the comparison."""
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32 = prev


class _ConvModel(torch.nn.Module):
    """holder -> Conv 4x3 (asymmetric 'same') -> holder -> Conv 1x1 stride 2."""

    def __init__(self, dtype, wq_kind, weight_cl=False):
        super().__init__()
        wq = (lambda C: Q.WeightsSymmetricInferableQuantizer(4, [0.5] * C, True, 0)) if wq_kind == "i4" else \
            (lambda C: Q.WeightsUniformInferableQuantizer(8, [-0.3] * C, [0.2] * C, True, 0))
        self.h0 = PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [-1.7], [2.3]))
        self.c0 = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(32, 64, (4, 3), padding="same"), {"weight": wq(64)})
        self.h1 = PytorchActivationQuantizationHolder(Q.ActivationSymmetricInferableQuantizer(8, [6.0], True))
        self.c1 = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(64, 48, 1, stride=2, bias=False), {"weight": wq(48)})
        self.to(dtype).cuda()
        if weight_cl:
            self.c0.layer.weight.data = self.c0.layer.weight.data.to(memory_format=torch.channels_last)

    def forward(self, x):
        return self.c1(self.h1(self.c0(self.h0(x))))


def _layer_reference(h, c, x):
    """The integer formula of one switched conv, with Q's codes of its input."""
    st = c._packed
    e = st.entries[0]
    s, z, qmin, qmax = _launch_args(h.activation_holder_quantizer)
    layer = c.layer
    qx, _ = ops.quantize_nhwc_i8(x, s, z, qmin, qmax, False)
    it = e.plan_item()
    shape = tuple(e.shape_out)
    qw = ops.weight_code_values(e.codes, e.kind, e.is_signed, shape[0], shape[1] * shape[2] * shape[3])
    if e.stride_out != torch.empty(shape, device="meta").stride():
        qw = qw.reshape(shape[0], shape[2], shape[3], shape[1]).permute(0, 3, 1, 2)
    f = torch.tensor(np.float32(s)).cuda() * it[8]
    return conv_reference(qx.permute(0, 3, 1, 2).to(torch.int64), z, qw.reshape(shape).to(torch.int64), it[9], f,
                          layer.bias, layer.stride, layer.dilation, ops.conv_padding(layer), x.dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("wq_kind", ["i8", "i4"])
@pytest.mark.parametrize("layout", ["nchw", "x_cl", "w_cl"])
def test_model_switch(dtype, wq_kind, layout):
    torch.manual_seed(0)
    model = _ConvModel(dtype, wq_kind, weight_cl=layout == "w_cl")
    x = (torch.randn(3, 32, 11, 10, device="cuda") * 1.5).to(dtype)
    if layout == "x_cl":
        x = x.to(memory_format=torch.channels_last)
    with torch.no_grad(), _no_tf32():
        y_packed = copy.deepcopy(model)
        PW.pack_model_weights(y_packed)
        y_float = y_packed(x)
        ref_strides = [model.c0(model.h0(x)).stride()]
        ref_strides.append(model.c1(model.h1(model.c0(model.h0(x)))).stride())
        report = PW.pack_model_weights(model, integer_conv=True)
        for name, holder in (("c0", "h0"), ("c1", "h1")):
            r = report[name]["weight"]
            assert r["packed"] and r["integer_conv"] and r["integer_conv_reason"] == "" and r["input_holder"] == holder
        a = model.c0(model.h0(x))
        assert torch.equal(a.float(), _layer_reference(model.h0, model.c0, model.h0(x)).float())
        assert a.stride() == ref_strides[0]
        b = model.h1(a)
        y = model.c1(b)
        assert torch.equal(y.float(), _layer_reference(model.h1, model.c1, b).float())
        assert y.stride() == ref_strides[1]
        assert torch.equal(model(x).float(), y.float())
        tol = 2e-2 if dtype != torch.float32 else 1e-4
        assert torch.allclose(y.float(), y_float.float(), atol=tol * float(y_float.abs().max()), rtol=0)
        # pickle, state_dict, .to
        buf = io.BytesIO()
        torch.save(model, buf)
        buf.seek(0)
        m2 = torch.load(buf, weights_only=False)
        assert m2.c0._packed.integer and torch.equal(m2(x).float(), y.float())
        m3 = copy.deepcopy(model)
        m3.load_state_dict(model.state_dict())
        assert set(m3.state_dict()) == set(model.state_dict()) and torch.equal(m3(x).float(), y.float())
        m4 = copy.deepcopy(model).to("cpu").to("cuda")
        assert torch.equal(m4(x).float(), y.float())
        assert pickle.loads(pickle.dumps(model.c0._packed)).integer


@pytest.mark.gpu
def test_fallbacks_and_graph(monkeypatch):
    torch.manual_seed(1)
    model = _ConvModel(torch.float32, "i8")
    x = torch.randn(4, 32, 9, 9, device="cuda")
    PW.pack_model_weights(model, integer_conv=True)
    with torch.no_grad():
        y = model(x)
        hx = model.h0(x)
    calls = []
    real = ops.IntegerConv2d.__call__
    monkeypatch.setattr(ops.IntegerConv2d, "__call__", lambda self, *a: calls.append(1) or real(self, *a))
    # autograd recording, forward hooks and an unbatched 3-D input: the packed path
    y_grad = model.c0(hx.clone().requires_grad_(True))
    assert calls == [] and y_grad.requires_grad
    h = model.c0.layer.register_forward_hook(lambda *a: None)
    with torch.no_grad():
        model.c0(hx)
    h.remove()
    with torch.no_grad():
        y3 = model.c0(hx[0])
        assert y3.dim() == 3
    assert calls == []
    with torch.no_grad():
        assert torch.equal(model(x), y) and len(calls) == 2
    # CUDA-graph capture after a warm-up replays the same bits
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.no_grad(), torch.cuda.stream(s):
        model(x)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            y_g = model(x)
    torch.cuda.current_stream().wait_stream(s)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(y_g, y)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["resnet18", "mobilenet_v2"])
def test_benchmark_models_switch(name):
    """The benchmark models packed with integer_conv=True: every switched conv's output equals its integer reference and
    stays within test_model_switch's tolerance of the packed conv on the same input.  (Whole-model outputs are not
    compared: a last-bit difference of one layer may move a holder's code, and 20 layers pass such moves on.)"""
    torch.manual_seed(0)
    model = _torchvision_models()[name]().cuda().eval()
    x = torch.randn(2, 3, 64, 64, device="cuda")
    with torch.no_grad(), _no_tf32():
        packed = copy.deepcopy(model)
        PW.pack_model_weights(packed)
        reports = PW.pack_model_weights(model, integer_conv=True, integer_linear=True)
        switched = [n for n, r in reports.items() if r["weight"].get("integer_conv")]
        assert switched
        seen = {}
        holders = {n: m for n, m in model.named_modules()}
        hooks = []
        for n in switched:
            w = model.get_submodule(n)
            hooks.append(w.register_forward_pre_hook(lambda m, a, n=n: seen.__setitem__(n, a[0])))
        # the pre-hooks sit on the wrapper (not on its layer), so the wrappers keep integer mode
        model(x)
        for hk in hooks:
            hk.remove()
        for n in switched:
            w = model.get_submodule(n)
            h = holders[reports[n]["weight"]["input_holder"]]
            out = w(seen[n])
            assert torch.equal(out.float(), _layer_reference(h, w, seen[n]).float()), n
            ref = packed.get_submodule(n)(seen[n])
            assert out.stride() == ref.stride()
            assert torch.allclose(out, ref, atol=1e-4 * float(ref.abs().max()), rtol=0), n
