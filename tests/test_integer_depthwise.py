"""Integer convolution mode for depthwise Conv2d: mctq_packed_dwconv2d_i8 (csrc/mctq_affine.cu) and the packed-wrapper mode
built on it (pytorch/packed_weights.py, integer_depthwise=True).  Every GPU result is checked bit for bit against an
independent reference of the formula in include/mctq.h: a float64 grouped convolution of the centred codes."""
import contextlib
import copy
import ctypes
import io
import pickle
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import mct_quantizers_b200 as mctq
from mct_quantizers_b200 import _native, ops
from mct_quantizers_b200.pytorch import packed_weights as PW
from mct_quantizers_b200.pytorch import quantizers as Q
from mct_quantizers_b200.pytorch.activation_quantization_holder import PytorchActivationQuantizationHolder
from mct_quantizers_b200.pytorch.packed_weights import integer_depthwise_eligibility

from test_integer_conv import (_act, _conv_wrapper, _fake_pack_model, _fake_packed_conv, _launch_args, _torchvision_models,
                               conv_reference)
from test_integer_lut import _lut_q
from test_packed_linear import _lin_desc

I8, I4, LU8, LI4 = _native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4, _native.PACK_LUT_U8, _native.PACK_LUT_I4
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
E_BADARG, E_DTYPE, E_RANGE, E_LUT = -1, -2, -3, -4
_TAG = {torch.float32: _native.F32, torch.bfloat16: _native.BF16, torch.float16: _native.F16}


# ------------------------------------------------------------------------------------------------ reference
def dw_reference(qx, zx, qw, zw, f, bias, stride, dilation, padding, out_dtype):
    """The formula of include/mctq.h: qx [N, C, H, W] codes, qw [Cout, 1, kh, kw] codes, zw and f with 1 or Cout entries,
    padding (pt, pb, pl, pr).  The centred codes are convolved in float64 with groups = C (exact: |c| < 2^31), the padding
    holds 0, then c is rounded once to f32, scaled, biased and rounded to out_dtype."""
    C, Cout = qx.shape[1], qw.shape[0]
    pt, pb, pl, pr = padding
    xc = F.pad(qx.to(torch.float64) - zx, (pl, pr, pt, pb))
    wc = qw.to(torch.float64) - zw.reshape(-1).to(torch.float64).expand(Cout).reshape(Cout, 1, 1, 1)
    c = F.conv2d(xc, wc, stride=stride, dilation=dilation, groups=C)
    y = c.to(torch.int64).to(torch.float32) * f.reshape(-1).to(torch.float32).expand(Cout)[None, :, None, None]
    if bias is not None:
        y = y + bias.to(torch.float32)[None, :, None, None]
    return y.to(out_dtype)


def test_reference_matches_the_sx_sw_form_channel_by_channel():
    g = torch.Generator().manual_seed(0)
    C, m = 5, 3
    qx = torch.randint(0, 256, (2, C, 9, 8), generator=g)
    qw = torch.randint(-128, 128, (C * m, 1, 3, 2), generator=g)
    zw = torch.randint(-128, 128, (C * m,), generator=g)
    f = torch.rand(C * m, generator=g) * 0.01
    bias = torch.randn(C * m, generator=g)
    args = ((2, 1), (1, 2), (2, 0, 1, 1))
    y = dw_reference(qx, 7, qw, zw, f, bias, *args, torch.float32)
    for o in range(C * m):
        ref = conv_reference(qx[:, o // m:o // m + 1], 7, qw[o:o + 1], zw[o:o + 1], f[o:o + 1], bias[o:o + 1], *args,
                             torch.float32)
        assert torch.equal(y[:, o:o + 1], ref), o


def test_reference_hand_worked():
    # one pixel of code 5, zx = 2, a 3x3 kernel of ones, padding 1: c = (5 - 2) * 1, the 8 padded taps contribute 0
    y = dw_reference(torch.full((1, 1, 1, 1), 5), 2, torch.ones((1, 1, 3, 3), dtype=torch.int64), torch.zeros(1),
                     torch.tensor([0.5]), torch.tensor([1.0]), (1, 1), (1, 1), (1, 1, 1, 1), torch.float32)
    assert y.item() == 2.5
    # zw = 1: every qw - zw is 0
    y = dw_reference(torch.full((1, 1, 1, 1), 5), 2, torch.ones((1, 1, 3, 3), dtype=torch.int64), torch.ones(1),
                     torch.tensor([0.5]), None, (1, 1), (1, 1), (1, 1, 1, 1), torch.float32)
    assert y.item() == 0.0
    # c above 2^24: 17 x 18 taps of 255 * 255, one of 255 * 254 -> c = 19897395 (odd) rounds to an f32 first
    qx = torch.full((1, 1, 17, 18), 255)
    qw = torch.full((1, 1, 17, 18), 255)
    qw[0, 0, 3, 4] = 254
    y = dw_reference(qx, 0, qw, torch.zeros(1), torch.ones(1), None, (1, 1), (1, 1), (0, 0, 0, 0), torch.float32)
    c = 305 * 255 * 255 + 255 * 254
    assert c == 19897395 and y.item() == float(np.float32(c)) and y.item() != c
    # channel multiplier 2: output channels 0, 1 read input channel 0, channels 2, 3 read input channel 1
    qx = torch.tensor([3, 10]).reshape(1, 2, 1, 1)
    y = dw_reference(qx, 1, torch.tensor([1, 2, 3, 4]).reshape(4, 1, 1, 1), torch.zeros(1), torch.ones(1), None, (1, 1),
                     (1, 1), (0, 0, 0, 0), torch.float32)
    assert y.reshape(-1).tolist() == [2.0, 4.0, 27.0, 36.0]


@pytest.mark.parametrize("padding,kernel,stride,dilation,m", [
    (0, 3, 1, 1, 1), (1, 3, 2, 1, 2), ((2, 1), (5, 3), (1, 2), 1, 3), ("valid", 3, 2, 2, 1), ("same", (4, 3), 1, (1, 2), 1),
    ("same", 2, 1, 1, 2), (3, 7, 3, 1, 1), ((0, 2), 1, (2, 1), 1, 1)])
def test_geometry_matches_conv2d(padding, kernel, stride, dilation, m):
    layer = torch.nn.Conv2d(6, 6 * m, kernel, stride=stride, padding=padding, dilation=dilation, groups=6)
    pad = ops.conv_padding(layer)
    for H, W in ((9, 11), (16, 16), (13, 8)):
        ref = layer(torch.randn(2, 6, H, W)).shape
        assert ops.conv_output_hw(H, W, layer.kernel_size, layer.stride, layer.dilation, pad) == tuple(ref[2:])
        y = dw_reference(torch.randint(0, 9, (2, 6, H, W)), 0, torch.ones(tuple(layer.weight.shape), dtype=torch.int64),
                         torch.zeros(1), torch.ones(1), None, layer.stride, layer.dilation, pad, torch.float32)
        assert y.shape == ref


# ------------------------------------------------------------------------------------------------ C-ABI rejections
def _geom(**k):
    g = dict(N=2, H=8, W=8, Cin=16, Ho=8, Wo=8, kh=3, kw=3, sh=1, sw=1, dh=1, dw=1, pt=1, pb=1, pl=1, pr=1)
    g.update(k)
    return _native.MctqConv2dGeom(*(g[f] for f, _ in _native.MctqConv2dGeom._fields_))


TABLE = (ctypes.c_int8 * 256)(*range(-128, 128))


def _dw_call(d, g=None, Cout=16, x=0x7f5000000000, dt=_native.F32, nhwc=0, zx=0, qmin=-128, qmax=127, factor=0x7f6200000000,
             y=0x7f6000000000, table=None):
    lib = _native.load()
    g = g if g is not None else _geom()
    return lib.mctq_packed_dwconv2d_i8(ctypes.byref(d) if d is not None else None, ctypes.byref(g) if g is not False else None,
                                       Cout, x, dt, nhwc, 0.5, zx, qmin, qmax, factor, None, y, table, None)


def test_c_abi_rejections():
    ok = lambda out_f=16, k=9, **kw: _lin_desc(out_f=out_f, in_f=k, **kw)        # noqa: E731
    assert _dw_call(None) == E_BADARG
    assert _dw_call(ok(), g=False) == E_BADARG
    for field in ("H", "W", "Cin", "Ho", "Wo", "kh", "kw", "sh", "sw", "dh", "dw"):
        assert _dw_call(ok(), g=_geom(**{field: 0})) == E_BADARG, field
    assert _dw_call(ok(), g=_geom(N=-1)) == E_BADARG
    for field in ("pt", "pb", "pl", "pr"):
        assert _dw_call(ok(), g=_geom(**{field: -1})) == E_BADARG, field
    assert _dw_call(ok(), nhwc=2) == E_BADARG
    assert _dw_call(ok(out_f=24), Cout=24) == E_BADARG                             # Cout % Cin
    assert _dw_call(ok(out_f=16, k=8)) == E_BADARG                                 # w->n != Cout * kh * kw
    assert _dw_call(ok(C=16, inner=3)) == E_BADARG                                 # parameter layout
    assert _dw_call(ok(C=4)) == E_BADARG
    assert _dw_call(ok(), x=None) == E_BADARG and _dw_call(ok(), y=None) == E_BADARG
    assert _dw_call(ok(), factor=None) == E_BADARG
    d = ok()
    d.codes = None
    assert _dw_call(d) == E_BADARG
    d = ok()
    d.zp = None
    assert _dw_call(d) == E_BADARG                                                 # affine weights need zero points
    assert _dw_call(ok(), table=TABLE) == E_BADARG                                 # a table with an affine kind
    assert _dw_call(ok(kind=LI4)) == E_BADARG                                      # a LUT kind without its table
    assert _dw_call(ok(kind=LU8), table=TABLE, g=_geom(N=0)) == 0
    assert _dw_call(ok(kind=LI4, K=17), table=TABLE) == E_LUT
    assert _dw_call(ok(kind=LU8, K=0), table=TABLE) == E_LUT
    assert _dw_call(ok(kind=LU8, dtype=_native.BF16), dt=_native.BF16, table=TABLE) == E_DTYPE    # LUT weights are f32
    assert _dw_call(ok(dtype=_native.BF16)) == E_DTYPE                             # x dtype != rebuilt dtype
    assert _dw_call(ok(dtype=7), dt=7) == E_DTYPE
    assert _dw_call(ok(), qmin=1, qmax=0) == E_RANGE
    assert _dw_call(ok(), qmin=-129) == E_RANGE and _dw_call(ok(), qmin=0, qmax=256) == E_RANGE
    assert _dw_call(ok(), zx=128) == E_RANGE and _dw_call(ok(), qmin=0, qmax=255, zx=-1) == E_RANGE
    assert _dw_call(ok(), qmin=-100, qmax=100, zx=101) == E_RANGE
    # kh * kw at the int32 bound of the centred sum: accepted (N = 0: no-op); above it: RANGE
    assert _dw_call(ok(k=33025), g=_geom(kh=5, kw=6605, N=0)) == 0
    assert _dw_call(ok(k=33026), g=_geom(kh=2, kw=16513)) == E_RANGE
    assert _dw_call(ok(), g=_geom(N=0)) == 0
    assert _dw_call(ok(out_f=48), Cout=48, g=_geom(N=0)) == 0                     # channel multiplier 3


# ------------------------------------------------------------------------------------------------ eligibility and reports
def _dw_wrapper(c=32, m=1, k=3, **kw):
    w = Q.WeightsSymmetricInferableQuantizer(8, [1.0] * (c * m), True, 0)
    return mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(c, c * m, k, groups=c, **kw), {"weight": w})


def test_eligibility():
    q = _act()
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper()), q) == (True, "")
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper(m=3, k=(5, 2))), q) == (True, "")
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper(c=3)), q) == (True, "")
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper(), channels_last=True), q) == (True, "")
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper(), C=1), q) == (True, "")
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper(), kind=I4), q) == (True, "")
    # the shared reasons, word for word as integer_conv_eligibility gives them
    pairs = [(_dw_wrapper(), _conv_wrapper()),
             (_fake_packed_conv(_dw_wrapper(padding=1, padding_mode="reflect")),
              _fake_packed_conv(_conv_wrapper(padding=1, padding_mode="reflect"))),
             (_fake_packed_conv(_dw_wrapper(), kind=LU8), _fake_packed_conv(_conv_wrapper(), kind=LU8))]
    for dw, dense in pairs:
        assert integer_depthwise_eligibility(dw, q) == PW.integer_conv_eligibility(dense, q)
    assert integer_depthwise_eligibility(_dw_wrapper(), q) == (False, "the weight is not packed")
    lin = mctq.PytorchQuantizationWrapper(torch.nn.Linear(32, 8), {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 8, True, 0)})
    assert integer_depthwise_eligibility(lin, q) == (False, "the layer is Linear, not torch.nn.Conv2d")
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper()), _act("lut")) == \
        PW.integer_conv_eligibility(_fake_packed_conv(_conv_wrapper()), _act("lut"))
    reuse = _act()
    reuse.enable_reuse = True
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper()), reuse) == \
        (False, "the input quantizer reuses its outputs (enable_reuse)")
    ok, why = integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper()), _act(bits=16))
    assert not ok and "8-bit codes" in why
    w = _fake_packed_conv(_dw_wrapper())
    w._packed.entries[0].C, w._packed.entries[0].inner = 32, 3
    assert integer_depthwise_eligibility(w, q) == \
        (False, "the parameters are not per tensor or per output channel (channel_axis 0)")
    # its own reasons
    grouped = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(32, 16, 3, groups=8),
                                              {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 16, True, 0)})
    assert integer_depthwise_eligibility(_fake_packed_conv(grouped), q) == \
        (False, "groups = 8: a grouped convolution with 4 input channels per group is not depthwise")
    assert integer_depthwise_eligibility(_fake_packed_conv(_conv_wrapper()), q) == \
        (False, "groups = 1: not a depthwise convolution")
    w = _fake_packed_conv(_dw_wrapper())
    w._packed.entries[0].stride_out = (1, 9, 3, 96)
    assert integer_depthwise_eligibility(w, q) == \
        (False, "the rebuilt weight is not a contiguous or channels_last [Cout, 1, kh, kw] tensor")
    big = _fake_packed_conv(_dw_wrapper(c=2, k=(2, 16513)))
    assert integer_depthwise_eligibility(big, q) == \
        (False, "kh * kw = 33026 exceeds 33025, the largest window whose int32 sum of code products cannot overflow")
    # under the int32 bound, but a window the kernel cannot stage in shared memory
    assert integer_depthwise_eligibility(_fake_packed_conv(_dw_wrapper(c=2, k=(5, 6605))), q) == \
        (False, "the dilated 5 x 6605 window (5 x 6605 input pixels) does not fit the depthwise kernel's shared memory")


@pytest.mark.parametrize("k,dilation,ok", [((3, 3), 112, True), ((3, 3), 113, False), ((1, 25597), 1, True),
                                           ((1, 25598), 1, False), ((5, 6605), 1, False), ((25597, 1), 1, True),
                                           ((3, 1), (25596, 1), False), ((3, 1), (25595, 1), True)])
def test_eligibility_window_bound(k, dilation, ok):
    """The smallest tile of the kernel (one output of one channel) needs 20 + 4 kh kw + 4 IH IW bytes of the 200 KB: 3x3 at
    dilation 112 (225 x 225 input pixels) fits, at 113 (227 x 227) it does not; a 1 x 25597 row fits, 1 x 25598 does not."""
    w = _fake_packed_conv(_dw_wrapper(c=2, k=k, dilation=dilation))
    got = integer_depthwise_eligibility(w, _act())
    kh, kw = k
    dh, dw = (dilation, dilation) if isinstance(dilation, int) else dilation
    ih, iw = (kh - 1) * dh + 1, (kw - 1) * dw + 1
    assert (20 + 4 * kh * kw + 4 * ih * iw <= 200 * 1024) == ok
    if ok:
        assert got == (True, "")
    else:
        assert got == (False, f"the dilated {kh} x {kw} window ({ih} x {iw} input pixels) does not fit the depthwise "
                              f"kernel's shared memory")
    # the kernel's own answer for a real input of that window, at N = 0 (a no-op when it plans)
    # the kernel's own answer for an input of that window and any of its paddings, both layouts
    for nhwc in (False, True):
        for pad in ((0, 0, 0, 0), (dh, dh, dw, dw)):
            assert (ops.dwconv_plan(2, 2, ih, iw, 2, k, (1, 1), (dh, dw), pad, nhwc) is not None) == ok, (nhwc, pad)


def _plan(N, C, H, W, m, k, stride, dilation, padding, nhwc):
    p = ops.dwconv_plan(N, C, H, W, C * m, k, stride, dilation, padding, nhwc)
    return p and (p["S"], p["TH"], p["TW"])


def test_plan_query():
    # hand-worked from the planner: 3x3, dilation 100, padding 100 on 300 x 300 NCHW planes.  S = 1 (90000 outputs a
    # plane), TW = 64, TH = 2048 / 64 = 32; the 232 x 264 window tile of 4 bytes a pixel is 245 KB: TH halves to 1
    # (201 x 264: 212 KB), then TW to 32 (201 x 232: 182 KB)
    p = ops.dwconv_plan(1, 1, 300, 300, 1, (3, 3), (1, 1), (100, 100), (100, 100, 100, 100))
    assert p == dict(S=1, TH=1, TW=32, IH=201, IW=232, smem_bytes=20 + 36 + 201 * 232 * 4)
    # 3x3, dilation 30, padding 30 on 8 x 8 planes, 32 or more of them: S = 32, TH = TW = 8, slots padded to SB = 34; TH
    # halves to 1 (61 x 68 x 34 x 2 bytes = 282 KB), then S to 16 (SB = 18: 150 KB)
    for nc in (32, 40, 1000):
        p = ops.dwconv_plan(1, nc, 8, 8, nc, (3, 3), (1, 1), (30, 30), (30, 30, 30, 30))
        assert p == dict(S=16, TH=1, TW=8, IH=61, IW=68, smem_bytes=16 * 20 + 9 * 16 * 4 + 61 * 68 * 18 * 2)
    # fewer planes than 32: S is the number of planes (no shrink)
    assert _plan(1, 5, 8, 8, 1, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), False) == (5, 8, 8)
    # NHWC starts at 32 channels of an 8 x 16 tile, whatever C is
    assert _plan(2, 3, 112, 112, 1, (3, 3), (2, 2), (1, 1), (0, 1, 0, 1), True) == (32, 8, 16)
    # a 56 x 56 NCHW plane: one plane per unit, the full width and 2048 / 56 = 36 rows
    assert _plan(2, 144, 56, 56, 1, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), False) == (1, 36, 56)
    # the largest windows that plan, and the first that do not
    assert _plan(1, 1, 225, 225, 1, (3, 3), (1, 1), (112, 112), (0, 0, 0, 0), False) == (1, 1, 1)
    assert _plan(1, 1, 227, 227, 1, (3, 3), (1, 1), (113, 113), (0, 0, 0, 0), False) is None
    assert _plan(1, 1, 1, 25597, 1, (1, 25597), (1, 1), (1, 1), (0, 0, 0, 0), True) == (1, 1, 1)
    assert _plan(1, 1, 1, 25598, 1, (1, 25598), (1, 1), (1, 1), (0, 0, 0, 0), True) is None
    # rejections: those of the launch
    lib = _native.load()
    out = _native.MctqDwPlan()
    assert lib.mctq_packed_dwconv2d_i8_plan(ctypes.byref(_geom()), 16, 0, None) == E_BADARG
    assert lib.mctq_packed_dwconv2d_i8_plan(None, 16, 0, ctypes.byref(out)) == E_BADARG
    assert lib.mctq_packed_dwconv2d_i8_plan(ctypes.byref(_geom()), 24, 0, ctypes.byref(out)) == E_BADARG
    assert lib.mctq_packed_dwconv2d_i8_plan(ctypes.byref(_geom(kh=0)), 16, 0, ctypes.byref(out)) == E_BADARG
    assert lib.mctq_packed_dwconv2d_i8_plan(ctypes.byref(_geom()), 16, 2, ctypes.byref(out)) == E_BADARG
    assert lib.mctq_packed_dwconv2d_i8_plan(ctypes.byref(_geom(kh=2, kw=16513)), 16, 0, ctypes.byref(out)) == E_RANGE
    assert lib.mctq_packed_dwconv2d_i8_plan(ctypes.byref(_geom()), 16, 1, ctypes.byref(out)) == 0
    assert (out.S, out.TH, out.TW, out.IH, out.IW) == (32, 8, 8, 10, 10)
    # the launch refuses exactly the windows the plan query refuses, before any CUDA call
    for kh, kw, d in ((5, 6605, 1), (3, 3, 113), (1, 25598, 1)):
        ih, iw = (kh - 1) * d + 1, (kw - 1) * d + 1
        g = _geom(N=1, Cin=1, H=ih, W=iw, Ho=1, Wo=1, kh=kh, kw=kw, dh=d, dw=d, pt=0, pb=0, pl=0, pr=0)
        assert lib.mctq_packed_dwconv2d_i8_plan(ctypes.byref(g), 1, 0, ctypes.byref(out)) == E_RANGE
        assert _dw_call(_lin_desc(out_f=1, in_f=kh * kw), g=g, Cout=1) == E_RANGE


def _lut_dw(kind=LI4, c=32, k=3, **q):
    w = _dw_wrapper(c=c, k=k)
    w.weights_quantizers["weight"] = _lut_q(c, 16 if kind == LI4 else 64, rank=4, **q)
    _fake_packed_conv(w, kind=kind)
    w._packed.entries[0].quantizer = w.weights_quantizers["weight"]
    w._packed.entries[0].is_signed = False
    return w


@pytest.mark.parametrize("kind", [LI4, LU8])
def test_lut_eligibility(kind):
    q = _act()
    ok, why = integer_depthwise_eligibility(_lut_dw(kind), q)
    assert not ok and "not as int8 / int4 affine codes" in why                     # lut=False
    assert integer_depthwise_eligibility(_lut_dw(kind), q, lut=True) == (True, "")
    assert integer_depthwise_eligibility(_lut_dw(kind, k=1), q, lut=True) == (True, "")   # no row-length multiple
    assert integer_depthwise_eligibility(_lut_dw(kind, pot=True), q, lut=True) == (True, "")
    bad = _lut_dw(kind, bw=9, lut=[-200.0, 0.0, 3.0])
    assert integer_depthwise_eligibility(bad, q, lut=True) == \
        (False, "a LUT value is not an integer in [-128, 127] (the integer modes take the centroids as int8 codes)")
    bad = _lut_dw(kind, thr=[2.0 ** -126] * 32)                                    # sw = 2^-133: subnormal
    assert integer_depthwise_eligibility(bad, q, lut=True) == \
        (False, "a threshold times 2^-(lut_values_bitwidth - 1) is not exact and normal in float32")


def test_flag_needs_integer_conv():
    with pytest.raises(ValueError, match="integer_depthwise=True needs integer_conv=True"):
        PW.pack_wrapper_weights(_dw_wrapper(), integer_depthwise=True, input_quantizer=_act())
    with pytest.raises(ValueError, match="integer_depthwise=True needs integer_conv=True"):
        PW.pack_model_weights(torch.nn.Sequential(_dw_wrapper()), integer_linear=True, integer_depthwise=True)
    with pytest.raises(ValueError, match="integer_depthwise=True needs integer_conv=True"):
        _dw_wrapper().pack_weights(integer_depthwise=True, input_quantizer=_act())


class _Net(torch.nn.Module):
    def __init__(self, wrappers, holders):
        super().__init__()
        self.h = torch.nn.ModuleList(holders)
        self.w = torch.nn.ModuleList(wrappers)

    def forward(self, x):
        return self.w[2](self.h[1](self.w[1](self.w[0](self.h[0](x)))))


def test_model_reports():
    H = lambda: PytorchActivationQuantizationHolder(_act())                      # noqa: E731
    mk = lambda: _Net([_fake_packed_conv(_dw_wrapper()), _fake_packed_conv(_dw_wrapper()),      # noqa: E731
                       _fake_packed_conv(_conv_wrapper(cin=32, cout=8))], [H(), H()])
    without = PW.pack_model_weights(mk(), integer_conv=True)
    net = mk()
    reports = PW.pack_model_weights(net, integer_conv=True, integer_depthwise=True)
    r0, r1, r2 = (reports[f"w.{i}"]["weight"] for i in range(3))
    assert (r0["integer_conv"], r0["integer_conv_reason"], r0["input_holder"]) == (True, "", "h.0")
    assert r1["integer_conv"] is False and "not the output of an activation quantization holder" in r1["integer_conv_reason"]
    assert r2 == without["w.2"]["weight"] and r2["integer_conv"] is True
    assert without["w.0"]["weight"]["integer_conv_reason"] == \
        "groups = 32: a grouped or depthwise convolution is not one matrix product"
    assert net.w[0]._packed.integer and not net.w[1]._packed.integer and net.w[2]._packed.integer


@pytest.mark.parametrize("name", ["resnet18", "mobilenet_v2"])
def test_benchmark_model_reports(name):
    models = _torchvision_models()
    reports = PW.pack_model_weights(_fake_pack_model(models[name]()), integer_conv=True, integer_depthwise=True)
    before = PW.pack_model_weights(_fake_pack_model(models[name]()), integer_conv=True)
    switched = {n for n, r in reports.items() if r["weight"]["integer_conv"]}
    if name == "resnet18":
        assert reports == before
        return
    want = {"features.1.conv.0.0", "features.1.conv.1"}
    want |= {f"features.{i}.conv.{j}" for i in range(2, 18) for j in ("1.0", "2")}
    assert switched == want and len(switched) == 34
    for i in range(2, 18):                                 # expansion convs read the previous block's un-quantized output
        n = f"features.{i}.conv.0.0"
        assert reports[n]["weight"] == before[n]["weight"]
        assert "not the output of an activation quantization holder" in reports[n]["weight"]["integer_conv_reason"]
    dw = {"features.1.conv.0.0"} | {f"features.{i}.conv.1.0" for i in range(2, 18)}
    assert all("groups" in before[n]["weight"]["integer_conv_reason"] for n in dw)
    assert all(reports[n] == before[n] for n in reports if n not in dw)


def test_fake_implementation():
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        x = torch.empty(2, 8, 9, 7)
        codes = torch.empty(16 * 6, dtype=torch.uint8)
        f = torch.empty(16)
        for cl in (False, True):
            y = torch.ops.mctq.packed_dwconv2d_i8(x, 0.1, 0, -128, 127, codes, I8, True, 16, [3, 2], [2, 1], [1, 2],
                                                  [1, 0, 2, 1], torch.zeros(16, dtype=torch.int32), f, None, None, cl)
            ref = torch.empty(2, 16, 4, 8)          # (9 + 1 - 3) // 2 + 1, (7 + 3 - 3) // 1 + 1
            assert y.shape == ref.shape and y.dtype == x.dtype
            assert y.stride() == (ref.to(memory_format=torch.channels_last) if cl else ref).stride()


# ------------------------------------------------------------------------------------------------ GPU: the kernel
def _scalar_codes(x, scale, zp, qmin, qmax):
    """Codes of mctq_fq_affine_scalar with code_mode INT8, in x's logical order (int64)."""
    lib = _native.load()
    xd = x.contiguous()
    y = torch.empty_like(xd)
    codes = torch.empty(xd.shape, dtype=torch.int8 if qmin < 0 else torch.uint8, device=x.device)
    rc = lib.mctq_fq_affine_scalar(xd.data_ptr(), y.data_ptr(), codes.data_ptr(), xd.numel(), _TAG[x.dtype],
                                   float(np.float32(scale)), zp, qmin, qmax, _native.CODES_INT8,
                                   torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "mctq_fq_affine_scalar")
    return codes.to(torch.int64)


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _dw_case(N, C, H, W, m, k, stride, dilation, padding, kind, w_signed, per_channel, zw_nonzero, x_signed, zx, dtype,
             with_bias, nhwc, seed, lut_k=None):
    """One mctq_packed_dwconv2d_i8 call against dw_reference, then the same call into the middle of a NaN buffer."""
    g = torch.Generator().manual_seed(seed)
    Cout, (kh, kw) = C * m, k
    Cw = Cout if per_channel else 1
    if kind in (LI4, LU8):
        table = torch.randint(-128, 128, (lut_k,), generator=g, dtype=torch.int32)
        idx = torch.randint(0, lut_k, (Cout, 1, kh, kw), generator=g, dtype=torch.int32)
        qw, zw, codes, lut = table[idx], torch.zeros(Cw, dtype=torch.int32), ops.pack_weight_codes(idx, kind, False), table
    else:
        lo, hi = ((-8, 7) if w_signed else (0, 15)) if kind == I4 else ((-128, 127) if w_signed else (0, 255))
        qw = torch.randint(lo, hi + 1, (Cout, 1, kh, kw), generator=g, dtype=torch.int32)
        zw = torch.randint(lo, hi + 1, (Cw,), generator=g, dtype=torch.int32) if zw_nonzero else torch.zeros(Cw, dtype=torch.int32)
        codes, lut = ops.pack_weight_codes(qw, kind, w_signed), None
    x_scale = 0.0371
    f = (torch.tensor(np.float32(x_scale)) * (torch.rand(Cw, generator=g) * 0.02 + 0.001)).float()
    qmin, qmax = (-128, 127) if x_signed else (0, 255)
    x = (torch.randn((N, C, H, W), generator=g) * x_scale * 60 + x_scale * (zx - (qmin + qmax) / 2)).to(dtype)
    flat = x.view(-1)
    flat[::97] = float("nan")
    flat[5::89] = float("inf")
    flat[7::83] = -float("inf")
    x = x.cuda()
    bias = (torch.randn(Cout, generator=g) * 3).to(dtype).cuda() if with_bias else None
    conv = ops.IntegerDepthwiseConv2d.from_parts(codes.cuda(), kind, w_signed, dtype, Cout, C, k, stride, dilation, padding,
                                                 f.cuda(), None if lut is not None else zw.cuda(), x_scale, zx, qmin, qmax,
                                                 lut)
    qx = _scalar_codes(x, x_scale, zx, qmin, qmax)
    ref = dw_reference(qx.cpu(), zx, qw, zw, f, bias.cpu() if bias is not None else None, stride, dilation, padding, dtype)
    xin = x.to(memory_format=torch.channels_last) if nhwc else x
    y = conv.conv(xin, bias, channels_last=nhwc)
    assert y.shape == ref.shape and y.is_contiguous(memory_format=torch.channels_last if nhwc else torch.contiguous_format)
    assert torch.equal(_bits(y.cpu()), _bits(ref)), f"{(y.cpu().float() - ref.float()).abs().max()}"
    n = y.numel()
    canary = torch.full((n + 64,), float("nan"), dtype=dtype, device="cuda")
    out = canary[32:32 + n]
    Ho, Wo = y.shape[2:]
    geo = _native.MctqConv2dGeom(N, H, W, C, Ho, Wo, kh, kw, *stride, *dilation, *padding)
    rc = _native.load().mctq_packed_dwconv2d_i8(conv._w._desc_ptr, ctypes.addressof(geo), Cout, xin.data_ptr(), _TAG[dtype],
                                                int(nhwc), conv.x_scale, zx, qmin, qmax, conv.factor.data_ptr(),
                                                bias.data_ptr() if bias is not None else None, out.data_ptr(),
                                                conv._w.lut.ctypes.data if lut is not None else None,
                                                torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "mctq_packed_dwconv2d_i8")
    assert torch.isnan(canary[:32]).all() and torch.isnan(canary[32 + n:]).all()
    assert torch.equal(_bits(out), _bits(y.permute(0, 2, 3, 1) if nhwc else y).reshape(-1))
    return conv


# (N, C, H, W, m, kernel, stride, dilation, padding (pt, pb, pl, pr))
_SHAPES = [
    (2, 32, 14, 14, 1, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1)),
    (3, 17, 11, 13, 2, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1)),
    (1, 3, 12, 10, 3, (5, 5), (1, 2), (2, 1), (4, 3, 2, 1)),                 # asymmetric, dilated, multiplier 3
    (2, 1, 15, 15, 1, (7, 7), (3, 3), (1, 1), (3, 3, 3, 3)),
    (1, 24, 10, 9, 1, (3, 2), (1, 1), (2, 2), (2, 0, 0, 2)),
    (4, 960, 7, 7, 1, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1)),
    (2, 40, 9, 70, 2, (1, 1), (2, 1), (1, 1), (0, 0, 0, 0)),
    (1, 16, 33, 66, 1, (4, 3), (1, 1), (1, 2), (1, 2, 2, 2)),                # 'same' of a 4 x 3 kernel, dilation (1, 2)
    (1, 8, 5, 6, 1, (6, 6), (1, 1), (1, 1), (2, 3, 2, 3)),
]
_CONFIGS = [(kind, ws, xs, zx) for kind in (I8, I4) for ws in (True, False) for xs, zx in ((True, 0), (True, -7), (False, 0),
                                                                                            (False, 128))]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ci", range(len(_CONFIGS)))
def test_dwconv_bit_exact(ci, dtype):
    kind, ws, xs, zx = _CONFIGS[ci]
    for si in range(ci % 3, len(_SHAPES), 3):
        N, C, H, W, m, k, st, dil, pad = _SHAPES[si]
        _dw_case(N, C, H, W, m, k, st, dil, pad, kind, ws, per_channel=(si + ci) % 2 == 0, zw_nonzero=(si + ci) % 3 != 0,
                 x_signed=xs, zx=zx, dtype=dtype, with_bias=si % 2 == 1, nhwc=(si + ci) % 4 < 2, seed=1000 * ci + si)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [LI4, LU8])
@pytest.mark.parametrize("nhwc", [False, True])
def test_dwconv_lut_bit_exact(kind, nhwc):
    for si, (N, C, H, W, m, k, st, dil, pad) in enumerate(_SHAPES):
        _dw_case(N, C, H, W, m, k, st, dil, pad, kind, False, per_channel=si % 2 == 0, zw_nonzero=False, x_signed=si % 3 == 1,
                 zx=(0, -3, 200)[si % 3], dtype=torch.float32, with_bias=si % 2 == 0, nhwc=nhwc, seed=50 + si,
                 lut_k=16 if kind == LI4 else (256, 200, 3)[si % 3])


@pytest.mark.gpu
def test_many_planes_and_a_large_input():
    # N * C above 65535, both layouts
    _dw_case(70, 1000, 5, 5, 1, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), I8, True, True, True, True, 3, torch.bfloat16, True,
             False, 7)
    _dw_case(70, 1000, 5, 5, 1, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1), I4, True, False, False, False, 0, torch.float16, False,
             True, 8)
    # one input of more than 2^31 elements (bf16): small integer values, scale 1, weight codes 1 -> y is the 3x3 box sum
    N, H, W = 2, 33000, 33000
    x = torch.randint(-3, 4, (N, 1, H, W), dtype=torch.int8, device="cuda").to(torch.bfloat16)
    assert x.numel() > 2 ** 31
    conv = ops.IntegerDepthwiseConv2d.from_parts(torch.ones(9, dtype=torch.int8, device="cuda"), I8, True, torch.bfloat16, 1,
                                                 1, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), torch.ones(1, device="cuda"),
                                                 torch.zeros(1, dtype=torch.int32, device="cuda"), 1.0, 0, -128, 127)
    y = conv.conv(x)
    for b in range(N):
        for r0 in range(0, H, 4096):
            r1 = min(H, r0 + 4096)
            xs = F.pad(x[b:b + 1, :, max(r0 - 1, 0):r1 + 1].float(), (1, 1, 1 if r0 == 0 else 0, 1 if r1 == H else 0))
            ref = F.avg_pool2d(xs, 3, stride=1, divisor_override=1).to(torch.bfloat16)
            assert torch.equal(_bits(y[b:b + 1, :, r0:r1]), _bits(ref)), (b, r0)
    del x, y


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("qname", ["s8", "u8", "uniform"])
def test_in_kernel_codes(dtype, qname):
    """A 1x1 weight of code 1, zw = 0, f = 1, no bias: y = qx - zx, element for element the codes of quantize_rows_i8."""
    q = {"s8": _act(), "u8": _act(signed=False), "uniform": Q.ActivationUniformInferableQuantizer(8, [-1.3], [2.9])}[qname]
    s, z, qmin, qmax = _launch_args(q)
    x = torch.randn(3, 19, 13, 11) * 3
    flat = x.view(-1)
    flat[::97] = float("nan")
    flat[5::89] = float("inf")
    flat[7::83] = -float("inf")
    steps = (torch.arange(flat.numel()) % 601 - 300).float()
    flat[1::7] = (steps[1::7] + 0.5) * float(np.float32(s))      # exact halves of the scale
    flat[2::71] = float(qmax - z) * float(np.float32(s)) * 1.5    # beyond the range ends
    flat[3::73] = float(qmin - z) * float(np.float32(s)) * 1.5
    x = x.to(dtype).cuda()
    conv = ops.IntegerDepthwiseConv2d.from_parts(torch.ones(19, dtype=torch.int8, device="cuda"), I8, True, dtype, 19, 19,
                                                 (1, 1), (1, 1), (1, 1), (0, 0, 0, 0), torch.ones(1, device="cuda"),
                                                 torch.zeros(1, dtype=torch.int32, device="cuda"), s, z, qmin, qmax)
    codes, _ = ops.quantize_rows_i8(x.permute(0, 2, 3, 1), s, z, qmin, qmax, False)
    want = (codes.to(torch.int32) - z).permute(0, 3, 1, 2).to(dtype)
    for cl in (False, True):
        y = conv.conv(x, None, cl)
        assert torch.equal(y.float(), want.float())
    assert {qmin - z, qmax - z} <= set(want.float().unique().tolist())


# ------------------------------------------------------------------------------------------------ GPU: module level
@contextlib.contextmanager
def _no_tf32():
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32 = prev


class _DwModel(torch.nn.Module):
    """holder -> depthwise Conv (multiplier m)."""

    def __init__(self, dtype, wq_kind, m=1, weight_cl=False, bias=True):
        super().__init__()
        C = 24
        if wq_kind == "lut":
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                wq = Q.WeightsLUTSymmetricInferableQuantizer(4, [float(v) for v in range(-64, 64, 8)],
                                                             [0.25 + 0.125 * (c % 4) for c in range(C * m)], True, 0, 4, 8)
        elif wq_kind == "i4":
            wq = Q.WeightsSymmetricInferableQuantizer(4, [0.5] * (C * m), True, 0)
        else:
            wq = Q.WeightsUniformInferableQuantizer(8, [-0.3] * (C * m), [0.2] * (C * m), True, 0)
        self.h0 = PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [-1.7], [2.3]))
        self.c0 = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(C, C * m, 3, padding=1, groups=C, bias=bias),
                                                  {"weight": wq})
        self.to(dtype).cuda()
        if weight_cl:
            self.c0.layer.weight.data = self.c0.layer.weight.data.to(memory_format=torch.channels_last)

    def forward(self, x):
        return self.c0(self.h0(x))


def _agree(y, hx, model_float, dtype):
    """|y - y64| <= 2^-21 (sum |Q(x) W| + |b|), y64 the f64 fake-quant conv; for bf16 / f16 also one rounding of T on each
    factor of every product (the holder's output and the rebuilt weight are T roundings of sx (qx - zx) and sw (qw - zw))
    and on y."""
    layer = model_float.c0.layer
    Wq = model_float.c0.get_quantized_weights()["weight"].double()
    b = layer.bias.double() if layer.bias is not None else None
    y64 = F.conv2d(hx.double(), Wq, b, padding=1, groups=layer.groups)
    mag = F.conv2d(hx.double().abs(), Wq.abs(), b.abs() if b is not None else None, padding=1, groups=layer.groups)
    u = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}[dtype]
    tol = (2.0 ** -21 + 2 * u) * mag + u * y64.abs() + (2.0 ** -24 if dtype == torch.float16 else 0.0)
    assert bool(((y.double() - y64).abs() <= tol).all()), float(((y.double() - y64).abs() - tol).max())


def _module_reference(model, x):
    """The formula for the switched model, with Q's codes of the holder's output."""
    e = model.c0._packed.entries[0]
    s, z, qmin, qmax = _launch_args(model.h0.activation_holder_quantizer)
    hx = model.h0(x)
    qx = _scalar_codes(hx, s, z, qmin, qmax)
    it = e.plan_item()
    Cout, _, kh, kw = e.shape_out
    qw = ops.weight_code_values(e.codes, e.kind, e.is_signed, Cout, kh * kw)
    sc, zw = it[8], it[9]
    if e.kind in _native.PACK_LUT_KINDS:
        wq = e.quantizer
        qw = torch.as_tensor(wq._lut_values_np).to(torch.int64).cuda()[qw.to(torch.int64)]
        sc, zw = sc * 2.0 ** -(int(wq.lut_values_bitwidth) - 1), torch.zeros(1, dtype=torch.int32, device="cuda")
    f = torch.tensor(np.float32(s)).cuda() * sc
    layer = model.c0.layer
    return hx, dw_reference(qx.cpu(), z, qw.reshape(Cout, 1, kh, kw).cpu(), zw.cpu(), f.cpu(),
                            layer.bias.cpu() if layer.bias is not None else None, layer.stride, layer.dilation,
                            ops.conv_padding(layer), x.dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,wq_kind,m,layout", [
    (torch.float32, "i8", 1, "nchw"), (torch.bfloat16, "i8", 2, "x_cl"), (torch.float16, "i4", 1, "w_cl"),
    (torch.bfloat16, "i4", 3, "nchw"), (torch.float32, "lut", 1, "x_cl"), (torch.float32, "lut", 2, "nchw"),
    (torch.float16, "i8", 1, "x_cl")])
def test_model_switch(dtype, wq_kind, m, layout):
    torch.manual_seed(0)
    model = _DwModel(dtype, wq_kind, m, weight_cl=layout == "w_cl", bias=m != 3)
    x = (torch.randn(3, 24, 11, 10, device="cuda") * 1.5).to(dtype)
    if layout == "x_cl":
        x = x.to(memory_format=torch.channels_last)
    with torch.no_grad(), _no_tf32():
        model_float = copy.deepcopy(model)
        packed = copy.deepcopy(model)
        PW.pack_model_weights(packed)
        y_packed = packed(x)
        lut = wq_kind == "lut"
        report = PW.pack_model_weights(model, integer_conv=True, integer_depthwise=True, integer_lut=lut)
        r = report["c0"]["weight"]
        assert (r["packed"], r["integer_conv"], r["integer_conv_reason"], r["input_holder"]) == (True, True, "", "h0")
        y = model(x)
        hx, ref = _module_reference(model, x)
        assert torch.equal(_bits(y.cpu()), _bits(ref))
        assert y.stride() == y_packed.stride()
        assert torch.equal(_bits(model(x)), _bits(y))                               # two calls, same bits
        _agree(y, hx, model_float, dtype)
        # pickle, state_dict, .to
        buf = io.BytesIO()
        torch.save(model, buf)
        buf.seek(0)
        m2 = torch.load(buf, weights_only=False)
        assert m2.c0._packed.integer and torch.equal(_bits(m2(x)), _bits(y))
        m3 = copy.deepcopy(model)
        m3.load_state_dict(model.state_dict())
        assert set(m3.state_dict()) == set(packed.state_dict()) and torch.equal(_bits(m3(x)), _bits(y))
        m4 = copy.deepcopy(model).to("cpu").to("cuda")
        assert torch.equal(_bits(m4(x)), _bits(y))
        assert pickle.loads(pickle.dumps(model.c0._packed)).integer
        # torch op = class
        e = model.c0._packed.entries[0]
        st = model.c0._packed.__dict__["_ilin"][1]
        lut_t = torch.as_tensor(st._w.lut.astype(np.int32)) if lut else None
        args = (st.x_scale, st.x_zp, st.x_qmin, st.x_qmax, e.codes, e.kind, e.is_signed, st.out_channels, [3, 3], [1, 1],
                [1, 1], [1, 1, 1, 1], None if lut else e.plan_item()[9], st.factor, lut_t, model.c0.layer.bias,
                y.is_contiguous(memory_format=torch.channels_last) and not y.is_contiguous())
        assert torch.equal(_bits(torch.ops.mctq.packed_dwconv2d_i8(hx, *args)), _bits(y))
        y_cpu = torch.ops.mctq.packed_dwconv2d_i8(hx.cpu(), *[a.cpu() if isinstance(a, torch.Tensor) else a for a in args])
        assert torch.equal(_bits(y_cpu), _bits(y.cpu()))


@pytest.mark.gpu
def test_switch_one_wrapper_in_place():
    torch.manual_seed(2)
    model = _DwModel(torch.float32, "i8")
    x = torch.randn(2, 24, 9, 9, device="cuda")
    with torch.no_grad():
        rep = model.c0.pack_weights(integer_conv=True, integer_depthwise=True,
                                    input_quantizer=model.h0.activation_holder_quantizer)
        assert rep["weight"]["integer_conv"] and model.c0._packed.integer
        assert torch.equal(_bits(model(x).cpu()), _bits(_module_reference(model, x)[1]))


@pytest.mark.gpu
def test_fallbacks_and_graph(monkeypatch):
    torch.manual_seed(1)
    model = _DwModel(torch.float32, "i8")
    x = torch.randn(4, 24, 9, 9, device="cuda")
    PW.pack_model_weights(model, integer_conv=True, integer_depthwise=True)
    with torch.no_grad():
        y = model(x)
        hx = model.h0(x)
    calls = []
    real = ops.IntegerDepthwiseConv2d.__call__
    monkeypatch.setattr(ops.IntegerDepthwiseConv2d, "__call__", lambda self, *a: calls.append(1) or real(self, *a))
    y_grad = model.c0(hx.clone().requires_grad_(True))
    assert calls == [] and y_grad.requires_grad
    h = model.c0.layer.register_forward_hook(lambda *a: None)
    with torch.no_grad():
        model.c0(hx)
    h.remove()
    with torch.no_grad():
        assert model.c0(hx[0]).dim() == 3
    assert calls == []
    with torch.no_grad():
        assert torch.equal(model(x), y) and len(calls) == 1
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
def test_mobilenet_v2_switches_34_convs():
    torch.manual_seed(0)
    model = _torchvision_models()["mobilenet_v2"]().cuda().eval()
    x = torch.randn(4, 3, 96, 96, device="cuda")
    with torch.no_grad():
        reports = PW.pack_model_weights(model, integer_conv=True, integer_depthwise=True)
        assert sum(bool(r["weight"]["integer_conv"]) for r in reports.values()) == 34
        y = model(x)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            model(x)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=s):
                y_g = model(x)
        torch.cuda.current_stream().wait_stream(s)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(_bits(y_g), _bits(y))
        dw = model.get_submodule("features.5.conv.1.0")
        assert isinstance(dw._packed.__dict__["_ilin"][1], ops.IntegerDepthwiseConv2d)
