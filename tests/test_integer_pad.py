"""Padded integer modes (integer_pad=True, DESIGN §7f): Linear rows and Conv2d channel counts off the GEMM's granule, their
codes padded with channel pads (x code zx, counted in K, Sx and Sw) and, for the narrow gather, a row tail.  Every output is
checked bit for bit against the unchanged references of the integer modes over the real row."""
import copy
import ctypes
import io
import pickle

import numpy as np
import pytest
import torch

import mct_quantizers_b200 as mctq
from mct_quantizers_b200 import _native, ops
from mct_quantizers_b200.pytorch import packed_weights as PW
from mct_quantizers_b200.pytorch import quantizers as Q
from mct_quantizers_b200.pytorch.activation_quantization_holder import PytorchActivationQuantizationHolder
from mct_quantizers_b200.pytorch.packed_weights import integer_conv_eligibility, integer_linear_eligibility

from test_integer_conv import (_act, _conv_wrapper, _fake_packed_conv, _fake_pack_model, _launch_args, _no_tf32,
                               _scalar_codes, _special_x, conv_reference)
from test_integer_lut import _lut_conv, _lut_lin
from test_packed_linear import _fake_packed, _lin_desc

I8, I4, LI4, LU8 = _native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4, _native.PACK_LUT_I4, _native.PACK_LUT_U8
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
E_BADARG, E_DTYPE, E_RANGE = -1, -2, -3
_TAG = {torch.float32: _native.F32, torch.bfloat16: _native.BF16, torch.float16: _native.F16}


# ------------------------------------------------------------------------------------------------ helpers on the host
def test_code_pitch():
    assert ops.conv_code_pitch(3, 7, 7, I8) == (4, 208)                # narrow: 196 + a row tail of 12
    assert ops.conv_code_pitch(3, 3, 3, I8) == (4, 48)
    assert ops.conv_code_pitch(3, 3, 3, I4) == (4, 64)
    assert ops.conv_code_pitch(6, 1, 1, LU8) == (8, 16)
    assert ops.conv_code_pitch(8, 1, 1, LI4) == (8, 32)
    assert ops.conv_code_pitch(10, 1, 1, I8) == (16, 16)
    assert ops.conv_code_pitch(120, 1, 1, I8) == (128, 128)
    assert ops.conv_code_pitch(24, 1, 1, I4) == (32, 32)               # 1 * 32 % 32 == 0
    assert ops.conv_code_pitch(40, 1, 1, I4) == (64, 64)               # 48 is not a multiple of 32: Cin rounded to 32
    assert ops.conv_code_pitch(40, 3, 3, I8) == (48, 432)
    assert [ops.linear_code_pitch(k, I8) for k in (1, 3, 24, 440, 1000)] == [16, 16, 32, 448, 1008]
    assert [ops.linear_code_pitch(k, LI4) for k in (3, 24, 440)] == [32, 32, 448]


@pytest.mark.parametrize("kind", [I8, I4, LI4, LU8])
@pytest.mark.parametrize("channels_last", [False, True])
def test_padded_code_rows(kind, channels_last):
    g = torch.Generator().manual_seed(kind)
    lo, hi = (-8, 8) if kind == I4 else (0, 16) if kind == LI4 else (-128, 128) if kind == I8 else (0, 256)
    signed = kind in (I8, I4)
    w = torch.randint(lo, hi, (5, 3, 2, 3), generator=g, dtype=torch.int32)          # [Cout, Cin, kh, kw]
    mem = w.permute(0, 2, 3, 1) if channels_last else w
    codes = ops.pack_weight_codes(mem.contiguous(), kind, signed)
    rows = ops.padded_code_rows(codes, kind, signed, 5, 3, 2, 3, channels_last, 4, 32)
    ref = torch.zeros((5, 32), dtype=torch.int32)
    for r in range(2):
        for s in range(3):
            for c in range(3):
                ref[:, (r * 3 + s) * 4 + c] = w[:, c, r, s]
    assert torch.equal(rows, ref)
    packed = ops.pack_code_rows(rows, kind, signed, codes)
    assert packed.dtype == codes.dtype
    assert torch.equal(ops.weight_code_values(packed, kind, signed, 5, 32), ref)
    lin = ops.padded_code_rows(ops.pack_weight_codes(w.reshape(5, 18), kind, signed), kind, signed, 5, 18, 1, 1, False, 32,
                               32)
    assert torch.equal(lin[:, :18], w.reshape(5, 18)) and not lin[:, 18:].any()


# ------------------------------------------------------------------------------------------------ eligibility
def _lin_wrapper(in_f, out_f=8):
    w = mctq.PytorchQuantizationWrapper(torch.nn.Linear(in_f, out_f),
                                        {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0] * out_f, True, 0)})
    return _fake_packed(w)


def _kinded(w, kind):
    w._packed.entries[0].kind = kind
    return w


CINS = [1, 3, 4, 6, 8, 10, 24, 40, 120, 200]


@pytest.mark.parametrize("kind", [I8, I4, LI4, LU8])
def test_eligibility_matrix(kind):
    q = _act()
    lut = kind in (LI4, LU8)
    step = 32 if kind in (I4, LI4) else 16
    for cin in CINS:
        for k in (1, 3):
            mk = (lambda: _lut_conv(cin=cin, k=k, kind=kind)) if lut else \
                (lambda: _fake_packed_conv(_conv_wrapper(cin=cin, k=k), kind=kind))
            before = integer_conv_eligibility(mk(), q, lut=lut)
            after = integer_conv_eligibility(mk(), q, lut=lut, pad=True)
            K = cin * k * k
            if cin % 16 == 0 and K % step == 0:
                assert before == after == (True, "")
            else:
                assert not before[0] and ("in_channels" in before[1] or "multiple of 32" in before[1]), before
                assert after == (True, ""), (cin, k, after)
            assert integer_conv_eligibility(mk(), q, lut=lut) == before          # the flag changes nothing afterwards
    for in_f in (3, 24, 440):
        mk = (lambda: _lut_lin(in_f=in_f, kind=kind)) if lut else (lambda: _kinded(_lin_wrapper(in_f), kind))
        before = integer_linear_eligibility(mk(), q, lut=lut)
        after = integer_linear_eligibility(mk(), q, lut=lut, pad=True)
        if in_f % step == 0:
            assert before == after == (True, "")
        else:
            assert not before[0] and f"in_features = {in_f} is not a multiple of {step}" in before[1]
            assert after == (True, "")


def test_padded_row_bound_reason():
    # int8 weights, uint8 x: bound 65793.  K = 65793 fits, padded to 65808 it does not
    q = _act(signed=False)
    ok, why = integer_linear_eligibility(_lin_wrapper(65793, 2), q, pad=True)
    assert not ok and why == ("in_features = 65793 padded to a row of 65808 exceeds 65793, the largest row length whose "
                              "int32 sum of code products cannot overflow")
    assert integer_linear_eligibility(_lin_wrapper(65792, 2), q, pad=True) == (True, "")
    ok, why = integer_linear_eligibility(_lin_wrapper(65809, 2), q, pad=True)
    assert not ok and why.startswith("in_features = 65809 exceeds 65793")
    ok, why = integer_conv_eligibility(_fake_packed_conv(_conv_wrapper(cin=65793, cout=2, k=1)), q, pad=True)
    assert not ok and "padded to a row of 65808 exceeds 65793" in why


def test_flag_needs_an_integer_mode():
    with pytest.raises(ValueError, match="integer_pad=True needs integer_linear=True and / or integer_conv=True"):
        PW.pack_wrapper_weights(_conv_wrapper(), integer_pad=True)
    with pytest.raises(ValueError, match="integer_pad=True needs"):
        PW.pack_model_weights(torch.nn.Sequential(_conv_wrapper()), integer_pad=True)
    with pytest.raises(ValueError, match="integer_pad=True needs"):
        _conv_wrapper().pack_weights(integer_pad=True)


# ------------------------------------------------------------------------------------------------ C-ABI rejections
def _geom(**k):
    g = dict(N=2, H=8, W=8, Cin=3, Ho=8, Wo=8, kh=3, kw=3, sh=1, sw=1, dh=1, dw=1, pt=1, pb=1, pl=1, pr=1)
    g.update(k)
    return _native.MctqConv2dGeom(*(g[f] for f, _ in _native.MctqConv2dGeom._fields_))


def _pconv(d, g=None, Cp=4, Cout=10, xq=0x7f5000000000, x_signed=1, zx=0, w_rowsum=0x7f6100000000, factor=0x7f6200000000,
           y=0x7f6000000000, nchw=1, table=None):
    g = g if g is not None else _geom()
    return _native.load().mctq_packed_conv2d_i8_padded(
        ctypes.byref(d) if d is not None else None, ctypes.byref(g) if g is not False else None, Cp, Cout, xq, x_signed, zx,
        None, w_rowsum, factor, None, d.y_dtype if d is not None else _native.F32, y, nchw, table, None)


def _plin(d, in_f=3, ldc=16, M=4, xq=0x7f5000000000, table=None):
    return _native.load().mctq_packed_linear_i8_padded(
        ctypes.byref(d) if d is not None else None, 10, in_f, ldc, xq, 1, 0, M, None, 0x7f6100000000, 0x7f6200000000, None,
        d.y_dtype if d is not None else _native.F32, 0x7f6000000000, 10, table, None)


def test_c_abi_rejections():
    table = (ctypes.c_int8 * 256)(*range(-128, 128))
    # conv: the narrow gather of Cp = 4 over a 3x3 window is a row of 36 codes rounded up to 48
    ok = lambda **k: _lin_desc(out_f=10, in_f=48, **k)                              # noqa: E731
    assert _pconv(ok(), g=_geom(N=0)) == 0
    assert _pconv(None) == E_BADARG and _pconv(ok(), g=False) == E_BADARG
    for cp in (2, 3, 5, 12, 20, 24):
        assert _pconv(ok(), Cp=cp) == E_BADARG, cp                                  # Cp not in {4, 8, 16k}
    assert _pconv(ok(), g=_geom(Cin=5)) == E_BADARG                                  # Cp < Cin
    assert _pconv(ok(), g=_geom(Cin=0)) == E_BADARG
    assert _pconv(_lin_desc(out_f=10, in_f=36)) == E_BADARG                          # the row tail is part of the row
    assert _pconv(_lin_desc(out_f=10, in_f=64, kind=I4), g=_geom(N=0)) == 0          # int4: 36 -> 64
    assert _pconv(_lin_desc(out_f=10, in_f=48, kind=I4)) == E_BADARG
    assert _pconv(_lin_desc(out_f=10, in_f=16 * 9), Cp=16, g=_geom(N=0)) == 0         # wide: Cin := Cp
    assert _pconv(_lin_desc(out_f=10, in_f=16, kind=I4), Cp=16, g=_geom(kh=1, kw=1)) == E_BADARG    # 16 % 32
    assert _pconv(_lin_desc(out_f=10, in_f=48, kind=LU8)) == E_BADARG                # LUT kind without a table
    assert _pconv(ok(), table=table) == E_BADARG                                     # a table for an affine kind
    assert _pconv(ok(), xq=0x7f5000000008) == E_BADARG
    assert _pconv(ok(), zx=3, w_rowsum=None) == E_BADARG
    assert _pconv(ok(dtype=_native.BF16), g=_geom(N=0)) == 0
    assert _pconv(ok(), x_signed=1, zx=128) == E_RANGE
    assert _pconv(ok(), g=_geom(N=2 ** 30, Ho=2, Wo=1)) == E_BADARG
    # the int32 bound applies to the kernel's row: Cp = 16 * 4097 over a 1x1 window with int8 x int8 (131071)
    assert _pconv(_lin_desc(out_f=2, in_f=16 * 8192), Cp=16 * 8192, g=_geom(Cin=16 * 8191 + 1, kh=1, kw=1), Cout=2) == E_RANGE
    # linear
    assert _plin(_lin_desc(out_f=10, in_f=16), M=0) == 0
    assert _plin(None) == E_BADARG
    assert _plin(_lin_desc(out_f=10, in_f=16), in_f=17) == E_BADARG                  # a pitch smaller than K
    assert _plin(_lin_desc(out_f=10, in_f=16), in_f=0) == E_BADARG
    assert _plin(_lin_desc(out_f=10, in_f=20), ldc=20) == E_BADARG                   # unaligned pitch
    assert _plin(_lin_desc(out_f=10, in_f=16, kind=I4), ldc=16) == E_BADARG          # int4: a multiple of 32
    assert _plin(_lin_desc(out_f=10, in_f=16), table=table) == E_BADARG
    assert _plin(_lin_desc(out_f=10, in_f=16, kind=LU8)) == E_BADARG
    assert _plin(_lin_desc(out_f=10, in_f=16), xq=0x7f5000000004) == E_BADARG
    lib = _native.load()
    qr = lambda **k: lib.mctq_quantize_rows_i8_padded(k.get("x", 0x7f5000000000), k.get("dt", _native.F32), k.get("M", 4),   # noqa: E731
                                                       k.get("K", 3), k.get("ldc", 4), 1.0, k.get("zp", 0),
                                                       k.get("qmin", -128), k.get("qmax", 127),
                                                       k.get("codes", 0x7f6000000000), None, None)
    assert qr(M=0) == 0
    assert qr(x=None) == E_BADARG and qr(codes=None) == E_BADARG and qr(K=0) == E_BADARG and qr(M=-1) == E_BADARG
    assert qr(ldc=2) == E_BADARG and qr(ldc=6) == E_BADARG and qr(codes=0x7f6000000002) == E_BADARG
    assert qr(dt=5) == E_DTYPE and qr(qmin=1, qmax=0) == E_RANGE and qr(zp=128) == E_RANGE
    assert qr(qmin=0, qmax=255, zp=-1) == E_RANGE
    qn = lambda **k: lib.mctq_quantize_nhwc_i8_padded(k.get("x", 0x7f5000000000), k.get("dt", _native.F32), k.get("N", 1),   # noqa: E731
                                                       k.get("C", 3), 4, 4, k.get("Cp", 4), 1.0, k.get("zp", 0), -128, 127,
                                                       k.get("codes", 0x7f6000000000), None, None)
    assert qn(N=0) == 0
    assert qn(x=None) == E_BADARG and qn(codes=None) == E_BADARG and qn(C=0) == E_BADARG
    assert qn(Cp=2) == E_BADARG and qn(C=5) == E_BADARG and qn(C=17, Cp=24) == E_BADARG
    assert qn(codes=0x7f6000000004) == E_BADARG
    assert qn(dt=5) == E_DTYPE and qn(zp=200) == E_RANGE


# ------------------------------------------------------------------------------------------------ model reports
_ACTS = (torch.nn.ReLU, torch.nn.ReLU6, torch.nn.Hardswish, torch.nn.SiLU)


def mct_style(model):
    """An MCT-style export: every Conv2d / Linear wrapped (int8 weights, per channel), a holder on the model input and a
    holder after every ReLU / ReLU6 / Hardswish / SiLU module."""
    def convert(parent):
        for name, child in list(parent.named_children()):
            if isinstance(child, (torch.nn.Conv2d, torch.nn.Linear)):
                q = Q.WeightsSymmetricInferableQuantizer(8, [1.0] * child.weight.shape[0], True, 0)
                setattr(parent, name, mctq.PytorchQuantizationWrapper(child, {"weight": q}))
            elif isinstance(child, _ACTS):
                h = PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [-1.0], [6.0]))
                setattr(parent, name, torch.nn.Sequential(type(child)(), h))
            else:
                convert(child)
    convert(model)
    holder = PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [-3.0], [3.0]))
    return torch.nn.Sequential(holder, model)


# model: holder-fed groups-1 convs (all of which switch with integer_pad)
_MODELS = {"resnet18": 19, "mobilenet_v2": 18, "mobilenet_v3_large": 16, "mobilenet_v3_small": 12, "efficientnet_b0": 17}
_ROW_REASONS = ("is not a multiple of 16", "is not a multiple of 32")


@pytest.mark.parametrize("name", list(_MODELS))
def test_mct_model_reports(name):
    tv = pytest.importorskip("torchvision")
    build = lambda: _fake_pack_model(mct_style(getattr(tv.models, name)(weights=None).eval()))   # noqa: E731
    before = PW.pack_model_weights(build(), integer_conv=True)
    model = build()
    after = PW.pack_model_weights(model, integer_conv=True, integer_pad=True)
    on = lambda rep: {n for n, r in rep.items() if r["weight"]["integer_conv"]}   # noqa: E731
    refused = {n for n, r in before.items() if any(s in r["weight"]["integer_conv_reason"] for s in _ROW_REASONS)}
    assert refused and on(after) == on(before) | refused
    for n, r in after.items():
        if n not in on(after):
            assert r["weight"]["integer_conv_reason"] == before[n]["weight"]["integer_conv_reason"], n
    g1 = [n for n, r in after.items() if r["weight"]["input_holder"] and isinstance(model.get_submodule(n).layer, torch.nn.Conv2d)
          and model.get_submodule(n).layer.groups == 1]
    assert len(g1) == _MODELS[name] and set(g1) <= on(after)
    # without the flag nothing changes, with integer_linear too
    assert PW.pack_model_weights(build(), integer_conv=True, integer_linear=True) == \
        PW.pack_model_weights(build(), integer_conv=True, integer_linear=True)


# ------------------------------------------------------------------------------------------------ fake implementations
def test_fake_implementations():
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        x = torch.empty(2, 5, 3)
        c, r = torch.ops.mctq.quantize_rows_i8_padded(x, 16, 0.1, 0, -128, 127, True)
        assert c.shape == (2, 5, 16) and c.dtype == torch.int8 and r.shape == (10,)
        x4 = torch.empty(2, 3, 7, 9, dtype=torch.bfloat16)
        c, p = torch.ops.mctq.quantize_nhwc_i8_padded(x4, 4, 0.1, 3, 0, 255, False)
        assert c.shape == (2, 7, 9, 4) and c.dtype == torch.uint8 and p.numel() == 0
        xc = torch.empty(6, 24, dtype=torch.int8)
        y = torch.ops.mctq.packed_linear_i8_padded(xc, 20, 0, None, torch.empty(10 * 24, dtype=torch.int8), I8, True, 10,
                                                   torch.zeros(1, dtype=torch.int32), torch.empty(10, dtype=torch.int32),
                                                   torch.empty(1), None, torch.bfloat16, None)
        assert y.shape == (6, 10) and y.dtype == torch.bfloat16
        y = torch.ops.mctq.packed_linear_i8_padded(xc, 20, 0, None, torch.empty(10 * 24, dtype=torch.uint8), LU8, False, 10,
                                                   None, torch.empty(10, dtype=torch.int32), torch.empty(10), None,
                                                   torch.bfloat16, [1, 2, 3])
        assert y.dtype == torch.float32
        xn = torch.empty(2, 9, 9, 4, dtype=torch.int8)
        y = torch.ops.mctq.packed_conv2d_i8_padded(xn, 3, 0, None, torch.empty(8 * 48, dtype=torch.int8), I8, True, 8, [3, 3],
                                                   [2, 2], [1, 1], [1, 1, 1, 1], torch.zeros(1, dtype=torch.int32),
                                                   torch.empty(8, dtype=torch.int32), torch.empty(1), None, torch.float16,
                                                   True, None)
        assert y.shape == (2, 8, 5, 5) and y.dtype == torch.float16 and y.is_contiguous(memory_format=torch.channels_last)


# ------------------------------------------------------------------------------------------------ GPU: padded quantizers
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", [(1, 1, 1, 1), (3, 3, 7, 9), (2, 4, 33, 17), (1, 6, 5, 5), (2, 8, 3, 3), (1, 10, 9, 9),
                                   (2, 120, 4, 5), (1, 3, 300, 230)])
@pytest.mark.parametrize("qname", ["s8", "u8"])
def test_padded_quantizers(dtype, shape, qname):
    q = {"s8": Q.ActivationSymmetricInferableQuantizer(8, [4.0], True),
         "u8": Q.ActivationUniformInferableQuantizer(8, [-1.3], [2.9])}[qname]
    s, z, qmin, qmax = _launch_args(q)
    x = _special_x(shape, dtype, sum(shape))
    ref = _scalar_codes(x, s, z, qmin, qmax).permute(0, 2, 3, 1).to(torch.int64).cpu()
    C = shape[1]
    cp = ops.conv_code_pitch(C, 1, 1, I8)[0]
    for xin in (x, x.to(memory_format=torch.channels_last)):
        codes, P = ops.quantize_nhwc_i8_padded(xin, cp, s, z, qmin, qmax, True)
        assert codes.shape == shape[:1] + shape[2:] + (cp,) and codes.is_contiguous()
        c = codes.cpu().to(torch.int64)
        assert torch.equal(c[..., :C], ref) and (c[..., C:] == z).all()
        assert torch.equal(P.cpu().to(torch.int64), c.sum(-1).reshape(-1))
    # rows: a [M, K] x into a pitch of K rounded up to 16 (and to 4 for a short row)
    xr = x.reshape(-1, shape[-1])
    for ldc in {ops.linear_code_pitch(xr.shape[1], I8), -(-xr.shape[1] // 4) * 4}:
        codes, rs = torch.ops.mctq.quantize_rows_i8_padded(xr, ldc, s, z, qmin, qmax, True)
        r = _scalar_codes(xr, s, z, qmin, qmax).cpu().to(torch.int64)
        c = codes.cpu().to(torch.int64)
        assert torch.equal(c[:, :xr.shape[1]], r) and (c[:, xr.shape[1]:] == z).all()
        assert torch.equal(rs.cpu().to(torch.int64), c.sum(-1))


@pytest.mark.gpu
def test_padded_quantizer_large_and_canary():
    # N*H*W above 65535 and a canary around the codes
    x = _special_x((2, 3, 200, 190), torch.float32, 5)
    s, z, qmin, qmax = 0.031, 7, -128, 127
    n = 2 * 200 * 190 * 4
    buf = torch.full((n + 64,), 0x5A, dtype=torch.uint8, device="cuda")
    out = buf[32:32 + n]
    P = torch.empty(2 * 200 * 190, dtype=torch.int32, device="cuda")
    rc = _native.load().mctq_quantize_nhwc_i8_padded(x.data_ptr(), _native.F32, 2, 3, 200, 190, 4, s, z, qmin, qmax,
                                                     out.data_ptr(), P.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "mctq_quantize_nhwc_i8_padded")
    assert (buf[:32] == 0x5A).all() and (buf[32 + n:] == 0x5A).all()
    ref = _scalar_codes(x, s, z, qmin, qmax).permute(0, 2, 3, 1)
    c = out.view(torch.int8).reshape(2, 200, 190, 4)
    assert torch.equal(c[..., :3], ref) and (c[..., 3] == z).all()


# ------------------------------------------------------------------------------------------------ GPU: conv and linear
def _weights(g, kind, ws, Cout, inner_shape, lut_no_zero):
    """(int32 codes / indices, zw, scale, lut table or None) of a random weight."""
    if kind in (LI4, LU8):
        n = 16 if kind == LI4 else 256
        table = torch.randint(1, 128, (n,), generator=g) * (torch.randint(0, 2, (n,), generator=g) * 2 - 1)
        if not lut_no_zero:
            table[3] = 0
        idx = torch.randint(0, n, (Cout,) + inner_shape, generator=g, dtype=torch.int32)
        scale = (torch.rand(Cout, generator=g) * 0.02 + 0.001).to(torch.float32)
        return idx, None, scale, table.to(torch.int32).tolist()
    lo, hi = ((-8, 7) if ws else (0, 15)) if kind == I4 else ((-128, 127) if ws else (0, 255))
    qw = torch.randint(lo, hi + 1, (Cout,) + inner_shape, generator=g, dtype=torch.int32)
    zw = torch.randint(lo, hi + 1, (Cout,), generator=g, dtype=torch.int32)
    scale = (torch.rand(Cout, generator=g) * 0.02 + 0.001).to(torch.float32)
    return qw, zw, scale, None


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _conv_pad_case(N, Cin, H, W, Cout, k, stride, dilation, padding, kind, ws, xs, zx, dtype, x_cl, w_cl, seed,
                   lut_no_zero=False, bias=True):
    g = torch.Generator().manual_seed(seed)
    kh, kw = k
    qw, zw, scale, lut = _weights(g, kind, ws, Cout, (Cin, kh, kw), lut_no_zero)
    dtype = torch.float32 if lut else dtype
    ws = ws and not lut
    shape = (Cout, Cin, kh, kw)
    mem = qw.permute(0, 2, 3, 1) if w_cl else qw
    codes = ops.pack_weight_codes(mem.contiguous(), kind, ws).cuda()
    wstride = torch.empty(shape, device="meta").to(memory_format=torch.channels_last if w_cl else torch.contiguous_format).stride()
    xlo, xhi = (-128, 127) if xs else (0, 255)
    x_scale = 0.0371
    conv = ops.IntegerConv2d(codes, kind, ws, dtype, Cout, Cin, k, wstride, stride, dilation, padding, scale.cuda(),
                             zw.cuda() if zw is not None else None, x_scale, zx, xlo, xhi, lut, pad=True)
    x = (torch.randn(N, Cin, H, W, generator=g) * 3).to(dtype).cuda()
    if x_cl:
        x = x.to(memory_format=torch.channels_last)
    b = (torch.randn(Cout, generator=g) * 3).to(dtype).cuda() if bias else None
    y = conv(x, b)
    qx = _scalar_codes(x, x_scale, zx, xlo, xhi).to(torch.int64)
    qv = torch.tensor(lut, dtype=torch.int64)[qw.long()] if lut else qw
    f = (torch.tensor(np.float32(x_scale)) * scale).to(torch.float32)
    ref = conv_reference(qx, zx, qv.cuda().to(torch.int64), (zw if zw is not None else torch.zeros(1, dtype=torch.int32)).cuda(),
                         f.cuda(), b, stride, dilation, padding, dtype)
    assert y.shape == ref.shape
    assert y.is_contiguous(memory_format=torch.channels_last if (x_cl or w_cl) else torch.contiguous_format)
    assert torch.equal(_bits(y), _bits(ref)), f"{(y.float() - ref.float()).abs().max()}"
    # canary around the same kernel's output, written as NCHW planes
    qxp, sx = conv.quantize(x)
    Ho, Wo = conv.output_hw(H, W)
    M = N * Ho * Wo
    canary = torch.full((M * Cout + 64,), float("nan"), dtype=dtype, device="cuda")
    out = canary[32:32 + M * Cout]
    gm = _native.MctqConv2dGeom(N, H, W, Cin, Ho, Wo, kh, kw, *stride, *dilation, *padding)
    rc = _native.load().mctq_packed_conv2d_i8_padded(
        conv._w._desc_ptr, ctypes.addressof(gm), conv.cp, Cout, qxp.data_ptr(), int(xs), zx,
        sx.data_ptr() if sx is not None else None, conv.w_rowsum.data_ptr(), conv.factor.data_ptr(),
        b.data_ptr() if b is not None else None, _TAG[dtype], out.data_ptr(), 1,
        conv._w.lut.ctypes.data if lut else None, torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "mctq_packed_conv2d_i8_padded")
    assert torch.isnan(canary[:32]).all() and torch.isnan(canary[32 + M * Cout:]).all()
    assert torch.equal(_bits(out), _bits(ref).reshape(-1))
    return conv


# (N, H, W, Cout, kernel, stride, dilation, padding (pt, pb, pl, pr))
_GEOMS = [
    (2, 9, 9, 24, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1)),
    (1, 16, 14, 40, (7, 7), (2, 2), (1, 1), (3, 3, 3, 3)),                      # a ResNet-style stem
    (2, 7, 6, 72, (1, 1), (1, 1), (1, 1), (0, 0, 0, 0)),
    (1, 12, 10, 33, (5, 5), (1, 2), (2, 1), (4, 3, 2, 1)),                      # asymmetric, dilated: taps outside every border
    (3, 5, 5, 130, (3, 3), (1, 1), (1, 1), (2, 0, 0, 2)),
]
_PAD_CINS = [1, 2, 3, 4, 5, 6, 8, 10, 20, 24, 28, 40, 72, 88, 120, 200]
_PAD_CONFIGS = [(kind, ws, xs, zx) for kind in (I8, I4, LI4, LU8) for ws, xs, zx in
                ((True, True, 0), (False, True, -7), (True, False, 128), (False, False, 0))]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ci", range(len(_PAD_CONFIGS)))
def test_conv_padded_bit_exact(ci, dtype):
    kind, ws, xs, zx = _PAD_CONFIGS[ci]
    if kind in (LI4, LU8) and dtype != torch.float32:
        pytest.skip("LUT weights rebuild as f32")
    for j, cin in enumerate(_PAD_CINS):
        N, H, W, Cout, k, st, dil, pad = _GEOMS[(ci + j) % len(_GEOMS)]
        _conv_pad_case(N, cin, H, W, Cout, k, st, dil, pad, kind, ws, xs, zx, dtype, x_cl=(ci + j) % 3 == 0,
                       w_cl=(ci + j) % 4 == 1, seed=100 * ci + j, lut_no_zero=j % 2 == 0, bias=j % 3 != 2)


@pytest.mark.gpu
def test_conv_padded_split_k_and_large_m():
    # split-K of 8: a small M with a long padded row; and M = 64 * 112 * 112 (a stem at batch 64) as many row tiles
    c = _conv_pad_case(1, 200, 4, 4, 128, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), I8, True, True, 3, torch.float32, False,
                       False, 1)
    assert c.cp == 208
    c = _conv_pad_case(64, 3, 224, 224, 32, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1), I8, True, False, 5, torch.bfloat16, True,
                       False, 2)
    assert c.cp == 4
    c = _conv_pad_case(2, 6, 40, 40, 64, (1, 1), (1, 1), (1, 1), (0, 0, 0, 0), I4, True, True, -3, torch.float16, False,
                       True, 3)
    assert c.cp == 8


def _lin_pad_case(M, K, N, kind, ws, xs, zx, dtype, seed, bias=True):
    g = torch.Generator().manual_seed(seed)
    qw, zw, scale, lut = _weights(g, kind, ws, N, (K,), seed % 2 == 0)
    dtype = torch.float32 if lut else dtype
    ws = ws and not lut
    codes = ops.pack_weight_codes(qw, kind, ws).cuda()
    xlo, xhi = (-128, 127) if xs else (0, 255)
    x_scale = 0.0213
    lin = ops.IntegerLinear(codes, kind, ws, dtype, N, K, scale.cuda(), zw.cuda() if zw is not None else None, x_scale, zx,
                            xlo, xhi, lut, pad=True)
    assert lin.ldc == ops.linear_code_pitch(K, kind)
    x = (torch.randn(M, K, generator=g) * 3).to(dtype).cuda()
    b = (torch.randn(N, generator=g) * 3).to(dtype).cuda() if bias else None
    y = lin(x, b)
    qx = _scalar_codes(x, x_scale, zx, xlo, xhi).to(torch.int64)
    qv = torch.tensor(lut, dtype=torch.int64)[qw.long()] if lut else qw
    f = (torch.tensor(np.float32(x_scale)) * scale).to(torch.float32)
    ref = conv_reference(qx[:, :, None, None], zx, qv.cuda().to(torch.int64)[:, :, None, None],
                         (zw if zw is not None else torch.zeros(1, dtype=torch.int32)).cuda(), f.cuda(), b, (1, 1), (1, 1),
                         (0, 0, 0, 0), dtype)[:, :, 0, 0]
    assert torch.equal(_bits(y), _bits(ref)), f"{(y.float() - ref.float()).abs().max()}"
    # canary: rows written into a wider buffer through `out`
    canary = torch.full((M, N + 8), float("nan"), dtype=dtype, device="cuda")
    qxp, rs = lin.quantize(x)
    lin.gemm(qxp, rs, b, out=canary[:, 4:4 + N])
    assert torch.isnan(canary[:, :4]).all() and torch.isnan(canary[:, 4 + N:]).all()
    assert torch.equal(_bits(canary[:, 4:4 + N]), _bits(ref))
    # the torch op over the same codes
    zp = zw.cuda() if zw is not None else None
    y2 = torch.ops.mctq.packed_linear_i8_padded(qxp, K, zx, rs if lin.needs_x_rowsum else None, lin._keep[0], kind, ws, N,
                                                zp, lin.w_rowsum, lin.factor, b, dtype, lut)
    assert torch.equal(_bits(y2), _bits(ref))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ci", range(len(_PAD_CONFIGS)))
def test_linear_padded_bit_exact(ci, dtype):
    kind, ws, xs, zx = _PAD_CONFIGS[ci]
    if kind in (LI4, LU8) and dtype != torch.float32:
        pytest.skip("LUT weights rebuild as f32")
    for j, K in enumerate((1, 3, 24, 40, 440, 1000)):
        for M in (1, 8, 256):
            _lin_pad_case(M, K, 72 + 8 * j, kind, ws, xs, zx, dtype, seed=1000 * ci + 10 * j + M, bias=M != 8)


@pytest.mark.gpu
def test_linear_padded_large_m():
    _lin_pad_case(65537, 40, 32, I8, True, False, 9, torch.bfloat16, 7)
    _lin_pad_case(65600, 3, 16, LI4, False, True, -5, torch.float32, 8)


@pytest.mark.gpu
def test_conv_padded_torch_op():
    conv = _conv_pad_case(2, 5, 9, 9, 16, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), I8, True, True, 2, torch.float32, False,
                          False, 9)
    x = torch.randn(2, 5, 9, 9, device="cuda")
    qx, sx = conv.quantize(x)
    ref = conv.gemm(qx, sx, None)
    y = torch.ops.mctq.packed_conv2d_i8_padded(qx, 5, 2, sx, conv._w._keep[0], I8, True, 16, [3, 3], [1, 1], [1, 1],
                                               [1, 1, 1, 1], conv._w._keep[2], conv.w_rowsum, conv.factor, None,
                                               torch.float32, False, None)
    assert torch.equal(y, ref)
    c2, p2 = torch.ops.mctq.quantize_nhwc_i8_padded(x, 8, conv.x_scale, 2, -128, 127, True)
    assert c2.shape == (2, 9, 9, 8) and torch.equal(c2[..., :5], qx[..., :5])


# ------------------------------------------------------------------------------------------------ GPU: module level
class _PadNet(torch.nn.Module):
    """holder -> stem Conv 3 -> 24 (3x3 s2) -> holder -> Conv 24 -> 10 (1x1) -> holder -> Conv 10 -> 6 (3x3) -> holder ->
    flatten -> Linear 150 -> 20: every layer off the granule."""

    def __init__(self, dtype, wq_kind):
        super().__init__()
        wq = (lambda C: Q.WeightsSymmetricInferableQuantizer(4, [0.5] * C, True, 0)) if wq_kind == "i4" else \
            (lambda C: Q.WeightsUniformInferableQuantizer(8, [-0.3] * C, [0.2] * C, True, 0))
        hq = lambda: PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [-1.7], [2.3]))  # noqa: E731
        self.h0, self.h1, self.h2, self.h3 = hq(), hq(), hq(), hq()
        self.c0 = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(3, 24, 3, stride=2, padding=1), {"weight": wq(24)})
        self.c1 = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(24, 10, 1), {"weight": wq(10)})
        self.c2 = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(10, 6, 3, padding=1, bias=False), {"weight": wq(6)})
        self.fc = mctq.PytorchQuantizationWrapper(torch.nn.Linear(150, 20), {"weight": wq(20)})
        self.to(dtype).cuda()

    def forward(self, x):
        a = self.c2(self.h2(self.c1(self.h1(self.c0(self.h0(x))))))
        return self.fc(torch.flatten(self.h3(a), 1))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("wq_kind", ["i8", "i4"])
def test_module_switch(dtype, wq_kind):
    torch.manual_seed(0)
    model = _PadNet(dtype, wq_kind)
    x = (torch.randn(3, 3, 10, 10, device="cuda") * 1.5).to(dtype)
    with torch.no_grad(), _no_tf32():
        packed = copy.deepcopy(model)
        PW.pack_model_weights(packed)
        plain = copy.deepcopy(packed)
        rep0 = PW.pack_model_weights(copy.deepcopy(model), integer_conv=True, integer_linear=True)
        assert not any(r["weight"]["integer_conv"] or r["weight"]["integer"] for r in rep0.values())
        report = PW.pack_model_weights(model, integer_conv=True, integer_linear=True, integer_pad=True)
        for name in ("c0", "c1", "c2"):
            assert report[name]["weight"]["integer_conv"], report[name]
        assert report["fc"]["weight"]["integer"], report["fc"]
        # each switched layer against the packed layer on the same input: the f64 tolerance of the integer tests
        h0 = model.h0(x)
        a0 = model.c0(h0)
        r0 = plain.c0(h0)
        tol = 2e-2 if dtype != torch.float32 else 1e-4
        assert torch.allclose(a0.float(), r0.float(), atol=tol * float(r0.abs().max()), rtol=0)
        h = model.h3(model.c2(model.h2(model.c1(model.h1(a0)))))
        yf = model.fc(torch.flatten(h, 1))
        rf = plain.fc(torch.flatten(h, 1))
        assert torch.allclose(yf.float(), rf.float(), atol=tol * float(rf.abs().max()), rtol=0)
        y = model(x)
        assert torch.equal(_bits(model(x)), _bits(y))
        assert set(model.state_dict()) == set(packed.state_dict())
        buf = io.BytesIO()
        torch.save(model, buf)
        buf.seek(0)
        m2 = torch.load(buf, weights_only=False)
        assert m2.c0._packed.integer and torch.equal(_bits(m2(x)), _bits(y))
        m3 = copy.deepcopy(model)
        m3.load_state_dict(model.state_dict())
        assert torch.equal(_bits(m3(x)), _bits(y))
        m4 = copy.deepcopy(model).to("cpu").to("cuda")
        assert torch.equal(_bits(m4(x)), _bits(y))
        assert pickle.loads(pickle.dumps(model.c0._packed)).integer
    # fallbacks: autograd recording and an unbatched input take the packed path
    y_grad = model.c0(h0.clone().requires_grad_(True))
    assert y_grad.requires_grad
    with torch.no_grad():
        assert model.c0(h0[0]).dim() == 3
    _graph_equals_eager(model, x)


def _graph_equals_eager(model, x):
    with torch.no_grad():
        y = model(x)
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
    assert torch.equal(_bits(y_g), _bits(y))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["efficientnet_b0", "mobilenet_v3_large"])
def test_mct_models_graph_replay(name):
    tv = pytest.importorskip("torchvision")
    torch.manual_seed(0)
    model = mct_style(getattr(tv.models, name)(weights=None).eval()).cuda()
    reports = PW.pack_model_weights(model, integer_linear=True, integer_conv=True, integer_lut=True,
                                    integer_depthwise=True, integer_pad=True)
    switched = sum(bool(r["weight"].get("integer_conv")) for r in reports.values())
    g1 = sum(1 for n, r in reports.items() if r["weight"]["input_holder"] and model.get_submodule(n).layer.__class__ is
             torch.nn.Conv2d and model.get_submodule(n).layer.groups == 1)
    assert g1 == _MODELS[name] and switched >= g1
    x = torch.randn(2, 3, 96, 96, device="cuda")
    with torch.no_grad():
        y1, y2 = model(x), model(x)
    assert torch.isfinite(y1).all() and torch.equal(_bits(y1), _bits(y2))
    _graph_equals_eager(model, x)
