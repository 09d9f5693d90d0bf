"""Integer linear and convolution modes for LUT weights: mctq_packed_linear_i8_lut / mctq_packed_conv2d_i8_lut
(csrc/mctq_packed_igemm.cu) and `integer_lut=True` of the packed wrappers (pytorch/packed_weights.py).  Every GPU result is
checked bit for bit against the exact integer formula of include/mctq.h with qw = lut[idx] and zw = 0."""
import copy
import ctypes
import io
import pickle
import warnings

import numpy as np
import pytest
import torch

import mct_quantizers_b200 as mctq
from mct_quantizers_b200 import _native, ops
from mct_quantizers_b200.pytorch import packed_weights as PW
from mct_quantizers_b200.pytorch import quantizers as Q
from mct_quantizers_b200.pytorch.activation_quantization_holder import PytorchActivationQuantizationHolder
from mct_quantizers_b200.pytorch.packed_weights import integer_conv_eligibility, integer_linear_eligibility

from test_integer_conv import _conv_wrapper, _fake_packed_conv, _no_tf32, conv_reference
from test_integer_linear import _Net, reference, reference_on_device
from test_packed_linear import _fake_packed, _lin_desc

I8, I4, LU8, LI4 = _native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4, _native.PACK_LUT_U8, _native.PACK_LUT_I4
E_BADARG, E_DTYPE, E_RANGE, E_LUT = -1, -2, -3, -4
TABLE = (ctypes.c_int8 * 256)(*range(-128, 128))


# ------------------------------------------------------------------------------------------------ integer reference
def lut_reference(qx, zx, idx, lut, f, bias):
    """The formula with qw = lut[idx], zw = 0, in numpy (reference() of the affine modes)."""
    qw = np.asarray(lut, np.int64)[np.asarray(idx, np.int64)]
    return reference(qx, zx, qw, 0, f, bias, torch.float32)


def test_reference_hand_worked():
    # lut = [-3, 5]; idx = [[1, 0], [0, 0]] -> qw = [[5, -3], [-3, -3]]; qx = [[2, 4]], zx = 1 -> (qx - zx) = [1, 3]
    # c = [5 - 9, -3 - 9] = [-4, -12]; f = [0.5, 0.25], bias = [1, 0]  ->  y = [-1, -3]
    y = lut_reference([[2, 4]], 1, [[1, 0], [0, 0]], [-3, 5], [0.5, 0.25], [1.0, 0.0])
    assert y.tolist() == [[-1.0, -3.0]]
    # c = acc - zx * Sw: acc = 1 + 1 = 2 and Sw = lut[1] + lut[1] = 2 for idx [[1, 1]], zx = -4  ->  c = 2 + 4 * 2 = 10
    assert lut_reference([[1, 1]], -4, [[1, 1]], [7, 1], [1.0], None).item() == 10.0


# ------------------------------------------------------------------------------------------------ C-ABI rejections
def _lcall(d, out_f=10, in_f=64, xq=0x7f5000000000, x_signed=1, zx=0, M=1, w_rowsum=0x7f6100000000, factor=0x7f6200000000,
           y_dtype=_native.F32, y=0x7f6000000000, table=TABLE):
    lib = _native.load()
    return lib.mctq_packed_linear_i8_lut(ctypes.byref(d) if d is not None else None, out_f, in_f, xq, x_signed, zx, M, None,
                                         w_rowsum, factor, None, y_dtype, y, out_f, table, None)


def _ccall(d, Cout=10, x_signed=1, zx=0, table=TABLE, **g):
    from test_integer_conv import _geom
    lib = _native.load()
    geo = _geom(**{**dict(Cin=32, kh=3, kw=3), **g})
    return lib.mctq_packed_conv2d_i8_lut(ctypes.byref(d) if d is not None else None, ctypes.byref(geo), Cout, 0x7f5000000000,
                                         x_signed, zx, None, 0x7f6100000000, 0x7f6200000000, None, _native.F32,
                                         0x7f6000000000, 1, table, None)


@pytest.mark.parametrize("kind", [LI4, LU8])
def test_c_abi_rejections(kind):
    """Every check runs before any CUDA call (the pointers are never touched): no GPU needed."""
    d = lambda **k: _lin_desc(out_f=10, in_f=k.pop("in_f", 64), kind=k.pop("kind", kind), **k)     # noqa: E731
    K = 32 * 9
    dc = lambda **k: _lin_desc(out_f=10, in_f=K, kind=k.pop("kind", kind), **k)                    # noqa: E731
    for call, desc in ((_lcall, d), (_ccall, dc)):
        assert call(None) == E_BADARG
        assert call(desc(kind=I8)) == E_BADARG and call(desc(kind=I4)) == E_BADARG       # affine kinds
        assert call(desc(), table=None) == E_BADARG                                     # no table
        assert call(desc(K=0)) == E_LUT and call(desc(K=17 if kind == LI4 else 257)) == E_LUT
        assert call(desc(dtype=_native.BF16)) == E_DTYPE                                # LUT weights rebuild as f32
        misaligned = desc()
        misaligned.codes = 0x7f0000000004
        assert call(misaligned) == E_BADARG
        assert call(desc(), x_signed=1, zx=128) == E_RANGE
    assert _lcall(d(), M=0) == 0 and _ccall(dc(), N=0) == 0
    # the existing entry points keep rejecting LUT kinds
    from test_integer_linear import _call
    assert _call(d()) == E_BADARG
    # row length: a multiple of 32 (4-bit indices) or 16 (8-bit indices)
    assert _lcall(d(in_f=48), in_f=48, M=0) == (E_BADARG if kind == LI4 else 0)
    assert _lcall(d(in_f=40), in_f=40, M=0) == E_BADARG
    assert _ccall(_lin_desc(out_f=10, in_f=16, kind=kind), Cin=16, kh=1, kw=1, N=0) == (E_BADARG if kind == LI4 else 0)
    # K over the signed-weight bound of the x signedness, whatever the descriptor's is_signed says
    for xs, bound in ((1, 131071), (0, 65793)):
        top = bound // 32 * 32
        for signed in (0, 1):
            dd = d(in_f=top + 32)
            dd.is_signed = signed
            assert _lcall(dd, out_f=10, in_f=top + 32, x_signed=xs) == E_RANGE
            dd = d(in_f=top)
            dd.is_signed = signed
            assert _lcall(dd, in_f=top, x_signed=xs, M=0) == 0
        cin = top // 16 * 16
        assert _ccall(_lin_desc(out_f=10, in_f=cin + 32, kind=kind), Cin=cin + 32, kh=1, kw=1, x_signed=xs) == E_RANGE


def test_code_values_of_lut_indices():
    idx = torch.arange(16, dtype=torch.int32).repeat(3).reshape(3, 16)             # every nibble, unsigned
    codes = ops.pack_weight_codes(idx, LI4, False)
    assert codes.numel() == 24 and codes[0].item() == 0x10 and codes[7].item() == 0xFE
    assert torch.equal(ops.weight_code_values(codes, LI4, False, 3, 16), idx)
    idx8 = torch.arange(256, dtype=torch.int32).reshape(4, 64)
    assert torch.equal(ops.weight_code_values(ops.pack_weight_codes(idx8, LU8, False), LU8, False, 4, 64), idx8)
    # the (r, s, c) reorder of a contiguous conv weight works on indices too
    g = torch.Generator().manual_seed(0)
    for kind, hi in ((LI4, 16), (LU8, 256)):
        w = torch.randint(0, hi, (5, 32, 3, 2), generator=g, dtype=torch.int32)
        rsc = ops.conv_codes_rsc(ops.pack_weight_codes(w, kind, False), kind, False, 5, 32, 3, 2)
        assert torch.equal(ops.weight_code_values(rsc, kind, False, 5, 32 * 6), w.permute(0, 2, 3, 1).reshape(5, -1))


def test_lut_code_table():
    assert ops.lut_code_table(LI4, torch.tensor([-128.0, 127.0]), "t").tolist() == [-128, 127]
    for bad in ([0.5], [128.0], list(range(17))):
        with pytest.raises(ValueError):
            ops.lut_code_table(LI4, bad, "t")
    with pytest.raises(ValueError, match="not a LUT"):
        ops.lut_code_table(I8, [1], "t")


# ------------------------------------------------------------------------------------------------ eligibility and reports
def _act(signed=True):
    return Q.ActivationSymmetricInferableQuantizer(8, [4.0], signed)


def _lut_q(C, K=16, bw=8, pot=False, thr=None, lut=None, rank=2):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        lut = lut if lut is not None else [float(v) for v in np.linspace(-2 ** (bw - 1), 2 ** (bw - 1) - 1, K).round()]
        nb = max(1, int(np.ceil(np.log2(K))))
        if pot:
            thr = thr if thr is not None else [2.0 ** -(c % 3) for c in range(C)]
            return Q.WeightsLUTPOTInferableQuantizer(nb, lut, thr, True, 0, rank, bw)
        thr = thr if thr is not None else [0.02 + 0.0001 * (c % 97) for c in range(C)]
        return Q.WeightsLUTSymmetricInferableQuantizer(nb, lut, thr, True, 0, rank, bw)


def _lut_lin(in_f=64, out_f=8, kind=LI4, **k):
    w = mctq.PytorchQuantizationWrapper(torch.nn.Linear(in_f, out_f), {"weight": _lut_q(out_f, 16 if kind == LI4 else 64, **k)})
    _fake_packed(w)
    w._packed.entries[0].kind, w._packed.entries[0].is_signed = kind, False
    return w


def _lut_conv(cin=32, cout=8, k=3, kind=LI4, **q):
    w = _conv_wrapper(cin=cin, cout=cout, k=k)
    w.weights_quantizers["weight"] = _lut_q(cout, 16 if kind == LI4 else 64, rank=4, **q)
    _fake_packed_conv(w, kind=kind)
    w._packed.entries[0].quantizer = w.weights_quantizers["weight"]
    w._packed.entries[0].is_signed = False
    return w


@pytest.mark.parametrize("kind", [LI4, LU8])
def test_eligibility(kind):
    q = _act()
    for elig, mk, what in ((integer_linear_eligibility, _lut_lin, "in_features"),
                           (integer_conv_eligibility, _lut_conv, "Cin * kh * kw")):
        # without lut=True: today's reasons, word for word
        assert elig(mk(kind=kind), q) == (False, f"the weight is packed as {PW._KIND_NAMES[kind]}, not as int8 / int4 "
                                                 f"affine codes")
        assert elig(mk(kind=kind), q, lut=True) == (True, "")
        assert elig(mk(kind=kind, pot=True), q, lut=True) == (True, "")
        ok, why = elig(mk(kind=kind, bw=9, lut=[-200.0, 0.0, 3.0]), q, lut=True)
        assert not ok and why.startswith("a LUT value is not an integer in [-128, 127]")
        ok, why = elig(mk(kind=kind, thr=[2.0 ** -126] * 8), q, lut=True)                  # sw = 2^-133: subnormal
        assert not ok and why.startswith("a threshold times 2^-(lut_values_bitwidth - 1) is not exact and normal")
        assert elig(mk(kind=kind), _act(signed=False), lut=True) == (True, "")
    ok, why = integer_linear_eligibility(_lut_lin(in_f=48, kind=kind), q, lut=True)
    assert (ok, why) == ((False, "in_features = 48 is not a multiple of 32 (4-bit LUT indices)") if kind == LI4 else (True, ""))
    ok, why = integer_linear_eligibility(_lut_lin(in_f=40, kind=kind), q, lut=True)
    assert not ok and why.startswith("in_features = 40 is not a multiple of")
    ok, why = integer_conv_eligibility(_lut_conv(cin=16, k=1, kind=kind), q, lut=True)
    assert (ok, why) == ((False, "Cin * kh * kw = 16 is not a multiple of 32 (4-bit LUT indices)") if kind == LI4 else (True, ""))
    # the signed-weight bound of the x signedness
    ok, why = integer_linear_eligibility(_lut_lin(in_f=65824, out_f=1, kind=kind), _act(signed=False), lut=True)
    assert not ok and "exceeds 65793" in why
    assert integer_linear_eligibility(_lut_lin(in_f=65824, out_f=1, kind=kind), _act(signed=True), lut=True)[0]
    # input-quantizer reasons come first, as for affine weights
    lutq = Q.ActivationLutPOTInferableQuantizer(8, [-2.0, 0.0, 1.0, 3.0], [4.0], True)
    assert "per-tensor affine" in integer_linear_eligibility(_lut_lin(kind=kind), lutq, lut=True)[1]


def test_integer_lut_alone_raises():
    with pytest.raises(ValueError, match="integer_lut=True needs"):
        PW.pack_wrapper_weights(_lut_lin(), integer_lut=True)
    with pytest.raises(ValueError, match="integer_lut=True needs"):
        PW.pack_model_weights(torch.nn.Sequential(), integer_lut=True)
    with pytest.raises(ValueError, match="integer_lut=True needs"):
        _lut_lin().pack_weights(integer_lut=True)


def _mlp_net():
    H = lambda: PytorchActivationQuantizationHolder(_act())                         # noqa: E731
    return _Net([H(), H()], [_lut_lin(64, 96), _lut_lin(96, 32, kind=LU8), _lut_lin(48, 8)],
                lambda m, x: m.w[1](m.h[1](m.w[0](m.h[0](x)))) + m.w[2](x[..., :48]).sum())


def test_model_reports_without_a_gpu():
    net = _mlp_net()
    reports = PW.pack_model_weights(net, integer_linear=True, integer_conv=True, integer_lut=True)
    r0, r1, r2 = (reports[f"w.{i}"]["weight"] for i in range(3))
    assert (r0["integer"], r0["integer_reason"], r0["input_holder"]) == (True, "", "h.0")
    assert (r1["integer"], r1["integer_reason"], r1["input_holder"]) == (True, "", "h.1")
    assert r0["integer_conv"] is False and r0["integer_conv_reason"] == "the layer is Linear, not torch.nn.Conv2d"
    assert r2["integer"] is False and "not the output of an activation quantization holder" in r2["integer_reason"]
    assert net.w[0]._packed.integer and net.w[1]._packed.integer and not net.w[2]._packed.integer
    # without integer_lut: the LUT reason of today, nothing switched
    net = _mlp_net()
    r = PW.pack_model_weights(net, integer_linear=True)["w.0"]["weight"]
    assert r["integer"] is False and r["integer_reason"] == "the weight is packed as lut_i4, not as int8 / int4 affine codes"
    assert not net.w[0]._packed.integer


def lut_quantize_model(model):
    """Wrap every Conv2d / Linear of a torchvision model with a 4-bit LUT POT weight quantizer (16 integer centroids on an
    8-bit grid, per-channel power-of-two thresholds) and put an 8-bit holder behind every ReLU."""
    def convert(parent):
        for name, child in list(parent.named_children()):
            if isinstance(child, (torch.nn.Conv2d, torch.nn.Linear)):
                w = child.weight.detach()
                thr = [2.0 ** float(np.ceil(np.log2(max(float(t), 1e-6)))) for t in w.abs().reshape(w.shape[0], -1).amax(1)]
                setattr(parent, name, mctq.PytorchQuantizationWrapper(child, {"weight": _lut_q(w.shape[0], pot=True, thr=thr, rank=w.dim())}))
            elif isinstance(child, (torch.nn.ReLU, torch.nn.ReLU6)):
                holder = PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [0.0], [4.0]))
                setattr(parent, name, torch.nn.Sequential(type(child)(inplace=False), holder))
            else:
                convert(child)
    convert(model)
    return model


def test_resnet18_lut_reports_without_a_gpu():
    tv = pytest.importorskip("torchvision")
    from mct_quantizers_b200.pytorch.quantize_wrapper import PytorchQuantizationWrapper
    model = lut_quantize_model(tv.models.resnet18())
    for m in model.modules():
        if isinstance(m, PytorchQuantizationWrapper):
            if isinstance(m.layer, torch.nn.Conv2d):
                _fake_packed_conv(m, kind=LI4)
            else:
                _fake_packed(m)
                m._packed.entries[0].kind = LI4
            m._packed.entries[0].quantizer, m._packed.entries[0].is_signed = m.weights_quantizers["weight"], False
    reports = PW.pack_model_weights(model, integer_linear=True, integer_conv=True, integer_lut=True)
    switched = {n for n, r in reports.items() if r["weight"]["integer_conv"]}
    # as with int8 weights: every block conv and downsample conv reads a ReLU holder, except the stem and layer1.0.conv1
    assert len(switched) == 18 and "layer2.0.downsample.0" in switched and "layer1.0.conv2" in switched
    assert reports["fc"]["weight"]["integer"] is False
    assert reports["conv1"]["weight"]["integer_conv"] is False


# ------------------------------------------------------------------------------------------------ GPU: the GEMM
def _table(kind, g, K=None):
    K = K or (16 if kind == LI4 else 200)
    return torch.randint(-128, 128, (K,), generator=g, dtype=torch.int32)


def _sw(C, pot, g, bw=8):
    thr = (2.0 ** -torch.randint(0, 6, (C,), generator=g)).float() if pot else (torch.rand(C, generator=g) * 0.5 + 0.01)
    return thr.float() * 2.0 ** -(bw - 1)


def _lin_case(M, N, K, kind, per_channel, pot, x_signed, zx, with_bias, seed, lut=None, idx=None, qx=None):
    g = torch.Generator().manual_seed(seed)
    lut = _table(kind, g) if lut is None else lut
    idx = torch.randint(0, lut.numel(), (N, K), generator=g, dtype=torch.int32) if idx is None else idx
    sw = _sw(N if per_channel else 1, pot, g)
    xlo, xhi = (-128, 127) if x_signed else (0, 255)
    qx = torch.randint(xlo, xhi + 1, (M, K), generator=g, dtype=torch.int32) if qx is None else qx
    xq = qx.to(torch.int8 if x_signed else torch.uint8).cuda()
    x_scale = 0.0371
    f = (torch.tensor(np.float32(x_scale)) * sw).float()
    bias = (torch.randn(N, generator=g) * 3).cuda() if with_bias else None
    codes = ops.pack_weight_codes(idx, kind, False).cuda()
    lin = ops.IntegerLinear.from_parts(codes, kind, False, torch.float32, N, K, f.cuda(), None, None, zx,
                                       lut_values=lut.tolist())
    assert torch.equal(lin.w_rowsum.cpu(), lut[idx.long()].sum(1).int())
    poison = torch.full((M, N + 9), float("nan"), device="cuda")
    y = lin.gemm(xq, None, bias, out=poison[:, 3:3 + N])
    y2 = lin.gemm(xq, None, bias)
    ref = reference_on_device(qx.cuda(), zx, lut.cuda()[idx.cuda().long()], torch.zeros(1, device="cuda"), f.cuda(), bias,
                              torch.float32)
    assert torch.equal(y.view(torch.int32), ref.view(torch.int32)), f"{(y - ref).abs().max()}"
    assert torch.equal(y2.view(torch.int32), y.view(torch.int32))                     # a second call: the same bits
    assert torch.isnan(poison[:, :3]).all() and torch.isnan(poison[:, 3 + N:]).all()   # nothing outside the view
    return lin


_SHAPES = [(1, 128, 32), (2, 127, 64), (15, 129, 160), (16, 1, 4096), (17, 128, 4096), (255, 300, 160), (256, 129, 32),
           (257, 127, 4096), (1, 11008, 4096), (64, 4096, 11008), (1024, 11008, 160)]
_CONFIGS = [(kind, pot, xs, zx) for kind in (LI4, LU8) for pot in (False, True) for xs, zx in ((True, 0), (True, -7),
                                                                                                (False, 0), (False, 128))]


@pytest.mark.gpu
@pytest.mark.parametrize("ci", range(len(_CONFIGS)))
def test_gemm_bit_exact(ci):
    kind, pot, xs, zx = _CONFIGS[ci]
    for si in range(ci % 2, len(_SHAPES), 2):
        M, N, K = _SHAPES[si]
        _lin_case(M, N, K, kind, per_channel=(si + ci) % 2 == 0, pot=pot, x_signed=xs, zx=zx, with_bias=si % 2 == 1,
                  seed=100 * ci + si)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [LI4, LU8])
def test_gemm_edges(kind):
    # M > 65535 row tiles' worth of rows in one launch range, tail rows and columns
    _lin_case(70001, 33, 64, kind, True, False, True, 5, True, 1)
    # split-K: N = 128, M = 16, K = 4096 runs as clusters of 8 CTAs; N = 11008, M = 1024 as single CTAs
    _lin_case(16, 128, 4096, kind, True, True, True, 3, True, 2)
    _lin_case(1024, 11008, 256, kind, False, False, False, 9, False, 3)
    # K at the bound of s8 x and of u8 x, every product at its extreme: -128 * -128 and 255 * -128
    lut = torch.tensor([-128] + [0] * (15 if kind == LI4 else 99), dtype=torch.int32)
    K = 131071 // 32 * 32
    _lin_case(3, 129, K, kind, False, True, True, 0, False, 4, lut=lut, idx=torch.zeros(129, K, dtype=torch.int32),
              qx=torch.full((3, K), -128, dtype=torch.int32))
    K = 65793 // 32 * 32
    _lin_case(5, 130, K, kind, True, False, False, 0, True, 5, lut=lut, idx=torch.zeros(130, K, dtype=torch.int32),
              qx=torch.full((5, K), 255, dtype=torch.int32))


def _conv_case(N, Cin, H, W, Cout, k, stride, dilation, padding, kind, per_channel, pot, x_signed, zx, channels_last, seed):
    g = torch.Generator().manual_seed(seed)
    kh, kw = k
    lut = _table(kind, g)
    idx = torch.randint(0, lut.numel(), (Cout, Cin, kh, kw), generator=g, dtype=torch.int32)
    sw = _sw(Cout if per_channel else 1, pot, g)
    xlo, xhi = (-128, 127) if x_signed else (0, 255)
    qx = torch.randint(xlo, xhi + 1, (N, Cin, H, W), generator=g, dtype=torch.int32)
    f = (torch.tensor(np.float32(0.0371)) * sw).float()
    bias = (torch.randn(Cout, generator=g) * 3).cuda() if seed % 2 else None
    codes = ops.pack_weight_codes(idx.permute(0, 2, 3, 1).contiguous(), kind, False).cuda()
    conv = ops.IntegerConv2d.from_parts(codes, kind, False, torch.float32, Cout, Cin, k, stride, dilation, padding,
                                        f.cuda(), None, None, zx, lut_values=lut)
    xq = qx.permute(0, 2, 3, 1).contiguous().to(torch.int8 if x_signed else torch.uint8).cuda()
    ref = conv_reference(qx.cuda(), zx, lut.cuda()[idx.cuda().long()], torch.zeros(1, device="cuda"), f.cuda(), bias,
                         stride, dilation, padding, torch.float32)
    y = conv.gemm(xq, None, bias, channels_last=channels_last)
    assert y.shape == ref.shape
    assert y.is_contiguous(memory_format=torch.channels_last if channels_last else torch.contiguous_format)
    assert torch.equal(y.contiguous().view(torch.int32), ref.contiguous().view(torch.int32)), f"{(y - ref).abs().max()}"
    # canary: the same call into the middle of a NaN buffer
    Ho, Wo = conv.output_hw(H, W)
    M = N * Ho * Wo
    canary = torch.full((M * Cout + 64,), float("nan"), device="cuda")
    out = canary[32:32 + M * Cout]
    geo = _native.MctqConv2dGeom(N, H, W, Cin, Ho, Wo, kh, kw, *stride, *dilation, *padding)
    rc = _native.load().mctq_packed_conv2d_i8_lut(
        conv._w._desc_ptr, ctypes.addressof(geo), Cout, xq.data_ptr(), int(x_signed), zx, None, conv.w_rowsum.data_ptr(),
        conv.factor.data_ptr(), bias.data_ptr() if bias is not None else None, _native.F32, out.data_ptr(),
        0 if channels_last else 1, conv._w.lut.ctypes.data, torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "mctq_packed_conv2d_i8_lut")
    assert torch.isnan(canary[:32]).all() and torch.isnan(canary[32 + M * Cout:]).all()
    assert torch.equal(out, (y.permute(0, 2, 3, 1) if channels_last else y).reshape(-1))


_CONV_SHAPES = [
    (1, 32, 5, 5, 8, (1, 1), (1, 1), (1, 1), (0, 0, 0, 0)),
    (2, 32, 9, 7, 130, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1)),
    (3, 32, 11, 13, 64, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1)),
    (1, 48, 12, 10, 40, (5, 5), (1, 2), (2, 1), (4, 3, 2, 1)),                      # asymmetric, dilated
    (2, 32, 15, 15, 96, (7, 7), (2, 2), (1, 1), (3, 3, 3, 3)),
    (1, 32, 10, 9, 33, (2, 4), (1, 1), (2, 2), (2, 0, 0, 2)),
    (1, 256, 7, 7, 512, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1)),                       # split-K clusters
    (64, 64, 8, 8, 64, (1, 1), (2, 2), (1, 1), (0, 0, 0, 0)),                         # strided 1x1 (downsample)
    (8, 32, 33, 31, 200, (6, 6), (3, 2), (1, 1), (2, 3, 1, 0)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("ci", range(len(_CONFIGS)))
def test_conv_bit_exact(ci):
    kind, pot, xs, zx = _CONFIGS[ci]
    for si in range(ci % 2, len(_CONV_SHAPES), 2):
        N, Cin, H, W, Cout, k, st, dil, pad = _CONV_SHAPES[si]
        if kind == LI4 and (Cin * k[0] * k[1]) % 32:                          # 4-bit indices: K % 32 == 0
            Cin = 32
        _conv_case(N, Cin, H, W, Cout, k, st, dil, pad, kind, per_channel=(si + ci) % 2 == 0, pot=pot, x_signed=xs, zx=zx,
                   channels_last=(si + ci) % 4 < 2, seed=100 * ci + si)


@pytest.mark.gpu
def test_torch_ops():
    g = torch.Generator().manual_seed(3)
    lut = _table(LI4, g)
    idx = torch.randint(0, 16, (64, 64), generator=g, dtype=torch.int32)
    codes = ops.pack_weight_codes(idx, LI4, False).cuda()
    f = (torch.rand(64, generator=g) * 0.01).cuda()
    lin = ops.IntegerLinear.from_parts(codes, LI4, False, torch.float32, 64, 64, f, None, None, 3, lut_values=lut)
    qx = torch.randint(-128, 128, (9, 64), generator=g, dtype=torch.int8).cuda()
    y = torch.ops.mctq.packed_linear_i8_lut(qx, 3, codes, LI4, 64, lut.tolist(), lin.w_rowsum, lin.factor, None)
    assert torch.equal(y, lin.gemm(qx))
    y_cpu = torch.ops.mctq.packed_linear_i8_lut(qx.cpu(), 3, codes.cpu(), LI4, 64, lut.tolist(), lin.w_rowsum.cpu(),
                                                lin.factor.cpu(), None)
    assert torch.equal(y_cpu, y.cpu())
    with pytest.raises(ValueError, match="LUT values"):
        torch.ops.mctq.packed_linear_i8_lut(qx, 3, codes, LI4, 64, lut.tolist() + [0], lin.w_rowsum, lin.factor, None)
    # conv: (r, s, c)-ordered indices
    cidx = torch.randint(0, 16, (24, 32, 3, 3), generator=g, dtype=torch.int32)
    ccodes = ops.pack_weight_codes(cidx.permute(0, 2, 3, 1).contiguous(), LI4, False).cuda()
    conv = ops.IntegerConv2d.from_parts(ccodes, LI4, False, torch.float32, 24, 32, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1),
                                        f[:24], None, None, 0, lut_values=lut)
    xq = torch.randint(-128, 128, (2, 6, 5, 32), generator=g, dtype=torch.int8).cuda()
    yc = torch.ops.mctq.packed_conv2d_i8_lut(xq, 0, ccodes, LI4, 24, [3, 3], [1, 1], [1, 1], [1, 1, 1, 1], lut.tolist(),
                                             conv.w_rowsum, conv.factor, None, False)
    assert torch.equal(yc, conv.gemm(xq))
    with torch._subclasses.fake_tensor.FakeTensorMode(allow_non_fake_inputs=True):
        fy = torch.ops.mctq.packed_conv2d_i8_lut(torch.empty(2, 6, 5, 32, dtype=torch.int8, device="cuda"), 0, ccodes, LI4,
                                                 24, [3, 3], [1, 1], [1, 1], [1, 1, 1, 1], lut.tolist(), conv.w_rowsum,
                                                 conv.factor, None, False)
        assert tuple(fy.shape) == tuple(yc.shape) and fy.dtype == torch.float32


# ------------------------------------------------------------------------------------------------ GPU: module level
class _LutModel(torch.nn.Module):
    """holder -> LUT Linear (4-bit indices) -> holder -> LUT Linear (8-bit indices); holder -> LUT Conv -> holder -> LUT Conv."""

    def __init__(self):
        super().__init__()
        W = mctq.PytorchQuantizationWrapper
        self.h0 = PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [-1.7], [2.3]))
        self.l0 = W(torch.nn.Linear(64, 96), {"weight": _lut_q(96, 16, pot=True, thr=[0.25] * 96)})
        self.h1 = PytorchActivationQuantizationHolder(Q.ActivationSymmetricInferableQuantizer(8, [6.0], True))
        self.l1 = W(torch.nn.Linear(96, 32, bias=False), {"weight": _lut_q(32, 100, thr=[0.3 + 0.01 * c for c in range(32)])})
        self.h2 = PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [-1.0], [3.0]))
        self.c0 = W(torch.nn.Conv2d(32, 48, (4, 3), padding="same"), {"weight": _lut_q(48, 16, thr=[0.2] * 48, rank=4)})
        self.h3 = PytorchActivationQuantizationHolder(Q.ActivationSymmetricInferableQuantizer(8, [4.0], False))
        self.c1 = W(torch.nn.Conv2d(48, 16, 1, stride=2), {"weight": _lut_q(16, 40, pot=True, thr=[0.5] * 16, rank=4)})
        self.cuda()

    def forward(self, x, img):
        a = self.l1(self.h1(self.l0(self.h0(x))))
        b = self.c1(self.h3(self.c0(self.h2(img))))
        return a, b


def _agree(y, hx, w, bias, conv=None):
    """|y - (Q(x) W + b)| <= 2^-21 (sum_k |Q(x)_k W_ok| + |b_o|): the product and its bound in f64 from the holder's output
    hx and the rebuilt weight w (the rounding of W to f32 and the f32 scaling of integer mode stay inside it)."""
    F = torch.nn.functional
    if conv is None:
        prod = lambda a, b: a @ b.T                                                  # noqa: E731
    else:
        prod = lambda a, b: F.conv2d(F.pad(a, conv._reversed_padding_repeated_twice), b, stride=conv.stride,   # noqa: E731
                                     dilation=conv.dilation)
    exact, mag = prod(hx.double(), w.double()), prod(hx.double().abs(), w.double().abs())
    if bias is not None:
        b = bias.double().reshape((1, -1) if conv is None else (1, -1, 1, 1))
        exact, mag = exact + b, mag + b.abs()
    err = (y.double() - exact).abs()
    assert bool((err <= 2.0 ** -21 * mag).all()), float((err / mag.clamp_min(1e-300)).max())


@pytest.mark.gpu
def test_model_switch():
    torch.manual_seed(0)
    model = _LutModel()
    x = torch.randn(37, 64, device="cuda") * 1.5
    img = torch.randn(3, 32, 11, 10, device="cuda")
    with torch.no_grad(), _no_tf32():
        packed = copy.deepcopy(model)
        PW.pack_model_weights(packed)
        report = PW.pack_model_weights(model, integer_linear=True, integer_conv=True, integer_lut=True)
        for name, holder, flag in (("l0", "h0", "integer"), ("l1", "h1", "integer"), ("c0", "h2", "integer_conv"),
                                   ("c1", "h3", "integer_conv")):
            r = report[name]["weight"]
            assert r["packed"] and r[flag] and r[flag + "_reason"] == "" and r["input_holder"] == holder, (name, r)
        assert [getattr(model, n)._packed.entries[0].kind for n in ("l0", "l1", "c0", "c1")] == [LI4, LU8, LI4, LU8]
        y = model(x, img)
        assert all(torch.equal(a, b) for a, b in zip(model(x, img), y))                 # a second call: the same bits
        # each switched layer against the packed path on the same holder input
        for h, l, inp in ((model.h0, "l0", x), (model.h1, "l1", model.l0(model.h0(x))), (model.h2, "c0", img),
                          (model.h3, "c1", model.c0(model.h2(img)))):
            hx = h(inp)
            wrapper = getattr(model, l)
            w_rebuilt = wrapper.get_quantized_weights()["weight"]
            _agree(wrapper(hx), hx, w_rebuilt, wrapper.layer.bias, wrapper.layer if l.startswith("c") else None)
        # pickle, state_dict, .to
        buf = io.BytesIO()
        torch.save(model, buf)
        buf.seek(0)
        m2 = torch.load(buf, weights_only=False)
        assert m2.l0._packed.integer and all(torch.equal(a, b) for a, b in zip(m2(x, img), y))
        m3 = copy.deepcopy(model)
        m3.load_state_dict(model.state_dict())
        assert set(m3.state_dict()) == set(model.state_dict()) == set(packed.state_dict())
        assert all(torch.equal(a, b) for a, b in zip(m3(x, img), y))
        m4 = copy.deepcopy(model).to("cpu").to("cuda")
        assert all(torch.equal(a, b) for a, b in zip(m4(x, img), y))
        assert pickle.loads(pickle.dumps(model.c0._packed)).integer
    # switching one wrapper in place
    w = mctq.PytorchQuantizationWrapper(torch.nn.Linear(64, 16), {"weight": _lut_q(16, 16)}).cuda()
    q = Q.ActivationSymmetricInferableQuantizer(8, [4.0], False)
    assert not w.pack_weights(integer_linear=True, input_quantizer=q)["weight"]["integer"]
    r = w.pack_weights(integer_linear=True, input_quantizer=q, integer_lut=True)["weight"]
    assert r["integer"] and r["integer_reason"] == "" and w._packed.integer


@pytest.mark.gpu
def test_fallbacks_and_graph(monkeypatch):
    torch.manual_seed(1)
    model = _LutModel()
    x, img = torch.randn(20, 64, device="cuda"), torch.randn(4, 32, 9, 9, device="cuda")
    PW.pack_model_weights(model, integer_linear=True, integer_conv=True, integer_lut=True)
    with torch.no_grad():
        y = model(x, img)
        hx, himg = model.h0(x), model.h2(img)
    calls = []
    for cls in (ops.IntegerLinear, ops.IntegerConv2d):
        real = cls.__call__
        monkeypatch.setattr(cls, "__call__", lambda self, *a, real=real: calls.append(1) or real(self, *a))
    model.l0(hx.clone().requires_grad_(True))                                          # autograd: the packed path
    h = model.c0.layer.register_forward_hook(lambda *a: None)
    with torch.no_grad():
        model.c0(himg)                                                                 # hooks: the packed path
        h.remove()
        assert model.c0(himg[0]).dim() == 3                                            # unbatched input: the packed path
    assert calls == []
    for x_other in (hx.double(), hx.cpu()):                                            # other dtype or device
        assert model.l0._packed.integer_forward(model.l0, x_other) is None
    with torch.no_grad():
        assert all(torch.equal(a, b) for a, b in zip(model(x, img), y)) and len(calls) == 4
    # CUDA-graph capture after a warm-up replays the same bits (the table travels in the kernel arguments)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.no_grad(), torch.cuda.stream(s):
        model(x, img)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            y_g = model(x, img)
    torch.cuda.current_stream().wait_stream(s)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(y_g, y))
