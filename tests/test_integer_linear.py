"""Integer linear mode: mctq_quantize_rows_i8 + mctq_packed_linear_i8 (csrc/mctq_packed_igemm.cu) and the packed-wrapper mode
built on them (pytorch/packed_weights.py).  Every GPU result is checked bit for bit against an exact integer reference."""
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
from mct_quantizers_b200.pytorch.fused_activation_holder import PytorchFusedActivationQuantizationHolder
from mct_quantizers_b200.pytorch.packed_weights import PackedState, integer_linear_edges, integer_linear_eligibility
from mct_quantizers_b200.pytorch.preserving_activation_quantization_holder import \
    PytorchPreservingActivationQuantizationHolder

from test_packed_linear import _fake_packed, _lin_desc

I8, I4, LU8 = _native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4, _native.PACK_LUT_U8
DTYPES = {torch.float32: _native.F32, torch.bfloat16: _native.BF16, torch.float16: _native.F16}


# ------------------------------------------------------------------------------------------------ integer reference
def reference(qx, zx, qw, zw, f, bias, out_dtype):
    """The formula of include/mctq.h in numpy: int64 sums, one f32 conversion, f32 product and bias, one rounding to T."""
    qx, qw = np.asarray(qx, np.int64), np.asarray(qw, np.int64)
    K = qx.shape[1]
    zw = np.broadcast_to(np.asarray(zw, np.int64).reshape(-1), (qw.shape[0],))
    f = np.broadcast_to(np.asarray(f, np.float32).reshape(-1), (qw.shape[0],))
    acc = qx @ qw.T
    c = acc - zw[None, :] * qx.sum(1)[:, None] - zx * qw.sum(1)[None, :] + K * zx * zw[None, :]
    y = c.astype(np.float32) * f[None, :]
    if bias is not None:
        y = y + np.asarray(bias, np.float32)[None, :]
    return torch.from_numpy(np.ascontiguousarray(y, dtype=np.float32)).to(out_dtype)


def reference_on_device(qx, zx, qw, zw, f, bias, out_dtype):
    """The same formula for large shapes: the code sums in f64 on the device are exact (|sum| < 2^53), the rest is f32."""
    qx, qw = qx.to(torch.float64), qw.to(torch.float64)
    K = qx.shape[1]
    zw = zw.reshape(-1).to(torch.float64).expand(qw.shape[0])
    c = qx @ qw.T - zw[None, :] * qx.sum(1)[:, None] - zx * qw.sum(1)[None, :] + K * zx * zw[None, :]
    c = c.to(torch.int64).to(torch.float32)          # exact integer, then one rounding to f32 (round to nearest even)
    y = c * f.reshape(-1).to(torch.float32).expand(qw.shape[0])[None, :]
    if bias is not None:
        y = y + bias.to(torch.float32)[None, :]
    return y.to(out_dtype)


def test_reference_hand_worked():
    # qx = [[3, -1]], zx = 2; qw = [[1, 4], [-2, 0]], zw = [1, -1]; f = [0.5, 0.25]; bias = [1, 0]
    # (qx - zx) = [1, -3]; (qw - zw) = [[0, 3], [-1, 1]]  ->  c = [-9, -4]  ->  y = [-9 * 0.5 + 1, -4 * 0.25] = [-3.5, -1]
    y = reference([[3, -1]], 2, [[1, 4], [-2, 0]], [1, -1], [0.5, 0.25], [1.0, 0.0], torch.float32)
    assert y.tolist() == [[-3.5, -1.0]]
    # c = 16777217 is not an f32: it rounds to 16777216 before the scaling (the formula's (float)c)
    y = reference([[1]], 0, [[1]], [-16777216], [1.0], None, torch.float32)
    assert y.item() == 16777216.0
    # one rounding to bf16 at the end: 1 + 2^-9 is a tie between two bf16 values and rounds to even
    y = reference([[1]], 0, [[1]], [0], [1.0 + 2.0 ** -9], None, torch.bfloat16)
    assert y.float().item() == 1.0


def test_max_k_table():
    lib = _native.load()
    for ws in (0, 1):
        for xs in (0, 1):
            k = _native.integer_linear_max_k(ws, xs)
            assert lib.mctq_packed_linear_i8_max_k(ws, xs) == k
            m = 128 * 128 if ws and xs else 255 * 128 if ws or xs else 255 * 255
            assert m * k < 2 ** 31 <= m * (k + 1)


# ------------------------------------------------------------------------------------------------ C-ABI rejections
def _call(d, out_f=10, in_f=32, xq=0x7f5000000000, x_signed=1, zx=0, M=1, x_rowsum=None, w_rowsum=0x7f6100000000,
          factor=0x7f6200000000, y_dtype=_native.F32, y=0x7f6000000000, ldy=None):
    lib = _native.load()
    return lib.mctq_packed_linear_i8(ctypes.byref(d) if d is not None else None, out_f, in_f, xq, x_signed, zx, M, x_rowsum,
                                     w_rowsum, factor, None, y_dtype, y, out_f if ldy is None else ldy, None)


def test_c_abi_rejections():
    E_BADARG, E_DTYPE, E_RANGE = -1, -2, -3
    ok = lambda **k: _lin_desc(out_f=10, in_f=32, **k)        # noqa: E731
    assert _call(None) == E_BADARG
    assert _call(_lin_desc(out_f=10, in_f=32, kind=LU8)) == E_BADARG                  # LUT kinds
    assert _call(_lin_desc(out_f=10, in_f=32, kind=_native.PACK_LUT_I4)) == E_BADARG
    assert _call(ok(dtype=_native.BF16)) == E_DTYPE                                   # y dtype != rebuilt dtype
    assert _call(ok(), y_dtype=7) == E_DTYPE
    assert _call(_lin_desc(out_f=10, in_f=24), in_f=24) == E_BADARG                   # in_features % 16
    assert _call(_lin_desc(out_f=10, in_f=48, kind=I4), in_f=48) == E_BADARG          # int4: in_features % 32
    assert _call(ok(), xq=0x7f5000000008) == E_BADARG                                 # misaligned x codes
    d = ok()
    d.codes = 0x7f0000000004
    assert _call(d) == E_BADARG                                                       # misaligned weight codes
    assert _call(ok(), xq=None) == E_BADARG
    assert _call(ok(), y=None) == E_BADARG
    assert _call(ok(), factor=None) == E_BADARG
    assert _call(ok(), zx=3, w_rowsum=None) == E_BADARG                               # zx != 0 needs Sw
    assert _call(ok(), ldy=9) == E_BADARG
    assert _call(ok(), M=-1) == E_BADARG
    d = ok()
    d.zp = None
    assert _call(d) == E_BADARG
    assert _call(ok(), x_signed=1, zx=128) == E_RANGE                                 # zx outside the x codes' range
    assert _call(ok(), x_signed=0, zx=-1) == E_RANGE
    for ws, xs, k in ((1, 1, 131071), (0, 1, 65793), (1, 0, 65793), (0, 0, 33025)):
        big = (k // 16 + 1) * 16
        d = _lin_desc(out_f=2, in_f=big)
        d.is_signed = ws
        assert _call(d, out_f=2, in_f=big, x_signed=xs) == E_RANGE                    # K over the int32 bound
        d = _lin_desc(out_f=2, in_f=k // 16 * 16)
        d.is_signed = ws
        assert _call(d, out_f=2, in_f=k // 16 * 16, x_signed=xs, M=0) == 0            # at the bound: accepted (M = 0: no-op)
    assert _call(ok(), M=0) == 0
    lib = _native.load()
    q = lambda **k: lib.mctq_quantize_rows_i8(k.get("x", 0x7f5000000000), k.get("dt", _native.F32), k.get("M", 1),   # noqa: E731
                                               k.get("K", 16), 1.0, 0, k.get("qmin", -128), k.get("qmax", 127),
                                               k.get("codes", 0x7f6000000000), None, None)
    assert q(x=None) == E_BADARG and q(codes=None) == E_BADARG and q(M=-1) == E_BADARG and q(K=0) == E_BADARG
    assert q(dt=5) == E_DTYPE
    assert q(qmin=1, qmax=0) == E_RANGE and q(qmin=-129) == E_RANGE and q(qmin=0, qmax=256) == E_RANGE
    assert q(M=0) == 0


# ------------------------------------------------------------------------------------------------ eligibility and edges
def _act(kind="sym", bits=8, signed=True):
    if kind == "sym":
        return Q.ActivationSymmetricInferableQuantizer(bits, [4.0], signed)
    if kind == "pot":
        return Q.ActivationPOTInferableQuantizer(bits, [4.0], signed)
    if kind == "uniform":
        return Q.ActivationUniformInferableQuantizer(bits, [-1.5], [3.0])
    return Q.ActivationLutPOTInferableQuantizer(bits, [-2.0, 0.0, 1.0, 3.0], [4.0], signed)


def _wrapper(in_f=32, out_f=8):
    w = Q.WeightsSymmetricInferableQuantizer(8, [1.0] * out_f, True, 0)
    return mctq.PytorchQuantizationWrapper(torch.nn.Linear(in_f, out_f), {"weight": w})


def test_eligibility():
    q = _act()
    assert integer_linear_eligibility(_fake_packed(_wrapper()), q) == (True, "")
    assert integer_linear_eligibility(_wrapper(), q) == (False, "the weight is not packed")
    lut = _fake_packed(_wrapper())
    lut._packed.entries[0].kind = LU8
    ok, why = integer_linear_eligibility(lut, q)
    assert not ok and "lut_u8" in why
    ok, why = integer_linear_eligibility(_fake_packed(_wrapper(in_f=40)), q)
    assert not ok and "multiple of 16" in why
    i4 = _fake_packed(_wrapper(in_f=48))
    i4._packed.entries[0].kind = I4
    ok, why = integer_linear_eligibility(i4, q)
    assert not ok and "multiple of 32" in why
    ok, why = integer_linear_eligibility(_fake_packed(_wrapper()), _act("lut"))
    assert not ok and "per-tensor affine" in why
    ok, why = integer_linear_eligibility(_fake_packed(_wrapper()), _act(bits=16))
    assert not ok and "8-bit codes" in why
    # K over the bound of the pair: u8 x u8 (unsigned weight codes, unsigned activation)
    big = _fake_packed(_wrapper(in_f=33040, out_f=1))
    big._packed.entries[0].is_signed = False
    ok, why = integer_linear_eligibility(big, _act(signed=False))
    assert not ok and "33025" in why
    assert integer_linear_eligibility(big, _act(signed=True))[0]                     # u8 x s8: bound 65793


class _Net(torch.nn.Module):
    def __init__(self, holders, wrappers, body):
        super().__init__()
        self.h = torch.nn.ModuleList(holders)
        self.w = torch.nn.ModuleList(wrappers)
        self.body = body

    def forward(self, x):
        return self.body(self, x)


def _edges(holders, wrappers, body):
    net = _Net(holders, [_fake_packed(w) for w in wrappers], body)
    edges, why, failure = integer_linear_edges(net)
    return {k: v[0] for k, v in edges.items()}, why, failure


def test_edges():
    H = lambda: PytorchActivationQuantizationHolder(_act())                           # noqa: E731
    # direct edge
    e, why, fail = _edges([H()], [_wrapper()], lambda m, x: m.w[0](m.h[0](x)))
    assert e == {"w.0": "h.0"} and not fail
    # through reshape / flatten / contiguous
    e, _, _ = _edges([H()], [_wrapper()], lambda m, x: m.w[0](m.h[0](x).reshape(-1, 32).contiguous().flatten(1)))
    assert e == {"w.0": "h.0"}
    # one holder feeding two linears; a fused holder
    fused = PytorchFusedActivationQuantizationHolder(_act(), "relu")
    e, _, _ = _edges([H(), fused], [_wrapper(), _wrapper(), _wrapper()],
                     lambda m, x: m.w[0](m.h[0](x)) + m.w[1](m.h[0](x)) + m.w[2](m.h[1](x)))
    assert e == {"w.0": "h.0", "w.1": "h.0", "w.2": "h.1"}
    # a non-holder producer
    e, why, _ = _edges([H()], [_wrapper()], lambda m, x: m.w[0](torch.relu(m.h[0](x))))
    assert e == {} and "not the output of an activation quantization holder" in why["w.0"]
    # a bypassed holder; a preserving holder that quantizes
    byp = PytorchPreservingActivationQuantizationHolder(_act(), quantization_bypass=True)
    keep = PytorchPreservingActivationQuantizationHolder(_act(), quantization_bypass=False)
    e, why, _ = _edges([byp, keep], [_wrapper(), _wrapper()], lambda m, x: m.w[0](m.h[0](x)) + m.w[1](m.h[1](x)))
    assert e == {"w.1": "h.1"} and "bypasses quantization" in why["w.0"]
    # an untraceable model: nothing is found, the reason is given
    def untraceable(m, x):
        if x.sum() > 0:
            return m.w[0](m.h[0](x))
        return x
    e, why, fail = _edges([H()], [_wrapper()], untraceable)
    assert e == {} and "cannot be traced" in fail


def test_model_reports_without_a_gpu():
    """pack_model_weights(integer_linear=True) on host-packed wrappers: its reports of switched, non-switched and
    untraceable models."""
    def untraceable(m, x):
        if x.sum() > 0:
            return m.w[0](m.h[0](x))
        return x
    net = _Net([PytorchActivationQuantizationHolder(_act())], [_fake_packed(_wrapper())], untraceable)
    r = PW.pack_model_weights(net, integer_linear=True)["w.0"]["weight"]
    assert r["integer"] is False and "cannot be traced" in r["integer_reason"] and r["input_holder"] is None
    assert net.w[0]._packed.integer is False

    net = _Net([PytorchActivationQuantizationHolder(_act())], [_fake_packed(_wrapper()), _fake_packed(_wrapper())],
               lambda m, x: m.w[0](m.h[0](x)) + m.w[1](torch.relu(x)))
    reports = PW.pack_model_weights(net, integer_linear=True)
    on, off = reports["w.0"]["weight"], reports["w.1"]["weight"]
    assert (on["integer"], on["integer_reason"], on["input_holder"]) == (True, "", "h.0")
    assert off["integer"] is False and off["input_holder"] is None
    assert "not the output of an activation quantization holder" in off["integer_reason"]
    assert net.w[0]._packed.integer and net.w[0]._packed.input_quantizer is net.h[0].activation_holder_quantizer
    assert net.w[1]._packed.integer is False


def test_default_state_and_old_pickles():
    st = PackedState([])
    assert st.integer is False and st.input_quantizer is None
    old = PackedState.__new__(PackedState)
    old.__dict__.update({'entries': [], 'fused': True, 'batched': False, '_plan': None, '_sig': None, '_lin': None})
    assert old.integer is False and old.input_quantizer is None
    st.integer, st.input_quantizer = True, _act()
    back = pickle.loads(pickle.dumps(st))
    assert back.integer and type(back.input_quantizer) is type(st.input_quantizer) and back._ilin is None


def test_wrapper_level_needs_an_input_quantizer():
    with pytest.raises(ValueError, match="input_quantizer"):
        PW.pack_wrapper_weights(_wrapper(), integer_linear=True)


# ------------------------------------------------------------------------------------------------ GPU: row quantizer
def _scalar_codes(x, scale, zp, qmin, qmax):
    """Codes of mctq_fq_affine_scalar with code_mode INT8."""
    lib = _native.load()
    xd = x.contiguous()
    y = torch.empty_like(xd)
    codes = torch.empty(xd.shape, dtype=torch.int8 if qmin < 0 else torch.uint8, device=x.device)
    rc = lib.mctq_fq_affine_scalar(xd.data_ptr(), y.data_ptr(), codes.data_ptr(), xd.numel(), DTYPES[x.dtype],
                                   float(np.float32(scale)), zp, qmin, qmax, _native.CODES_INT8,
                                   torch.cuda.current_stream().cuda_stream)
    _native.check(rc, "mctq_fq_affine_scalar")
    return codes


def _quantizers():
    return {"sym_s8": _act("sym"), "sym_u8": _act("sym", signed=False), "pot": _act("pot"),
            "uniform": Q.ActivationUniformInferableQuantizer(8, [-1.3], [2.9]),       # zp != 0, non-power-of-two scale
            "uniform_worst": Q.ActivationUniformInferableQuantizer(8, [-0.37], [5.11])}


def _launch_args(q):
    from mct_quantizers_b200.pytorch.fused_activation_holder import affine_scalar_params
    s, z, _, _ = affine_scalar_params(q)
    return q._validated_launch_args(s, z)[1]


def _special_x(M, K, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, K, generator=g) * 3
    flat = x.view(-1)
    flat[::97] = float("nan")
    flat[5::89] = float("inf")
    flat[7::83] = -float("inf")
    flat[11::79] = 1e6
    flat[13::73] = -1e6
    return x.to(dtype).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("qname", list(_quantizers()))
@pytest.mark.parametrize("M,K", [(1, 16), (7, 40), (33, 4096), (70001, 16), (5, 3)])
def test_row_quantizer_codes_and_sums(dtype, qname, M, K):
    q = _quantizers()[qname]
    s, z, qmin, qmax = _launch_args(q)
    x = _special_x(M, K, dtype, M * 31 + K)
    codes, rowsum = ops.quantize_rows_i8(x, s, z, qmin, qmax, True)
    ref = _scalar_codes(x, s, z, qmin, qmax)
    assert codes.dtype == ref.dtype and torch.equal(codes, ref)
    assert torch.equal(rowsum.cpu().to(torch.int64), codes.cpu().to(torch.int64).sum(1))
    c2, r2 = torch.ops.mctq.quantize_rows_i8(x, s, z, qmin, qmax, False)
    assert torch.equal(c2, codes) and r2.numel() == 0
    # idempotence: the codes of holder(x) are the codes of x
    hx = PytorchActivationQuantizationHolder(q)(x)
    c3, _ = ops.quantize_rows_i8(hx, s, z, qmin, qmax, False)
    nan = torch.isnan(x)
    assert torch.equal(c3[~nan], codes[~nan])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_idempotence_worst_case_grids(dtype):
    """Every grid point of 8-bit uniform grids with awkward scales, rounded to T, and a dense sweep: holder(x) re-quantizes
    to the codes of x."""
    for lo, hi in ((-0.37, 5.11), (-3.3, 0.71), (-1e-3, 7.77e-3), (-200.1, 13.9)):
        q = Q.ActivationUniformInferableQuantizer(8, [lo], [hi])
        s, z, qmin, qmax = _launch_args(q)
        grid = (torch.arange(qmin, qmax + 1, dtype=torch.float32) - z) * np.float32(s)
        sweep = torch.linspace(lo * 1.2, hi * 1.2, (1 << 16) - 256)
        x = torch.cat([grid, sweep]).to(dtype).cuda().reshape(-1, 64)
        hx = PytorchActivationQuantizationHolder(q)(x)
        a, _ = ops.quantize_rows_i8(x, s, z, qmin, qmax, False)
        b, _ = ops.quantize_rows_i8(hx, s, z, qmin, qmax, False)
        assert torch.equal(a, b), (lo, hi)


# ------------------------------------------------------------------------------------------------ GPU: the GEMM
def _weight(kind, signed, N, K, per_channel, zw_nonzero, dtype, g, extreme=None):
    lo, hi = ((-8, 7) if signed else (0, 15)) if kind == I4 else ((-128, 127) if signed else (0, 255))
    qw = torch.randint(lo, hi + 1, (N, K), generator=g, dtype=torch.int32) if extreme is None else \
        torch.full((N, K), extreme, dtype=torch.int32)
    C = N if per_channel else 1
    zw = torch.randint(lo, hi + 1, (C,), generator=g, dtype=torch.int32) if zw_nonzero else torch.zeros(C, dtype=torch.int32)
    scale = (torch.rand(C, generator=g) * 0.02 + 0.001).to(torch.float32)
    if kind == I4:
        u = (qw & 15).to(torch.uint8).reshape(-1, 2)
        codes = (u[:, 0] | (u[:, 1] << 4)).contiguous()
    else:
        codes = qw.to(torch.int8 if signed else torch.uint8).reshape(-1)
    return codes.cuda(), qw, zw, scale


def _gemm_case(M, N, K, kind, w_signed, per_channel, zw_nonzero, x_signed, zx, dtype, with_bias, seed, extreme=None):
    g = torch.Generator().manual_seed(seed)
    codes, qw, zw, scale = _weight(kind, w_signed, N, K, per_channel, zw_nonzero, dtype, g,
                                   None if extreme is None else extreme[0])
    xlo, xhi = (-128, 127) if x_signed else (0, 255)
    qx = torch.randint(xlo, xhi + 1, (M, K), generator=g, dtype=torch.int32) if extreme is None else \
        torch.full((M, K), extreme[1], dtype=torch.int32)
    xq = qx.to(torch.int8 if x_signed else torch.uint8).cuda()
    x_scale = 0.0371
    f = (torch.tensor(np.float32(x_scale)) * scale).to(torch.float32)
    bias = (torch.randn(N, generator=g) * 3).to(dtype).cuda() if with_bias else None
    lin = ops.IntegerLinear(codes, kind, w_signed, dtype, N, K, scale.cuda(), zw.cuda(), x_scale, zx, xlo, xhi)
    assert torch.equal(lin.factor.cpu(), f)
    rowsum = qx.sum(1).to(torch.int32).cuda()
    poison = torch.full((M, N + 9), float("nan"), dtype=dtype, device="cuda")
    out = poison[:, 3:3 + N]
    y = lin.gemm(xq, rowsum, bias, out=out)
    y2 = lin.gemm(xq, rowsum, bias)
    ref = reference_on_device(qx.cuda(), zx, qw.cuda(), zw.cuda(), f.cuda(), bias.float() if bias is not None else None, dtype)
    bits = lambda t: t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)   # noqa: E731
    assert torch.equal(bits(y), bits(ref)), f"{(y.float() - ref.float()).abs().max()}"
    assert torch.equal(bits(y2), bits(y))                                             # two calls, the same bits
    assert torch.isnan(poison[:, :3]).all() and torch.isnan(poison[:, 3 + N:]).all()  # nothing outside the view
    return lin


_SHAPES = [(1, 128, 16), (2, 127, 32), (15, 129, 144), (16, 1, 4096), (17, 128, 4096), (255, 128, 144), (256, 129, 32),
           (257, 127, 4096), (4099, 1, 16), (1, 11008, 4096), (64, 4096, 11008), (1024, 11008, 144), (3, 300, 11008)]
_CONFIGS = [(kind, ws, xs, zx) for kind in (I8, I4) for ws in (True, False) for xs, zx in ((True, 0), (True, -7), (False, 0),
                                                                                            (False, 128))]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("ci", range(len(_CONFIGS)))
def test_gemm_bit_exact(ci, dtype):
    kind, ws, xs, zx = _CONFIGS[ci]
    for si in range(ci % 3, len(_SHAPES), 3):
        M, N, K = _SHAPES[si]
        if kind == I4:
            K = (K + 31) // 32 * 32
        _gemm_case(M, N, K, kind, ws, per_channel=(si + ci) % 2 == 0, zw_nonzero=(si + ci) % 3 != 0, x_signed=xs, zx=zx,
                   dtype=dtype, with_bias=si % 2 == 1, seed=1000 * ci + si)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [I8, I4])
def test_gemm_at_the_bound(kind):
    # u8 x u8 at K = 33024 (the largest multiple of 16 under 33025): every product 255 * 255, the int32 sum just below 2^31
    K = 33024 if kind == I8 else 33024 // 32 * 32
    ext = (255 if kind == I8 else 15, 255)
    _gemm_case(5, 130, K, kind, False, True, False, False, 0, torch.float32, False, 7, extreme=ext)
    # s8 x s8 extremes at their bound: (-128) * (-128) everywhere
    K = 131071 // 32 * 32
    ext = (-128 if kind == I8 else -8, -128)
    _gemm_case(3, 129, K, kind, True, False, False, True, 0, torch.float32, True, 8, extreme=ext)


@pytest.mark.gpu
def test_split_k_of_1_and_8_agree():
    # N = 128, M = 16, K = 4096 runs as clusters of 8 CTAs; N = 11008, M = 1024 as single CTAs; the bits match the reference
    _gemm_case(16, 128, 4096, I8, True, True, True, True, 3, torch.float32, True, 11)
    _gemm_case(1024, 11008, 256, I8, True, True, True, True, 3, torch.float32, True, 12)


@pytest.mark.gpu
def test_torch_ops_match_integer_linear():
    g = torch.Generator().manual_seed(3)
    codes, qw, zw, scale = _weight(I4, True, 64, 64, True, True, torch.float32, g)
    lin = ops.IntegerLinear(codes, I4, True, torch.bfloat16, 64, 64, scale.cuda(), zw.cuda(), 0.05, 2, -128, 127)
    x = torch.randn(9, 64, device="cuda").to(torch.bfloat16)
    qx, rs = torch.ops.mctq.quantize_rows_i8(x, 0.05, 2, -128, 127, True)
    y = torch.ops.mctq.packed_linear_i8(qx, 2, rs, codes, I4, True, 64, zw.cuda(), lin.w_rowsum, lin.factor, None,
                                        torch.bfloat16)
    assert torch.equal(y.view(torch.int16), lin(x).view(torch.int16))
    y_cpu = torch.ops.mctq.packed_linear_i8(qx.cpu(), 2, rs.cpu(), codes.cpu(), I4, True, 64, zw, lin.w_rowsum.cpu(),
                                            lin.factor.cpu(), None, torch.bfloat16)
    assert torch.equal(y_cpu.view(torch.int16), y.cpu().view(torch.int16))
    # malformed calls raise: one zero point for 64 per-channel factors, and no x row sums while a zero point is not 0
    with pytest.raises(ValueError, match="zero points"):
        torch.ops.mctq.packed_linear_i8(qx, 2, rs, codes, I4, True, 64, zw[:1].cuda(), lin.w_rowsum, lin.factor, None,
                                        torch.bfloat16)
    with pytest.raises(RuntimeError, match="row sums"):
        torch.ops.mctq.packed_linear_i8(qx, 2, None, codes, I4, True, 64, zw.cuda(), lin.w_rowsum, lin.factor, None,
                                        torch.bfloat16)


# ------------------------------------------------------------------------------------------------ GPU: module level
class _Model(torch.nn.Module):
    """holder -> Linear -> holder -> reshape -> Linear (+ a second use of the first holder's output)."""

    def __init__(self, dtype, wq_kind):
        super().__init__()
        wq = (lambda C: Q.WeightsSymmetricInferableQuantizer(4, [0.5] * C, True, 0)) if wq_kind == "i4" else \
            (lambda C: Q.WeightsUniformInferableQuantizer(8, [-0.3] * C, [0.2] * C, True, 0))
        self.h0 = PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [-1.7], [2.3]))
        self.l0 = mctq.PytorchQuantizationWrapper(torch.nn.Linear(64, 96), {"weight": wq(96)})
        self.h1 = PytorchActivationQuantizationHolder(Q.ActivationSymmetricInferableQuantizer(8, [6.0], True))
        self.l1 = mctq.PytorchQuantizationWrapper(torch.nn.Linear(96, 32, bias=False), {"weight": wq(32)})
        self.to(dtype).cuda()

    def forward(self, x):
        a = self.l0(self.h0(x))
        return self.l1(self.h1(a).reshape(-1, 96))


def _model_reference(model, x):
    """The numpy integer formula of each switched layer, with Q's codes of its input."""
    out = x
    for h, l in ((model.h0, model.l0), (model.h1, model.l1)):
        st = l._packed
        e = st.entries[0]
        s, z, qmin, qmax = _launch_args(h.activation_holder_quantizer)
        qx, _ = ops.quantize_rows_i8(out.reshape(-1, l.layer.in_features), s, z, qmin, qmax, False)
        it = e.plan_item()
        qw = ops.weight_code_values(e.codes, e.kind, e.is_signed, l.layer.out_features, l.layer.in_features)
        f = (torch.tensor(np.float32(s)) * it[8].cpu()).numpy()
        bias = l.layer.bias.float().cpu().numpy() if l.layer.bias is not None else None
        out = reference(qx.cpu().numpy(), z, qw.cpu().numpy(), it[9].cpu().numpy(), f, bias, out.dtype).cuda()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("wq_kind", ["i8", "i4"])
def test_model_switch(dtype, wq_kind):
    torch.manual_seed(0)
    model = _Model(dtype, wq_kind)
    x = (torch.randn(37, 64, device="cuda") * 1.5).to(dtype)
    with torch.no_grad():
        y_float = model(x)
        report = PW.pack_model_weights(model, integer_linear=True)
        for name, holder in (("l0", "h0"), ("l1", "h1")):
            r = report[name]["weight"]
            assert r["packed"] and r["integer"] and r["integer_reason"] == "" and r["input_holder"] == holder
        assert model.l0._packed.integer and model.l1._packed.integer
        y = model(x)
        ref = _model_reference(model, x)
        assert torch.equal(y.float(), ref.float())
        tol = 2e-2 if dtype != torch.float32 else 1e-4
        assert torch.allclose(y.float(), y_float.float(), atol=tol * float(y_float.abs().max()), rtol=0)
        # pickle, state_dict, .to
        buf = io.BytesIO()
        torch.save(model, buf)
        buf.seek(0)
        m2 = torch.load(buf, weights_only=False)
        assert m2.l0._packed.integer and torch.equal(m2(x).float(), y.float())
        m3 = copy.deepcopy(model)
        m3.load_state_dict(model.state_dict())
        assert set(m3.state_dict()) == set(model.state_dict()) and torch.equal(m3(x).float(), y.float())
        m4 = copy.deepcopy(model).to("cpu").to("cuda")
        assert torch.equal(m4(x).float(), y.float())


@pytest.mark.gpu
def test_fallbacks_graph_and_dependent_launch(monkeypatch):
    torch.manual_seed(1)
    model = _Model(torch.float32, "i8")
    x = torch.randn(20, 64, device="cuda")
    PW.pack_model_weights(model, integer_linear=True)
    with torch.no_grad():
        y = model(x)
    calls = []
    real = ops.IntegerLinear.__call__
    monkeypatch.setattr(ops.IntegerLinear, "__call__", lambda self, *a: calls.append(1) or real(self, *a))
    # autograd recording: the exact packed path, not integer mode
    with torch.no_grad():
        hx = model.h0(x)
    y_grad = model.l0(hx.clone().requires_grad_(True))
    assert calls == [] and y_grad.requires_grad
    # forward hooks: the exact packed path
    h = model.l0.layer.register_forward_hook(lambda *a: None)
    with torch.no_grad():
        model.l0(hx)
    h.remove()
    assert calls == []
    with torch.no_grad():
        assert torch.equal(model(x), y) and len(calls) == 2
    # CUDA-graph capture replays the same bits
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
    # dependent-launch orders 2 and 3 (fake-quant -> row quantizer -> GEMM chains) give the default order's bits
    lib = _native.load()
    for order in (2, 3):
        prev = lib.mctq_set_tuning(3, order)
        try:
            with torch.no_grad():
                outs = [model(x) for _ in range(3)]
            torch.cuda.synchronize()
        finally:
            lib.mctq_set_tuning(3, prev)
        assert all(torch.equal(o, y) for o in outs)


@pytest.mark.gpu
def test_wrapper_level_switch_and_reports():
    torch.manual_seed(2)
    q = Q.ActivationSymmetricInferableQuantizer(8, [4.0], False)
    w = mctq.PytorchQuantizationWrapper(torch.nn.Linear(48, 16), {"weight": Q.WeightsSymmetricInferableQuantizer(8, [0.5] * 16, True, 0)}).cuda()
    r = w.pack_weights(integer_linear=True, input_quantizer=q)["weight"]
    assert r["packed"] and r["integer"] and r["input_holder"] is None
    x = PytorchActivationQuantizationHolder(q)(torch.rand(5, 48, device="cuda") * 4)
    with torch.no_grad():
        y = w(x)
        w2 = copy.deepcopy(w)
        w2._packed.integer = False
        assert torch.allclose(y, w2(x), atol=1e-4 * float(y.abs().max()), rtol=0)
    # LUT weights stay on their paths
    lut = mctq.PytorchQuantizationWrapper(torch.nn.Linear(32, 8), {"weight": Q.WeightsLUTSymmetricInferableQuantizer(
        8, [-3.0, -1.0, 0.0, 2.0], [1.0] * 8, True, 0, 2)}).cuda()
    r = lut.pack_weights(integer_linear=True, input_quantizer=q)["weight"]
    assert r["packed"] and not r["integer"] and "lut" in r["integer_reason"]
