"""Batched packed linear (csrc/mctq_packed_gemm.cu, torch.ops.mctq.packed_linear_batched, batched linear mode of packed
wrappers) against the f64 product with the weight of the independent host decoder (test_packed_variants.decoded_f64)."""
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
from mct_quantizers_b200.pytorch.packed_weights import (FUSED_BATCHED_MAX_ROWS, FUSED_LINEAR_MAX_ROWS, PackedState,
                                                        batched_linear_eligibility, pack_model_weights)
from test_packed_linear import _exact_path, _fake_packed, _lin_desc, _lut_q, _wrapped_linear
from test_packed_variants import (DT, HALF_SUBNORMAL, I4, I8, INT4_KINDS, KIND_DTYPES, LI4, LU8, LUT_KINDS, U_OUT, _dev,
                                  _lin_data, _np_bits, _ref, _same_pattern, _weight, _x)


def _batched(x, data, kind, N, bias=None):
    codes, is_signed, scale, zp, quot = data
    return torch.ops.mctq.packed_linear_batched(x, _dev(codes), kind, is_signed, N, _dev(scale), _dev(zp), _dev(quot), bias)


def _assert_exact(y, x, w, bias, what):
    want, _ = _ref(x, w, bias)
    got, ref = _np_bits(y).reshape(want.shape), _np_bits(torch.from_numpy(want).to(y.dtype)).reshape(want.shape)
    if not np.array_equal(got, ref):
        bad = np.argwhere(got != ref)
        raise AssertionError(f"{what}: {len(bad)} outputs differ, first (row, col) {bad[:4].tolist()}")


def _bound(y, x, w, bias):
    """The bound of include/mctq.h: (2^-22 (in / 16 + 8)) sum|x w| + u_T |y| + 2^-126 sum|w| (x below the normal range) and
    the subnormal grain of the output."""
    want, mag = _ref(x, w, bias)
    K = x.shape[-1]
    got = y.double().cpu().numpy().reshape(want.shape)
    wsum = np.abs(w).sum(1)[None, :]
    lim = (2.0 ** -22 * (K / 16 + 8)) * mag + U_OUT[y.dtype] * np.abs(want) + 2.0 ** -126 * wsum + \
        HALF_SUBNORMAL[y.dtype] + 4 * 2.0 ** -149
    err = np.abs(got - want)
    return bool(np.all(err <= lim)), float(np.max(err - lim))


# --------------------------------------------------------------------------------------------- CPU
def _call_b(d, out_f=10, in_f=33, x=0x7f5000000000, M=1, y=0x7f6000000000, quot_host=None):
    lib = _native.load()
    p = ctypes.addressof(d) if d is not None else None
    q = quot_host.ctypes.data if quot_host is not None else None
    return lib.mctq_packed_linear_batched(p, out_f, in_f, x, d.y_dtype if d is not None else 0, M, None, y, q, None)


def test_c_abi_rejections():
    """The argument checks of mctq_packed_linear, and LUT quotients that are not exact in bf16, before any CUDA call."""
    assert _call_b(_lin_desc(), M=0) == 0
    assert _call_b(None) == -1
    assert _call_b(_lin_desc(kind=0)) == -1 and _call_b(_lin_desc(kind=5)) == -1
    assert _call_b(_lin_desc(), x=None) == -1 and _call_b(_lin_desc(), y=None) == -1
    d = _lin_desc()
    d.zp = None
    assert _call_b(d) == -1
    assert _call_b(_lin_desc(), in_f=34) == -1
    assert _call_b(_lin_desc(C=5, inner=33)) == -1
    assert _call_b(_lin_desc(dtype=_native.BF16, kind=_native.PACK_LUT_U8)) == -2
    assert _call_b(_lin_desc(), M=-1) == -1
    good = (np.arange(16, dtype=np.float32) - 8) / 128
    assert _call_b(_lin_desc(kind=LI4), quot_host=good, M=0) == 0
    assert _call_b(_lin_desc(kind=LI4), quot_host=None) == -4                        # no host copy of the quotients
    assert _call_b(_lin_desc(kind=LI4, K=17), quot_host=good) == -4
    bad = good.copy()
    bad[5] = np.float32(1.0 + 2.0 ** -9)                                             # needs more than bf16's 8 bits
    assert _call_b(_lin_desc(kind=LI4), quot_host=bad) == -4
    assert _call_b(_lin_desc(kind=LI4), quot_host=bad, M=0) == -4                     # checked before the M == 0 return
    # several faults: the order of mctq_packed_linear, then the host quotients
    assert _call_b(_lin_desc(kind=5, dtype=3)) == -1
    assert _call_b(_lin_desc(kind=LI4, dtype=_native.BF16, K=17)) == -2
    assert _call_b(_lin_desc(kind=LI4, K=17), in_f=34, quot_host=good) == -1
    assert _call_b(_lin_desc(kind=LI4), x=None, quot_host=bad) == -1
    assert _call_b(_lin_desc(kind=LI4, K=17), quot_host=bad) == -4
    assert _call_b(_lin_desc(kind=LI4), quot_host=None, M=0) == -4


def _lut_np(values, bw=8):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return Q.WeightsLUTSymmetricInferableQuantizer(4, [float(v) for v in values], [1.0] * 4, True, 0, 2, bw)


def test_eligibility_and_reports():
    sym = Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 4, True, 0)
    lin = mctq.PytorchQuantizationWrapper(torch.nn.Linear(6, 4), {"weight": sym})
    assert batched_linear_eligibility(lin) == (False, "the weight is not packed")
    assert batched_linear_eligibility(_fake_packed(lin)) == (True, "")
    # LUT: integer centroids on an 8-bit grid are bf16-exact quotients; a 12-bit grid with 9 significant bits is not
    for values, bw, ok in (([-128, -3, 5, 127], 8, True), ([-2047, 3, 5, 1023], 12, False)):
        w = mctq.PytorchQuantizationWrapper(torch.nn.Linear(6, 4), {"weight": _lut_np(values, bw)})
        _fake_packed(w)
        w._packed.entries[0].kind = LI4
        got = batched_linear_eligibility(w)
        assert got[0] == ok and (ok or "bfloat16" in got[1]), got
    conv = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(3, 4, 1), {"weight": sym})
    ok, why = batched_linear_eligibility(_fake_packed(conv, shape=(4, 3), stride=(3, 1), C=4, inner=3))
    assert not ok and "Conv2d" in why
    with pytest.raises(ValueError):
        PW.pack_wrapper_weights(lin, fused_linear=False, batched_linear=True)
    with pytest.raises(ValueError):
        pack_model_weights(torch.nn.Sequential(lin), batched_linear=True)


def test_default_state_and_old_pickles():
    st = PackedState([])
    assert st.batched is False and "batched" in st.__getstate__()
    assert pickle.loads(pickle.dumps(st)).batched is False
    old = PackedState.__new__(PackedState)          # unpickling a state written before batched mode existed
    old.__dict__.update({'entries': [], 'fused': True, '_plan': None, '_sig': None, '_lin': None})
    assert old.batched is False and old.fused is True


def test_row_limits():
    for dt in (torch.float32, torch.bfloat16, torch.float16):
        assert FUSED_BATCHED_MAX_ROWS[dt] >= FUSED_LINEAR_MAX_ROWS[dt]


# --------------------------------------------------------------------------------------------- GPU: exact
SIGNED_CASES = [(k, dt, s) for k, dt in KIND_DTYPES for s in ((True, False) if k not in LUT_KINDS else (False,))]


def _shapes(kind):
    shapes = [(M, 17, 33) for M in (9, 16, 17, 255, 256, 257)]
    shapes += [(20, N, 64) for N in (1, 127, 128, 129, 4097)]
    ks = (1, 7, 8, 9, 63, 64, 65, 127, 128, 129, 511, 513, 1040, 4095)
    shapes += [(9, 33, K) for K in ks]
    shapes += [(130, 129, 4096 + 1), (24, 4096, 11008)]
    return shapes


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype,is_signed", SIGNED_CASES)
@pytest.mark.parametrize("per_channel", [True, False])
@pytest.mark.parametrize("with_bias", [True, False])
def test_exact_against_the_decoder(kind, dtype, is_signed, per_channel, with_bias):
    """Exactly representable data: the output equals the f64 product with the decoder's weight, rounded once.  Rows of x
    around the 16-row MMA step and the 256 / 128-row CTA tile, rows of W around the 128-row tile, the row length around the
    64-element chunk and the split-K ranges of a cluster (up to 8 CTAs), odd lengths (int4 rows starting in a high nibble)."""
    rng = np.random.default_rng(kind * 100 + DT[dtype] * 10 + 4 * is_signed + 2 * per_channel + with_bias)
    for M, N, K in _shapes(kind):
        data = _lin_data(kind, dtype, N, K, per_channel, is_signed, rng)
        x = _x(rng, (M, K), dtype)
        bias = _x(rng, (N,), dtype) * 4 if with_bias else None
        y = _batched(x, data, kind, N, bias)
        assert y.shape == (M, N) and y.dtype == dtype
        _assert_exact(y, x, _weight(data, kind, dtype, N, K), bias, (M, N, K))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", KIND_DTYPES)
def test_misaligned_inputs_give_the_same_bits(kind, dtype):
    """x at a 4-byte offset and codes at a 1-byte offset take the element-wise loads: same bits as the aligned call."""
    rng = np.random.default_rng(7 + kind)
    for M, N, K in ((17, 33, 64), (40, 129, 1024), (9, 40, 11008)):
        data = _lin_data(kind, dtype, N, K, True, True, rng, exact=False)
        codes, is_signed, scale, zp, quot = data
        x = _x(rng, (M, K), dtype, exact=False)
        bias = _x(rng, (N,), dtype, exact=False)
        args = (kind, is_signed, N, _dev(scale), _dev(zp), _dev(quot), bias)
        aligned = torch.ops.mctq.packed_linear_batched(x, _dev(codes), *args)
        esz = x.element_size()
        xbuf = torch.empty(M * K + 16, dtype=dtype, device="cuda")
        xo = xbuf[4 // esz: 4 // esz + M * K].view(M, K)
        xo.copy_(x)
        cbuf = torch.empty(codes.size + 16, dtype=torch.uint8, device="cuda")
        co = cbuf[1: 1 + codes.size]
        co.copy_(_dev(codes))
        for xa, ca in ((xo, _dev(codes)), (x, co), (xo, co)):
            got = torch.ops.mctq.packed_linear_batched(xa, ca, *args)
            assert np.array_equal(_np_bits(got), _np_bits(aligned)), (M, N, K, xa is xo, ca is co)
        ok, worst = _bound(aligned, x, _weight(data, kind, dtype, N, K), bias)
        assert ok, (M, N, K, worst)


# --------------------------------------------------------------------------------------------- GPU: error bound
@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", [(I4, torch.bfloat16), (I8, torch.bfloat16), (I4, torch.float16), (I8, torch.float32),
                                        (LI4, torch.float32), (LU8, torch.float32)])
def test_error_bound_at_llama_shapes(kind, dtype):
    rng = np.random.default_rng(11 + kind + DT[dtype])
    for M, N, K in ((64, 11008, 4096), (33, 4096, 11008)):
        data = _lin_data(kind, dtype, N, K, True, True, rng, exact=False)
        x = _x(rng, (M, K), dtype, exact=False)
        bias = _x(rng, (N,), dtype, exact=False)
        ok, worst = _bound(_batched(x, data, kind, N, bias), x, _weight(data, kind, dtype, N, K), bias)
        assert ok, (M, N, K, worst)


def _one_hot(kind, N, K, rng):
    """A weight with one nonzero element per row, power-of-two scales: y = x_k * w exactly, whatever x's mantissa."""
    q = np.zeros((N, K), dtype=np.int64)
    cols = rng.integers(0, K, N)
    q[np.arange(N), cols] = 1
    from test_packed_variants import lut_quotients_np, pack_codes
    codes = pack_codes(q, kind)
    scale = (2.0 ** rng.integers(-3, 3, N)).astype(np.float32)
    if kind in LUT_KINDS:
        return (codes, False, scale, None, lut_quotients_np(np.array([0, 128] + [0] * 14), 8, True)), cols
    return (codes, False, scale, np.zeros(N, dtype=np.int32), None), cols


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [I8, I4, LU8, LI4])
def test_f32_x_full_mantissas(kind):
    """f32 x with full 24-bit mantissas across exponents passes through the three bf16 terms exactly (a one-hot weight makes
    every output one product); subnormal x within the bound; NaN / inf rows give the f64 product's pattern."""
    rng = np.random.default_rng(17 + kind)
    M, N, K = 40, 129, 200
    data, cols = _one_hot(kind, N, K, rng)
    mant = rng.integers(1 << 23, 1 << 24, (M, K)).astype(np.float64) * rng.choice([-1.0, 1.0], (M, K))
    x = torch.from_numpy((mant * 2.0 ** rng.integers(-100, 100, (M, K)).astype(np.float64) * 2.0 ** -23).astype(np.float32)).cuda()
    w = _weight(data, kind, torch.float32, N, K)
    _assert_exact(_batched(x, data, kind, N), x, w, None, "24-bit mantissas")
    # subnormal x
    xs = (torch.from_numpy(rng.standard_normal((M, K)).astype(np.float32)) * 2.0 ** -130).cuda()
    ok, worst = _bound(_batched(xs, data, kind, N), xs, w, None)
    assert ok, worst
    # non-finite rows with a dense weight
    data = _lin_data(kind, torch.float32, N, K, True, False, rng)
    w = _weight(data, kind, torch.float32, N, K)
    x = _x(rng, (M, K), torch.float32)
    x[1, 5] = float("nan")
    x[2, 7] = float("inf")
    x[3, 11] = float("-inf")
    x[3, K - 2] = float("inf")
    x[20, 0] = float("inf")
    want, _ = _ref(x, w, None, elementwise=True)
    _same_pattern(_batched(x, data, kind, N), want, "non-finite x")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", [(k, dt) for k in (I8, I4) for dt in (torch.bfloat16, torch.float16)])
def test_non_finite_16bit(kind, dtype):
    """NaN / inf in 16-bit x, and f16 weights that round to +-inf (the decoded value of code 0 included, so that a row tail
    decoded without its mask turns into NaN), reach exactly the outputs the f64 product gives them."""
    rng = np.random.default_rng(5 + kind + DT[dtype])
    for M, N, K in ((20, 33, 1040), (17, 17, 33)):
        data = _lin_data(kind, dtype, N, K, True, True, rng)
        w = _weight(data, kind, dtype, N, K)
        x = _x(rng, (M, K), dtype)
        x[1, 5] = float("nan")
        x[2, 7] = float("inf")
        x[3, 11] = float("-inf")
        want, _ = _ref(x, w, None, elementwise=True)
        _same_pattern(_batched(x, data, kind, N), want, (M, N, K))
    if dtype == torch.float16:
        for K in (63, 65, 100):
            M, N = 17, 24
            data = _lin_data(kind, dtype, N, K, True, False, rng)
            data[2][::3] = 2.0 ** 12 if kind == I8 else 2.0 ** 13
            data[3][::3] = 200 if kind == I8 else 12                    # code 0 decodes to -inf in those rows
            w = _weight(data, kind, dtype, N, K)
            assert np.isinf(w).any() and np.isfinite(w).any()
            x = _x(rng, (M, K), dtype)
            want, _ = _ref(x, w, None, elementwise=True)
            _same_pattern(_batched(x, data, kind, N), want, ("f16 weights at +-inf", K))


# --------------------------------------------------------------------------------------------- GPU: determinism, graphs, guards
@pytest.mark.gpu
def test_deterministic_graph_and_guards():
    rng = np.random.default_rng(23)
    for kind, dtype in ((LI4, torch.float32), (I4, torch.bfloat16)):
        M, N, K = 100, 4097, 11008
        data = _lin_data(kind, dtype, N, K, True, True, rng, exact=False)
        codes, is_signed, scale, zp, quot = data
        pl = ops.PackedLinear(_dev(codes), kind, is_signed, dtype, N, K, _dev(scale), _dev(zp), _dev(quot))
        x = _x(rng, (M, K), dtype, exact=False)
        bias = _x(rng, (N,), dtype, exact=False)
        a, b = pl.batched(x, bias), pl.batched(x, bias)
        assert np.array_equal(_np_bits(a), _np_bits(b))
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            pl.batched(x, bias)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            y = pl.batched(x, bias)
        graph.replay()
        torch.cuda.synchronize()
        assert np.array_equal(_np_bits(y), _np_bits(a))
    # y and bias inside NaN-poisoned buffers, x followed by NaN rows: every guard keeps its bits
    lib = _native.load()
    GAP = 37
    for kind, dtype in KIND_DTYPES:
        for M, N, K in ((17, 17, 33), (255, 129, 1040), (9, 7, 4097)):
            data = _lin_data(kind, dtype, N, K, True, True, rng, lut_k=5 if kind == LI4 else 100)
            codes, is_signed, scale, zp, quot = data
            pl = ops.PackedLinear(_dev(codes), kind, is_signed, dtype, N, K, _dev(scale), _dev(zp), _dev(quot))
            xbuf = torch.full((M + 3, K), float("nan"), dtype=dtype, device="cuda")
            x = _x(rng, (M, K), dtype)
            xbuf[:M] = x
            ybuf = torch.full((M * N + 2 * GAP,), float("nan"), dtype=dtype, device="cuda")
            bbuf = torch.full((N + 2 * GAP,), float("nan"), dtype=dtype, device="cuda")
            bias = _x(rng, (N,), dtype)
            bbuf[GAP: GAP + N] = bias
            before = _np_bits(ybuf).copy(), _np_bits(bbuf).copy(), _np_bits(xbuf).copy()
            qh = quot if quot is None else np.ascontiguousarray(quot, dtype=np.float32)
            rc = lib.mctq_packed_linear_batched(pl._desc_ptr, N, K, xbuf.data_ptr(), DT[dtype], M, bbuf[GAP:].data_ptr(),
                                                ybuf[GAP:].data_ptr(), qh.ctypes.data if qh is not None else None,
                                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0
            torch.cuda.synchronize()
            after = _np_bits(ybuf)
            assert np.array_equal(after[:GAP], before[0][:GAP]) and np.array_equal(after[GAP + M * N:], before[0][GAP + M * N:])
            assert np.array_equal(_np_bits(bbuf), before[1]) and np.array_equal(_np_bits(xbuf), before[2])
            y = ybuf[GAP: GAP + M * N].view(M, N)
            _assert_exact(y, x, _weight(data, kind, dtype, N, K), bias, ("guarded", kind, dtype, M, N, K))


# --------------------------------------------------------------------------------------------- GPU: wrappers
def _batched_wrapper(out_f, in_f, qname, dtype, seed=0):
    m = _wrapped_linear(out_f, in_f, qname, dtype, seed=seed)
    report = m.pack_weights(fused_linear=True, batched_linear=True)
    assert report["weight"]["fused"] and report["weight"]["batched"], report
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("qname,dtype", [("lut16", torch.float32), ("sym4", torch.bfloat16), ("uni8", torch.float16)])
def test_wrapper_row_ranges(qname, dtype, monkeypatch):
    """Batched mode: up to FUSED_LINEAR_MAX_ROWS rows the fused kernel (today's bits), above it up to FUSED_BATCHED_MAX_ROWS
    the batched kernel, above that and for grad / hooks / compilation the exact path."""
    limit = max(FUSED_BATCHED_MAX_ROWS[dtype], 64)
    monkeypatch.setitem(FUSED_BATCHED_MAX_ROWS, dtype, limit)
    m = _batched_wrapper(130, 200, qname, dtype)
    ref = _wrapped_linear(130, 200, qname, dtype)
    ref.pack_weights(fused_linear=True)
    lo = FUSED_LINEAR_MAX_ROWS[dtype]
    st = m._packed
    lin = None
    with torch.no_grad():
        x = torch.randn(lo, 200, device="cuda").to(dtype)
        assert torch.equal(m(x), ref(x))                                             # the fused kernel's bits
        lin = st._lin[1]
        for M in (lo + 1, 33, limit):
            x = torch.randn(M, 200, device="cuda").to(dtype)
            assert torch.equal(m(x), lin.batched(x, m.layer.bias))
        before = _native.launch_count()
        m(torch.randn(2, 3, 10, 200, device="cuda").to(dtype))                      # 60 rows of a 4-D x: one launch
        assert _native.launch_count() - before == 1
        big = torch.randn(limit + 1, 200, device="cuda").to(dtype)
        assert torch.equal(m(big), _exact_path(m, big))
    x = torch.randn(lo + 5, 200, device="cuda").to(dtype)
    xg = x.clone().requires_grad_(True)
    y = m(xg)
    assert y.grad_fn is not None and torch.equal(y.detach(), _exact_path(m, xg).detach())
    calls = []
    h = m.layer.register_forward_hook(lambda mod, i, o: calls.append(1))
    with torch.no_grad():
        assert torch.equal(m(x), _exact_path(m, x)) and calls
    h.remove()
    with torch.no_grad():
        st.batched = False
        assert torch.equal(m(x), _exact_path(m, x))                                  # fused mode alone: exact path
        st.batched = True


@pytest.mark.gpu
def test_wrapper_under_compile_falls_back():
    m = _batched_wrapper(64, 96, "sym4", torch.bfloat16)
    x = torch.randn(20, 96, device="cuda", dtype=torch.bfloat16)
    with torch.no_grad():
        want = _exact_path(m, x)
        got = torch.compile(m, backend="eager", fullgraph=False)(x)
    assert torch.equal(got, want)


@pytest.mark.gpu
def test_round_trips(tmp_path):
    m = _batched_wrapper(130, 200, "lut16", torch.float32)
    x = torch.randn(40, 200, device="cuda")
    with torch.no_grad():
        want = m(x)
        c = copy.deepcopy(m)
        assert c._packed.batched and torch.equal(c(x), want)
        buf = io.BytesIO()
        torch.save(m, buf)
        buf.seek(0)
        loaded = torch.load(buf, weights_only=False)
        assert loaded._packed.batched and torch.equal(loaded(x), want)
        other = _wrapped_linear(130, 200, "lut16", torch.float32, seed=1)
        other.pack_weights(fused_linear=True, batched_linear=True)
        other.load_state_dict(m.state_dict())
        assert torch.equal(other(x), want)
        moved = copy.deepcopy(m).to("cuda")
        assert torch.equal(moved(x), want)


@pytest.mark.gpu
def test_reports_without_batched_are_unchanged():
    a = _wrapped_linear(64, 96, "sym4", torch.bfloat16)
    ra = a.pack_weights(fused_linear=True)
    assert "batched" not in ra["weight"] and "batched_reason" not in ra["weight"]
    assert a._packed.batched is False
    rb = a.pack_weights(fused_linear=True, batched_linear=True)              # on a model packed earlier: switches the mode
    assert rb["weight"]["batched"] and rb["weight"]["batched_reason"] == ""
    conv = mctq.PytorchQuantizationWrapper(torch.nn.Conv2d(3, 4, 1).cuda(),
                                           {"weight": Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 4, True, 0)})
    rc = conv.pack_weights(fused_linear=True, batched_linear=True)
    assert not rc["weight"]["batched"] and "Conv2d" in rc["weight"]["batched_reason"]


@pytest.mark.gpu
def test_memory_of_a_batched_forward(monkeypatch):
    monkeypatch.setitem(FUSED_BATCHED_MAX_ROWS, torch.float32, max(FUSED_BATCHED_MAX_ROWS[torch.float32], 64))
    torch.cuda.synchronize()
    torch.manual_seed(0)
    layers, in_f, out_f = [], 4096, 11008
    for _ in range(2):
        lin = torch.nn.Linear(in_f, out_f, bias=False, device="cuda")
        layers.append(mctq.PytorchQuantizationWrapper(lin, {"weight": _lut_q(16, out_f)}))
        in_f, out_f = out_f, in_f
    model = torch.nn.Sequential(*layers)
    M = 64
    x = torch.randn(M, 4096, device="cuda")
    with torch.no_grad():
        report = pack_model_weights(model, fused_linear=True, batched_linear=True)
        assert all(r["batched"] for rep in report.values() for r in rep.values())
        ops.clear_lut_caches()
        model(x)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        resident = torch.cuda.memory_allocated()
        model(x)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - resident
    activations = M * (4096 + 11008 + 4096) * 4
    assert peak <= activations + (1 << 20), peak


# --------------------------------------------------------------------------------------------- GPU: dependent launches
@pytest.mark.gpu
def test_chain_under_private_stream_orders():
    """Fake-quant emits int8 codes -> batched linear reads them, fake-quant writes x -> batched linear reads it: the opt-in
    overlap orders (key 3 = 2, 3) give the bits of the default order."""
    lib = _native.load()
    dev = "cuda"
    N, K, M = 4096, 4096, 64
    gen = torch.Generator(device=dev).manual_seed(21)
    w_src = torch.empty(N, K, device=dev).uniform_(-1, 1, generator=gen)
    x_src = torch.empty(M, K, device=dev).uniform_(-4, 4, generator=gen)
    big_src = torch.empty(48 << 20, device=dev).uniform_(-4, 4, generator=gen)
    wscale = torch.full((N,), 1.0 / 127, device=dev)
    wzp = torch.zeros(N, dtype=torch.int32, device=dev)
    codes = torch.zeros(N * K, dtype=torch.uint8, device=dev)
    pl = ops.PackedLinear(codes, I8, True, torch.float32, N, K, wscale, wzp, None)
    x, y, big = torch.empty(M, K, device=dev), torch.empty(M, N, device=dev), torch.empty(48 << 20, device=dev)
    one, zero = torch.ones(1, device=dev), torch.zeros(1, dtype=torch.int32, device=dev)
    xs = torch.full((1,), 0.05, device=dev)
    vp = ctypes.c_void_p

    def st():
        return vp(torch.cuda.current_stream().cuda_stream)

    def fq(src, dst, codes_out=None, C=1, inner=1, s=one, zp=zero, qmin=0, qmax=255):
        assert lib.mctq_fq_affine(vp(src.data_ptr()), vp(dst.data_ptr()) if dst is not None else None,
                                  vp(codes_out.data_ptr()) if codes_out is not None else None, src.numel(), 0,
                                  vp(s.data_ptr()), vp(zp.data_ptr()), C, inner, 0, qmin, qmax,
                                  1 if codes_out is not None else 0, st()) == 0

    def sequence():
        codes.zero_()
        for t in (x, y, big):
            t.fill_(float("nan"))
        torch.cuda.synchronize()
        fq(big_src, big, s=xs)
        fq(w_src, None, codes_out=codes, C=N, inner=K, s=wscale, zp=wzp, qmin=-128, qmax=127)
        fq(x_src, x, s=xs)
        assert lib.mctq_packed_linear_batched(pl._desc_ptr, N, K, vp(x.data_ptr()), 0, M, None, vp(y.data_ptr()), None,
                                              st()) == 0
        fq(x_src, x, s=xs)                                         # overwrites the x just read
        torch.cuda.synchronize()
        return [t.clone() for t in (codes, x, y)]

    want = sequence()
    assert not any(bool(torch.isnan(t.float()).any()) for t in want)
    for mode in (2, 3):
        prev = lib.mctq_set_tuning(3, mode)
        try:
            for _ in range(3):
                for a, b in zip(want, sequence()):
                    assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), mode
        finally:
            lib.mctq_set_tuning(3, prev)


@pytest.mark.gpu
def test_opcheck():
    rng = np.random.default_rng(3)
    data = _lin_data(I4, torch.bfloat16, 33, 64, True, True, rng)
    codes, is_signed, scale, zp, quot = data
    x = _x(rng, (20, 64), torch.bfloat16)
    torch.library.opcheck(torch.ops.mctq.packed_linear_batched,
                          (x, _dev(codes), I4, is_signed, 33, _dev(scale), _dev(zp), None, None))


# --------------------------------------------------------------------------------------------- GPU: LUT tables, graphs, devices
@pytest.mark.gpu
def test_lut_ops_capture_in_cuda_graphs():
    """Neither LUT op synchronises once warm: torch.ops.mctq.packed_linear (no host copy at all) and
    packed_linear_batched (its host copy of the quotients is taken by the eager call before capture) replay the eager bits."""
    rng = np.random.default_rng(29)
    N, K = 129, 200
    codes, is_signed, scale, zp, quot = _lin_data(LI4, torch.float32, N, K, True, False, rng)
    args = (_dev(codes), LI4, False, N, _dev(scale), None, _dev(quot), None)
    for op, M in ((torch.ops.mctq.packed_linear, 3), (torch.ops.mctq.packed_linear_batched, 40)):
        x = _x(rng, (M, K), torch.float32)
        want = op(x, *args)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            op(x, *args)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            y = op(x, *args)
        graph.replay()
        torch.cuda.synchronize()
        assert np.array_equal(_np_bits(y), _np_bits(want)), op


def _lut_wrapper(values, out_f, in_f, seed):
    torch.manual_seed(seed)
    lin = torch.nn.Linear(in_f, out_f, device="cuda")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        q = Q.WeightsLUTSymmetricInferableQuantizer(4, [float(v) for v in values], [1.0] * out_f, True, 0, 2, 8)
    m = mctq.PytorchQuantizationWrapper(lin, {"weight": q})
    m.pack_weights(fused_linear=True, batched_linear=True)
    return m


@pytest.mark.gpu
def test_batched_reads_the_loaded_lut_table(monkeypatch):
    """A state_dict brings its own LUT table (the quotient buffer): the batched kernel uses it like the fused kernel and the
    exact path, not the table of the receiving wrapper's quantizer."""
    monkeypatch.setitem(FUSED_BATCHED_MAX_ROWS, torch.float32, max(FUSED_BATCHED_MAX_ROWS[torch.float32], 64))
    a = _lut_wrapper(range(-128, 128, 16), 130, 200, 0)
    b = _lut_wrapper(range(-120, 120, 15), 130, 200, 1)
    x = torch.randn(40, 200, device="cuda")
    with torch.no_grad():
        b(x)                                                     # b's batched state is built from its own table first
        b.load_state_dict(a.state_dict())
        assert torch.equal(b(x), a(x))
        w = b.get_quantized_weights()["weight"].double().cpu().numpy()          # rebuilt from the loaded codes and table
        ok, worst = _bound(b(x), x, w, b.layer.bias)
        assert ok, worst


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_batched_on_a_second_device():
    """The launch settings (dynamic shared memory above 48 KB) hold on every device, not only on the first one used."""
    rng = np.random.default_rng(31)
    N, K, M = 300, 1040, 200
    data = _lin_data(LI4, torch.float32, N, K, True, False, rng)
    codes, is_signed, scale, zp, quot = data
    w = _weight(data, LI4, torch.float32, N, K)
    for dev in ("cuda:0", "cuda:1"):
        x = _x(rng, (M, K), torch.float32).to(dev)
        t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)   # noqa: E731
        with torch.cuda.device(dev):
            y = torch.ops.mctq.packed_linear_batched(x, t(codes), LI4, False, N, t(scale), None, t(quot), None)
        _assert_exact(y, x, w, None, dev)
