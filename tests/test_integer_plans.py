"""The integer kernels on the launch plans that real layers reach.  The host planners pick a row tile nt, a split-K S and
launches over row ranges for the integer GEMMs (launch_igemm / tc_launch_rows), and a tile of slots and output pixels for
the depthwise kernel (dw_plan).  Every case here is checked bit for bit against the references of the integer test files,
and each test asserts the plan it covers, read from the profiler's trace (GEMMs) or from mctq_packed_dwconv2d_i8_plan
(depthwise), so that the coverage does not rest on guessing occupancy:
  long rings       S = 1 with at least 17 chunks of 128 codes per CTA: more than two wraps of the deepest (8-stage) ring,
                   for every producer variant (TMA int8, int4 / LUT producers, the 16-channel, narrow and padded gathers)
                   in both row-tile regimes (nt = 16 and nt = 240 / 256)
  every split S    S = 1 .. 8, uneven chunk splits, conv ranks with fewer chunks than the gather keeps in flight
  tile edges       row and feature counts on both sides of the tile sizes, all output dtypes and weight formats
  two launches     more than 65535 row tiles: the second launch's rows (m0 > 0), compared on both sides of the boundary
  depthwise        every depthwise layer of MobileNetV2, MobileNetV3-Large and EfficientNet-B0 at 224 x 224, and each
                   class of the planner (slot groups, partial tiles, shrink steps, the largest windows)"""
import ctypes
import functools
import json
import os
import tempfile

import pytest
import torch

from mct_quantizers_b200 import _native, ops

from test_integer_conv import _conv_case, conv_reference
from test_integer_depthwise import _dw_case
from test_integer_linear import _gemm_case, reference_on_device
from test_integer_lut import _conv_case as _lut_conv_case
from test_integer_lut import _lin_case as _lut_lin_case
from test_integer_pad import _conv_pad_case

I8, I4, LI4, LU8 = _native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4, _native.PACK_LUT_I4, _native.PACK_LUT_U8
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
_TAG = {torch.float32: _native.F32, torch.bfloat16: _native.BF16, torch.float16: _native.F16}
FMTS = ["i8", "i4s", "i4u", "lut4", "lut8"]
_LUT = {"lut4": LI4, "lut8": LU8}
_GEMM_KERNELS = ("packed_igemm_kernel", "packed_iconv_kernel", "packed_iconv_narrow_kernel")
_ROWS_PER_LAUNCH = 65535            # row tiles per launch (grid.y)


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


@pytest.fixture(autouse=True)
def _release_device_memory():
    """Return the cached device memory of each case (up to a few GB) once it is done: the GPU may be shared."""
    yield
    if torch.cuda.is_initialized():
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ plan observation
def _launches(fn):
    """(fn(), [(kernel, grid.x, grid.y)] of the integer GEMM launches fn makes, in issue order), read from the trace of
    torch.profiler.  A launch without a grid in the trace fails the test."""
    from torch.profiler import ProfilerActivity, profile
    lib = _native.load()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        n0 = lib.mctq_launch_count()
        out = fn()
        torch.cuda.synchronize()
        launched = lib.mctq_launch_count() - n0
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    found = []
    for e in sorted(events, key=lambda e: e.get("ts", 0)):
        name = e.get("name", "")
        if e.get("cat") != "kernel" or not any(k in name for k in _GEMM_KERNELS):
            continue
        grid = e.get("args", {}).get("grid")
        assert grid is not None and len(grid) == 3, f"the trace gives no grid for {name}"
        found.append((name, int(grid[0]), int(grid[1])))
    kernels = [(e.get("cat"), e.get("name", "")[:60]) for e in events if "kernel" in str(e.get("cat", "")).lower()]
    assert found, \
        f"no integer GEMM launch in the trace: {launched} library launches, {len(events)} events, {kernels[:8]}"
    return out, found


def _plan(fn, N):
    """(fn(), S, row tiles of each launch, kernel names): the split S = grid.x / ceil(N / 128), one value for every launch."""
    out, found = _launches(fn)
    tiles = -(-N // 128)
    assert all(gx % tiles == 0 for _, gx, _ in found), (found, N)
    splits = {gx // tiles for _, gx, _ in found}
    assert len(splits) == 1, found
    return out, splits.pop(), [gy for _, _, gy in found], {n for n, _, _ in found}


def _chunks(K):
    return -(-K // 128)


# ------------------------------------------------------------------------------------------------ case runners
def _linear(fmt, M, N, K, seed, dtype=torch.float32):
    """One bit-exact linear case of weight format fmt (the builders of test_integer_linear / test_integer_lut: the
    reference on the device, NaN outside the output view)."""
    xs = seed % 2 == 0
    zx = (5, -7, 0)[seed % 3] if xs else (200, 0, 128)[seed % 3]
    if fmt in _LUT:
        return _lut_lin_case(M, N, K, _LUT[fmt], per_channel=seed % 2 == 1, pot=seed % 3 == 0, x_signed=xs, zx=zx,
                             with_bias=seed % 4 != 3, seed=seed)
    return _gemm_case(M, N, K, I8 if fmt == "i8" else I4, fmt != "i4u", per_channel=seed % 2 == 0,
                      zw_nonzero=seed % 3 != 0, x_signed=xs, zx=zx, dtype=dtype, with_bias=seed % 4 != 3, seed=seed)


def _conv(fmt, N, Cin, H, W, Cout, k, seed, dtype=torch.float32, stride=(1, 1), dilation=(1, 1), padding=(1, 1, 1, 1),
          channels_last=None):
    """One bit-exact conv case (the builders of test_integer_conv / test_integer_lut: NHWC codes fed to the GEMM, the
    reference, then the C ABI into the middle of a NaN buffer)."""
    xs = seed % 2 == 1
    zx = (3, -7, 0)[seed % 3] if xs else (200, 0, 128)[seed % 3]
    cl = seed % 4 < 2 if channels_last is None else channels_last
    if fmt in _LUT:
        return _lut_conv_case(N, Cin, H, W, Cout, k, stride, dilation, padding, _LUT[fmt], per_channel=seed % 2 == 0,
                              pot=seed % 3 == 1, x_signed=xs, zx=zx, channels_last=cl, seed=seed)
    return _conv_case(N, Cin, H, W, Cout, k, stride, dilation, padding, I8 if fmt == "i8" else I4, fmt != "i4u",
                      per_channel=seed % 2 == 0, zw_nonzero=seed % 3 != 2, x_signed=xs, zx=zx, dtype=dtype,
                      with_bias=seed % 4 != 1, channels_last=cl, seed=seed)


# ------------------------------------------------------------------------------------------------ long rings
# (what, runner, N, the kernel's row length K, row tiles (nt = 16: one tile of <= 16 rows))
def _long_cases():
    cases = []
    for i, fmt in enumerate(FMTS):
        # nt = 16: one row tile, 300 feature tiles (more than two CTAs per SM fit), K = 2304: 18 chunks
        cases.append((f"linear {fmt} nt=16", lambda fmt=fmt, i=i: _linear(fmt, 16, 38400, 2304, 10 + i), 38400, 2304))
        cases.append((f"conv {fmt} nt=16", lambda fmt=fmt, i=i: _conv(fmt, 1, 256, 4, 4, 38400, (3, 3), 20 + i), 38400,
                      2304))
        # full row tiles: 4 x 40 (linear) and 49 x 4 (ResNet-18 layer4 3x3 at batch 256, K = 4608: 36 chunks) CTAs; one
        # int4 signedness each
        if fmt != "i4u":
            cases.append((f"linear {fmt} full rows", lambda fmt=fmt, i=i: _linear(fmt, 1024, 5120, 2304, 30 + i), 5120,
                          2304))
        if fmt != "i4s":
            cases.append((f"conv {fmt} resnet18 layer4",
                          lambda fmt=fmt, i=i: _conv(fmt, 256, 512, 7, 7, 512, (3, 3), 40 + i, dtype=DTYPES[i % 3]),
                          512, 4608))
    # the narrow gather over 19 x 64 x 64 = 77824 output pixels: Cp = 4 with a 24 x 24 window (K = 2304), Cp = 8 with
    # 17 x 17 (K = 2312 + a row tail: 2320, 2336 for 4-bit codes)
    for i, (cin, kk, kind) in enumerate(((3, 24, I8), (6, 17, I8), (3, 24, LI4), (6, 17, LU8))):
        K = ops.conv_code_pitch(cin, kk, kk, kind)[1]
        cases.append((f"narrow Cin={cin} {kk}x{kk} kind={kind}",
                      lambda cin=cin, kk=kk, kind=kind, i=i: _conv_pad_case(
                          19, cin, 63 + kk, 63 + kk, 48, (kk, kk), (1, 1), (1, 1), (0, 0, 0, 0), kind, i % 3 != 1,
                          i % 2 == 0, (0, 128, -7, 9)[i], DTYPES[i % 3], i % 2 == 1, False, 50 + i), 48, K))
    # the padded wide gather: Cin = 200 -> Cp = 208, a 4 x 4 window: K = 3328 (26 chunks), nt = 16
    cases.append(("padded Cin=200", lambda: _conv_pad_case(1, 200, 4, 4, 38400, (4, 4), (1, 1), (1, 1), (2, 1, 2, 1), I8,
                                                           True, False, 9, torch.bfloat16, True, False, 60), 38400, 3328))
    return cases


_LONG = _long_cases()


@pytest.mark.gpu
@pytest.mark.parametrize("ci", range(len(_LONG)), ids=[c[0].replace(" ", "-") for c in _LONG])
def test_long_rings(ci):
    what, run, N, K = _LONG[ci]
    _, S, rows, names = _plan(run, N)
    assert S == 1 and _chunks(K) >= 17, (what, S, _chunks(K))
    assert len(set(rows)) == 1 and len(names) == 1, (rows, names)
    if "nt=16" in what or "padded" in what:
        assert rows[0] == 1
    if "narrow" in what:
        assert all("narrow" in n for n in names)


# ------------------------------------------------------------------------------------------------ every split S
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_every_split(fmt):
    """Linear M = 16, N = 128 T, K = 1168 (1184 for 4-bit codes): 10 chunks over T feature tiles.  Whether one or two CTAs
    fit an SM, the T below give every S from 2 to 8 (mostly not dividing 10: uneven chunk ranges), and T = 300 gives
    S = 1.  One kernel per format (one dtype), so that the CTAs per SM stay the same over the sweep."""
    seen = set()
    K = 1184 if fmt in ("i4s", "i4u", "lut4") else 1168
    dtype = DTYPES[FMTS.index(fmt) % 3]
    for i, T in enumerate((18, 21, 24, 29, 37, 42, 49, 59, 74, 98, 148, 300)):
        _, S, rows, _ = _plan(lambda: _linear(fmt, 16, 128 * T, K, 100 + i, dtype), 128 * T)
        assert rows == [1] * len(rows) and 1 <= S <= min(8, _chunks(K))
        seen.add(S)
    assert seen >= set(range(1, 9)), sorted(seen)


@pytest.mark.gpu
def test_conv_ranks_with_few_chunks():
    """Split-K conv where ranks hold 1 or 2 chunks, fewer than the kIConvAhead = 3 stages the gather keeps in flight, and
    feature counts that are not multiples of 128."""
    # (fmt, N, Cin, H, W, Cout): K = Cin * 9
    for i, (fmt, N, Cin, H, W, Cout) in enumerate((("i8", 1, 16, 4, 4, 128), ("i4s", 1, 64, 4, 4, 300),
                                                   ("lut8", 1, 32, 4, 4, 383), ("i8", 1, 128, 4, 4, 129),
                                                   ("lut4", 1, 128, 4, 4, 1), ("i4u", 1, 32, 3, 5, 255))):
        K = Cin * 9
        _, S, _, _ = _plan(lambda: _conv(fmt, N, Cin, H, W, Cout, (3, 3), 200 + i, DTYPES[i % 3]), Cout)
        nch = _chunks(K)
        per_rank = [nch * (r + 1) // S - nch * r // S for r in range(S)]
        assert S > 1 and min(per_rank) < 3, (fmt, Cin, Cout, S, per_rank)


# ------------------------------------------------------------------------------------------------ row and feature edges
_MS = [1, 15, 16, 17, 255, 256, 257, 4097]
_NS = [1, 127, 128, 129, 383]
# conv images of exactly M output pixels (3x3, padding 1): N, H, W
_CONV_M = {1: (1, 1, 1), 15: (1, 3, 5), 16: (1, 4, 4), 17: (1, 1, 17), 255: (1, 15, 17), 256: (1, 16, 16), 257: (1, 1, 257),
           4097: (1, 17, 241)}
_EDGE_CONFIGS = [(fmt, dt) for fmt in FMTS for dt in DTYPES if fmt not in _LUT or dt == torch.float32]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,dtype", _EDGE_CONFIGS)
def test_row_and_feature_edges(fmt, dtype):
    """Every M against two of the N (every N against several M) for linear; every M for conv, N rotating.  M = 257 runs
    nt = 144: 9 column blocks of 16 rows, an odd number shared by two epilogue warps."""
    rows_seen = set()
    for i, M in enumerate(_MS):
        for j in (0, 2):
            N = _NS[(i + j) % len(_NS)]
            _, S, rows, _ = _plan(lambda: _linear(fmt, M, N, 288, 1000 * FMTS.index(fmt) + 10 * i + j, dtype), N)
            rows_seen.update(rows)
        n, H, W = _CONV_M[M]
        N = _NS[i % len(_NS)]
        _conv(fmt, n, 32, H, W, N, (3, 3), 2000 * FMTS.index(fmt) + i, dtype, channels_last=i % 2 == 0)
    assert 1 in rows_seen and max(rows_seen) >= 17, rows_seen               # M = 4097: 17 row tiles of 256 (18 of 240)


# ------------------------------------------------------------------------------------------------ two launches
# These cases hold 16.8 million rows.  The codes are int8 and the float64 reference is computed a slice at a time, so that
# a case takes about 2 GB of device memory (the whole-output reference would take 10-15 GB of temporaries).
_REF_ROWS = 1 << 21


def _library_launches(fn):
    """(fn(), the number of kernel launches the library made in fn), from its own counter (mctq_launch_count).  The
    launches of these cases run for milliseconds, and on a GPU shared with other processes the profiler was seen to lose
    the records of such kernels, so the two-launch cases count launches here instead of reading the trace."""
    lib = _native.load()
    torch.cuda.synchronize()
    n0 = lib.mctq_launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, lib.mctq_launch_count() - n0


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["i8", "lut8"])
def test_linear_rows_over_two_launches(fmt):
    """M = 65535 nt + 1 rows: the second launch holds the last row (m0 = 65535 nt), read from the TMA row coordinate and
    x_rowsum and written at its own row."""
    lut = fmt == "lut8"
    nt = 240 if lut else 256
    M, K, N = _ROWS_PER_LAUNCH * nt + 1, 16, 16
    dtype = torch.float32 if lut else torch.bfloat16
    g = torch.Generator().manual_seed(nt)
    gd = torch.Generator(device="cuda").manual_seed(nt)
    xq = torch.randint(-128, 128, (M, K), generator=gd, device="cuda", dtype=torch.int8)
    f = (torch.rand(N, generator=g) * 0.01 + 0.001).cuda()
    bias = (torch.randn(N, generator=g) * 3).to(dtype).cuda()
    if lut:
        table = torch.randint(-128, 128, (256,), generator=g, dtype=torch.int32)
        idx = torch.randint(0, 256, (N, K), generator=g, dtype=torch.int32)
        lin = ops.IntegerLinear.from_parts(ops.pack_weight_codes(idx, LU8, False).cuda(), LU8, False, dtype, N, K, f, None,
                                           None, 3, lut_values=table.tolist())
        qw, zw, rowsum = table[idx.long()].cuda(), torch.zeros(1, dtype=torch.int32, device="cuda"), None
    else:
        qw = torch.randint(-128, 128, (N, K), generator=g, dtype=torch.int32)
        zw = torch.randint(-128, 128, (N,), generator=g, dtype=torch.int32)          # nonzero: x_rowsum is read
        lin = ops.IntegerLinear.from_parts(ops.pack_weight_codes(qw, I8, True).cuda(), I8, True, dtype, N, K, f, zw.cuda(),
                                           None, 3)
        qw, zw, rowsum = qw.cuda(), zw.cuda(), xq.sum(1, dtype=torch.int32)
    poison = torch.full((M, N), float("nan"), dtype=dtype, device="cuda")
    _, launched = _library_launches(lambda: lin.gemm(xq, rowsum, bias, out=poison))
    assert launched == 2                                 # 65535 row tiles of nt rows, then the last row
    ref = lambda r0, r1: reference_on_device(xq[r0:r1], 3, qw, zw, f, bias.float(), dtype)    # noqa: E731
    edge = _ROWS_PER_LAUNCH * nt
    assert torch.equal(_bits(poison[edge - 3:]), _bits(ref(edge - 3, M)))     # both sides of the launch boundary
    for r0 in range(0, M, _REF_ROWS):
        r1 = min(M, r0 + _REF_ROWS)
        assert torch.equal(_bits(poison[r0:r1]), _bits(ref(r0, r1))), r0


@pytest.mark.gpu
def test_conv_rows_over_two_launches():
    """A 1x1 conv, Cin = Cout = 16, over 1340 x 112 x 112 = 16808960 pixels written as NCHW planes: the second launch
    starts at pixel 65535 * 256 = 16776960, inside image 1337, so its image index and plane offsets come from m0 > 0."""
    N, C, H, W, nt = 1340, 16, 112, 112, 256
    M = N * H * W
    dtype, zx = torch.float16, -5
    g = torch.Generator().manual_seed(7)
    gd = torch.Generator(device="cuda").manual_seed(7)
    qx = torch.randint(-128, 128, (N, C, H, W), generator=gd, device="cuda", dtype=torch.int8)
    xq = qx.permute(0, 2, 3, 1).contiguous()
    qw = torch.randint(-128, 128, (C, C, 1, 1), generator=g, dtype=torch.int32)
    zw = torch.randint(-128, 128, (C,), generator=g, dtype=torch.int32)
    f = (torch.rand(C, generator=g) * 0.01 + 0.001).cuda()
    bias = (torch.randn(C, generator=g) * 3).to(dtype).cuda()
    codes = ops.pack_weight_codes(qw.reshape(C, C), I8, True).cuda()
    conv = ops.IntegerConv2d.from_parts(codes, I8, True, dtype, C, C, (1, 1), (1, 1), (1, 1), (0, 0, 0, 0), f, zw.cuda(),
                                        None, zx)
    sx = ops.conv_window_sums(qx.sum(1, dtype=torch.int32).reshape(-1), N, H, W, C, (1, 1), (1, 1), (1, 1), (0, 0, 0, 0), zx)
    canary = torch.full((M * C + 64,), float("nan"), dtype=dtype, device="cuda")
    out = canary[32:32 + M * C]
    geo = _native.MctqConv2dGeom(N, H, W, C, H, W, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0)

    def call():
        return _native.load().mctq_packed_conv2d_i8(conv._w._desc_ptr, ctypes.addressof(geo), C, xq.data_ptr(), 1, zx,
                                                    sx.data_ptr(), conv.w_rowsum.data_ptr(), conv.factor.data_ptr(),
                                                    bias.data_ptr(), _TAG[dtype], out.data_ptr(), 1,
                                                    torch.cuda.current_stream().cuda_stream)
    rc, launched = _library_launches(call)
    _native.check(rc, "mctq_packed_conv2d_i8")
    assert launched == 2                                 # 65535 row tiles of 256 pixels, then 125 tiles
    assert torch.isnan(canary[:32]).all() and torch.isnan(canary[32 + M * C:]).all()
    qw, zw = qw.cuda(), zw.cuda()
    ref = lambda b0, b1: conv_reference(qx[b0:b1], zx, qw, zw, f, bias, (1, 1), (1, 1), (0, 0, 0, 0),   # noqa: E731
                                        dtype).reshape(b1 - b0, C, H * W)
    y = out.view(N, C, H * W)
    b, p = divmod(_ROWS_PER_LAUNCH * nt, H * W)
    assert torch.equal(_bits(y[b, :, p - 3:p + 3]), _bits(ref(b, b + 1)[0, :, p - 3:p + 3]))   # both sides of the boundary
    assert torch.equal(_bits(y[N - 1, :, -3:]), _bits(ref(N - 1, N)[0, :, -3:]))
    step = _REF_ROWS // (H * W)
    for b0 in range(0, N, step):
        b1 = min(N, b0 + step)
        assert torch.equal(_bits(y[b0:b1]), _bits(ref(b0, b1))), b0


# ------------------------------------------------------------------------------------------------ depthwise
@functools.lru_cache(maxsize=None)
def _production_dw_layers():
    """Every depthwise Conv2d of MobileNetV2, MobileNetV3-Large and EfficientNet-B0 at 224 x 224, with its input size:
    (C, H, W, m, kernel, stride, dilation, padding (pt, pb, pl, pr)), collected with forward hooks on the CPU."""
    tv = pytest.importorskip("torchvision")
    found = set()
    for name in ("mobilenet_v2", "mobilenet_v3_large", "efficientnet_b0"):
        with torch.device("meta"):                       # shapes only: no weights are initialised, nothing is computed
            model = getattr(tv.models, name)(weights=None).eval()
        hooks = [m.register_forward_hook(lambda mod, a, y: found.add(
                     (mod.in_channels, a[0].shape[2], a[0].shape[3], mod.out_channels // mod.in_channels, mod.kernel_size,
                      mod.stride, mod.dilation, ops.conv_padding(mod))))
                 for m in model.modules() if isinstance(m, torch.nn.Conv2d) and m.groups == m.in_channels > 1]
        with torch.no_grad():
            model(torch.zeros(1, 3, 224, 224, device="meta"))
        for h in hooks:
            h.remove()
    return sorted(found)


def _dw_run(i, N, C, H, W, m, k, stride, dilation, padding, nhwc, dtype, kind=None):
    """One bit-exact depthwise case (test_integer_depthwise's builder: dw_reference, a NaN buffer around the C-ABI output);
    the weight format, zero points and per-channel / per-tensor parameters rotate with i.  Returns the plan."""
    kinds = [I8, I4, LI4, LU8] if dtype == torch.float32 else [I8, I4]
    kind = kinds[i % len(kinds)] if kind is None else kind
    xs = i % 3 != 1
    zx = (0, -7, 4)[i % 3] if xs else (0, 128, 255)[i % 3]
    _dw_case(N, C, H, W, m, k, stride, dilation, padding, kind, i % 2 == 0, per_channel=i % 4 < 2, zw_nonzero=i % 3 != 0,
             x_signed=xs, zx=zx, dtype=dtype, with_bias=i % 5 != 4, nhwc=nhwc, seed=3000 + i,
             lut_k=16 if kind == LI4 else (256, 200, 7)[i % 3])
    plan = ops.dwconv_plan(N, C, H, W, C * m, k, stride, dilation, padding, nhwc)
    assert plan is not None
    return plan


def test_production_dw_layers_collected():
    layers = _production_dw_layers()
    ks = {l[4] for l in layers}
    assert ks == {(3, 3), (5, 5)} and {l[5] for l in layers} == {(1, 1), (2, 2)}
    assert max(l[1] for l in layers) == 112 and min(l[1] for l in layers) == 7 and max(l[0] for l in layers) == 1152


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_production_depthwise(dtype):
    """Every production depthwise geometry at batch 2, both layouts, the weight formats rotating (LUT formats in f32)."""
    strided_multi_row = set()
    for i, (C, H, W, m, k, stride, dilation, padding) in enumerate(_production_dw_layers()):
        for nhwc in (False, True):
            plan = _dw_run(2 * i + nhwc + 7 * DTYPES.index(dtype), 2, C, H, W, m, k, stride, dilation, padding, nhwc, dtype)
            Ho, _ = ops.conv_output_hw(H, W, k, stride, dilation, padding)
            if stride[0] == 2 and Ho > plan["TH"]:
                strided_multi_row.add(nhwc)
    assert strided_multi_row == {False, True}                               # ty > 0 at stride 2 in both layouts


# (N, C, H, W, m, kernel, stride, dilation, padding, nhwc, the planner classes the case must reach)
_DW_CLASSES = [
    (2, 672, 14, 14, 1, (5, 5), (1, 1), (1, 1), (2, 2, 2, 2), False, {"nchw S>1 partial group", "group crosses images",
                                                                     "generic kernel"}),
    (2, 24, 150, 150, 1, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), False, {"S=1 partial tiles stride 1", "3x3"}),
    (2, 8, 150, 150, 1, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1), False, {"S=1 partial tiles stride 2"}),
    (3, 16, 20, 21, 1, (3, 3), (1, 1), (1, 1), (1, 1, 1, 1), True, {"nhwc C<32"}),
    (2, 72, 28, 28, 2, (3, 3), (2, 2), (1, 1), (1, 1, 1, 1), True, {"nhwc C%32", "m>1 nhwc"}),
    (2, 10, 17, 19, 3, (5, 5), (1, 2), (1, 1), (2, 2, 2, 2), False, {"m>1 nchw", "group crosses images"}),
    (1, 40, 8, 8, 1, (3, 3), (1, 1), (30, 30), (30, 30, 30, 30), False, {"shrink TH", "shrink S"}),
    (1, 1, 300, 300, 1, (3, 3), (1, 1), (100, 100), (100, 100, 100, 100), False, {"shrink TW"}),
    (1, 2, 225, 225, 1, (3, 3), (1, 1), (112, 112), (0, 0, 0, 0), False, {"largest 3x3 window"}),
    (1, 2, 225, 225, 1, (3, 3), (1, 1), (112, 112), (0, 0, 0, 0), True, {"largest 3x3 window"}),
    (1, 2, 1, 25597, 1, (1, 25597), (1, 1), (1, 1), (0, 0, 0, 0), False, {"largest row window"}),
]


def _dw_classes(N, C, H, W, m, k, stride, dilation, padding, nhwc, p):
    """The planner classes a plan p of this geometry falls in."""
    Ho, Wo = ops.conv_output_hw(H, W, k, stride, dilation, padding)
    S, TH, TW = p["S"], p["TH"], p["TW"]
    out = {"3x3" if tuple(k) == (3, 3) else "generic kernel"}
    if m > 1:
        out.add("m>1 nhwc" if nhwc else "m>1 nchw")
    if nhwc:
        out.update({"nhwc C<32"} if C < 32 else {"nhwc C%32"} if C % 32 else set())
    elif S > 1:
        planes = N * C
        if planes % S:
            out.add("nchw S>1 partial group")
        if any(g * S // C != (min(g * S + S, planes) - 1) // C for g in range(-(-planes // S))):
            out.add("group crosses images")
    if S == 1 and Ho % TH and Wo % TW and Ho > TH and Wo > TW:
        out.add(f"S=1 partial tiles stride {stride[0]}")
    # the hand-worked shrinks of test_integer_depthwise.test_plan_query
    if (S, TH, TW) == (16, 1, 8) and tuple(dilation) == (30, 30):
        out.update({"shrink TH", "shrink S"})
    if (S, TH, TW) == (1, 1, 32) and tuple(dilation) == (100, 100):
        out.add("shrink TW")
    if (TH, TW) == (1, 1) and (tuple(dilation) == (112, 112) or tuple(k) == (1, 25597)):
        out.add("largest 3x3 window" if tuple(k) == (3, 3) else "largest row window")
    return out


@pytest.mark.gpu
def test_depthwise_planner_classes():
    reached = set()
    for i, (N, C, H, W, m, k, st, dil, pad, nhwc, want) in enumerate(_DW_CLASSES):
        dtype = DTYPES[i % 3]
        p = _dw_run(i, N, C, H, W, m, k, st, dil, pad, nhwc, dtype)
        got = _dw_classes(N, C, H, W, m, k, st, dil, pad, nhwc, p)
        assert want <= got, (i, p, got)
        reached |= got
    assert reached >= set().union(*(c[-1] for c in _DW_CLASSES)) | {"3x3", "generic kernel"}
