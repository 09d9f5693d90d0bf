"""Parity of the CUDA path (through the public quantizer API and through the raw C ABI) against
  (a) the golden fixtures generated from the unmodified reference, and
  (b) the CPU oracle (oracle/mctq_oracle.c) on seeded inputs, including ragged sizes, slices and large tensors.
Bit-exact everywhere: f32 values, bf16/f16 values, integer codes and LUT indices.
"""
import ctypes

import numpy as np
import pytest
import torch

import golden_util as G
import oracle

pytestmark = pytest.mark.gpu

CASES = G.case_names()
DEV = "cuda:0"


@pytest.fixture(scope="module")
def Q():
    from mct_quantizers_b200.pytorch import quantizers
    return quantizers


@pytest.fixture(scope="module")
def lib():
    from mct_quantizers_b200 import _native
    return _native.load()


def _vp(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# ------------------------------------------------------------------------------------------- golden fixtures
@pytest.mark.parametrize("name", CASES)
def test_quantizer_matches_reference_fixture(name, Q):
    """Public API on a CUDA tensor == output of the unmodified reference on CPU torch (bitwise)."""
    case = G.get_case(name)
    q = getattr(Q, case["cls"])(**case["args"])
    x = G.to_torch(case["x"], case["x_dtype"], DEV)
    y = q(x)
    assert str(y.dtype).replace("torch.", "") == case["y_dtype"]
    assert tuple(y.shape) == tuple(case["shape"])
    got = G.from_torch(y)
    assert G.bits_equal(got, case["y"]), G.mismatch_report(got, case["y"], case["x"])


@pytest.mark.parametrize("name", [n for n in CASES if n.startswith(("wl_", "al_"))])
def test_lut_indices_match_reference_fixture(name, lib):
    """LUT index emission (uint8 and packed 4-bit) == argmin assignment re-derived with the reference's helper."""
    from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
    case = G.get_case(name)
    p = G.derive_params(case)
    x = G.to_torch(case["x"], case["x_dtype"], DEV).contiguous()
    n = x.numel()
    table = lut_search_table(p["lut"], p["bw"], p["signed"]).to(DEV)
    K = int(p["lut"].size)
    want = case["idx"].reshape(-1)
    for mode in (1, 2):
        if mode == 2 and K > 16:
            continue
        idx = torch.full(((n if mode == 1 else (n + 1) // 2) + 8,), 0xEE, dtype=torch.uint8, device=DEV)
        y = torch.empty(n, dtype=torch.float32, device=DEV)
        if p["act"]:
            d = np.float32(np.float64(p["thr"]) + np.float64(p["eps"]))
            rc = lib.mctq_fq_lut_scalar(_vp(x), _vp(y), _vp(idx), n, G.DT_TAG[case["x_dtype"]], _vp(table), K, float(d),
                                        float(np.float32(p["thr"])), int(case["x_dtype"] != "float32"), mode, _stream())
        else:
            thr = torch.from_numpy(p["thr"]).to(DEV)
            rc = lib.mctq_fq_lut(_vp(x), _vp(y), _vp(idx), n, G.DT_TAG[case["x_dtype"]], _vp(table), K, _vp(thr), p["C"],
                                 p["inner"], 0, float(np.float32(p["eps"])), mode, _stream())
        assert rc == 0
        torch.cuda.synchronize()
        got = idx.cpu().numpy()
        if mode == 1:
            assert np.array_equal(got[:n].astype(np.int32), want)
            assert (got[n:] == 0xEE).all()
        else:
            nb = (n + 1) // 2
            lo, hi = got[:nb] & 0xF, got[:nb] >> 4
            un = np.stack([lo, hi], 1).reshape(-1)[:n].astype(np.int32)
            assert np.array_equal(un, want)
            assert (got[nb:] == 0xEE).all()
        assert G.bits_equal(y.cpu().numpy().reshape(case["y"].shape), case["y"])


@pytest.mark.parametrize("name", [n for n in CASES if n.startswith("wl_")])
def test_prepared_lut_indices_match_reference_fixture(name):
    """Index emission through the operator (prepared per-channel decision tables) == reference argmin assignment."""
    from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
    case = G.get_case(name)
    p = G.derive_params(case)
    a = case["args"]
    x = G.to_torch(case["x"], case["x_dtype"], DEV)
    table = lut_search_table(p["lut"], p["bw"], p["signed"])
    K = int(p["lut"].size)
    thr = torch.from_numpy(p["thr"]).to(DEV)
    want = case["idx"].reshape(-1)
    n = x.numel()
    per_channel = bool(a["per_channel"])
    axis = a.get("channel_axis") or 0
    idx8 = torch.ops.mctq.lut_indices(x, table, K, thr, per_channel, axis, p["eps"], 1)
    assert np.array_equal(idx8.cpu().numpy().reshape(-1).astype(np.int32), want)
    if K <= 16:
        idx4 = torch.ops.mctq.lut_indices(x, table, K, thr, per_channel, axis, p["eps"], 2).cpu().numpy()
        un = np.stack([idx4 & 0xF, idx4 >> 4], 1).reshape(-1)[:n].astype(np.int32)
        assert np.array_equal(un, want)


def test_prepared_lut_special_inputs(Q):
    """NaN -> LUT index 0 (argmin over NaN distances), +-inf saturate, huge / tiny magnitudes; prepared == generic kernel."""
    lut = [25.0, -100.0, 0.0, 127.0, -128.0, 64.0, -7.0, 3.0]           # unsorted: index 0 is not the smallest
    thr = [0.7, 1e-3, 30.0]
    q = Q.WeightsLUTSymmetricInferableQuantizer(3, lut, thr, True, 0, 2)
    row = torch.tensor([float('nan'), float('inf'), -float('inf'), 3e38, -3e38, 1e-38, -1e-38, 0.0, -0.0, 0.35, float('nan'), 0.1],
                       dtype=torch.float32)
    x = torch.stack([row, row * 1e-3, row * 40]).to(DEV)
    y = q(x.clone())
    y0 = (torch.tensor(lut[0]) / 128) * torch.tensor(thr, dtype=torch.float32)
    assert torch.equal(y[:, 0].cpu(), y0) and torch.equal(y[:, 10].cpu(), y0)
    top = (torch.tensor(127.0) / 128) * torch.tensor(thr, dtype=torch.float32)
    bot = (torch.tensor(-128.0) / 128) * torch.tensor(thr, dtype=torch.float32)
    assert torch.equal(y[:, 1].cpu(), top) and torch.equal(y[:, 2].cpu(), bot)
    finite = torch.isfinite(x)
    want = oracle.fq_lut(np.nan_to_num(x.cpu().numpy(), nan=0.0, posinf=3e38, neginf=-3e38), oracle.F32, np.asarray(lut, np.float32),
                         np.asarray(thr, np.float32), 3, 12, 8, True, 1e-8)
    assert np.array_equal(y.cpu().numpy()[finite.cpu().numpy()], want[finite.cpu().numpy()])


# ------------------------------------------------------------------------------------------- raw C ABI vs oracle
def _rand_x(rng, n, dtype, scale=1.0):
    v = (rng.standard_normal(n) * scale).astype(np.float32)
    t = torch.from_numpy(v)
    if dtype == "bfloat16":
        t = t.bfloat16()
    elif dtype == "float16":
        t = t.half()
    return t


SIZES = [1, 3, 4, 5, 7, 8, 9, 31, 255, 1023, 1024, 1025, 4095, 4096, 4097, 8191, 8193, 16385, 100003]


def _affine_call(lib, prepared, xd, y, codes, n, tag, sd, zd, C, inner, elem_offset, qmin, qmax, code_mode):
    """mctq_fq_affine, or mctq_affine_prepare + mctq_fq_affine_prepared (TMA-staged parameters) on the same arguments."""
    if not prepared:
        return lib.mctq_fq_affine(_vp(xd), _vp(y), _vp(codes), n, tag, _vp(sd), _vp(zd), C, inner, elem_offset, qmin, qmax,
                                  code_mode, _stream())
    nb = lib.mctq_affine_prepared_bytes(C)
    blob = torch.full((nb,), 0xA5, dtype=torch.uint8, device=DEV)
    rc = lib.mctq_affine_prepare(_vp(sd), _vp(zd), C, _vp(blob), nb, _stream())
    assert rc == 0
    rc = lib.mctq_fq_affine_prepared(_vp(xd), _vp(y), _vp(codes), n, tag, _vp(blob), C, inner, elem_offset, qmin, qmax,
                                     code_mode, _stream())
    torch.cuda.synchronize()         # blob must outlive the launch
    return rc


@pytest.mark.parametrize("prepared", [False, True])
@pytest.mark.parametrize("dtype", ["float32", "bfloat16", "float16"])
@pytest.mark.parametrize("code_mode", [0, 1, 2])
def test_affine_ragged_sizes_and_codes(dtype, code_mode, prepared, lib):
    """Every tail path of the tile kernel, per-tensor and per-channel, values + int8 / int4 codes vs the oracle."""
    rng = np.random.default_rng(7)
    tag = G.DT_TAG[dtype]
    for n in SIZES:
        for (C, inner) in [(1, 1), (3, 1), (5, 7), (4, 8), (2, 4096), (7, 1000), (8, 1), (12, 1), (16, 3), (300, 2)]:
            bits = 4 if code_mode == 2 else 8
            signed = (n + C) % 2 == 0
            qmin, qmax = (-(2 ** (bits - 1)), 2 ** (bits - 1) - 1) if signed else (0, 2 ** bits - 1)
            scale = (np.abs(rng.standard_normal(C)) * 0.05 + 0.01).astype(np.float32)
            zp = rng.integers(qmin, qmax + 1, size=C).astype(np.int32) if not signed else np.zeros(C, np.int32)
            x = _rand_x(rng, n, dtype, 1.5)
            xd = x.to(DEV)
            y = torch.empty_like(xd)
            ncode = n if code_mode == 1 else (n + 1) // 2
            codes = torch.full((ncode + 8,), 0x5A, dtype=torch.uint8, device=DEV) if code_mode else None
            sd, zd = torch.from_numpy(scale).to(DEV), torch.from_numpy(zp).to(DEV)     # keep alive across the launch
            rc = _affine_call(lib, prepared, xd, y, codes, n, tag, sd, zd, C, inner, 0, qmin, qmax, code_mode)
            assert rc == 0, (n, C, inner)
            torch.cuda.synchronize()
            want_y, want_codes = oracle.fq_affine(G.from_torch(x), tag, scale, zp, C, inner, qmin, qmax, want_codes=True)
            got_y = G.from_torch(y)
            assert G.bits_equal(got_y, want_y), (n, C, inner, G.mismatch_report(got_y, want_y))
            if code_mode:
                got = codes.cpu().numpy()
                assert (got[ncode:] == 0x5A).all(), "wrote past the end of the code buffer"
                if code_mode == 1:
                    g = got[:n].view(np.int8).astype(np.int32) if signed else got[:n].astype(np.int32)
                else:
                    nib = np.stack([got[:ncode] & 0xF, got[:ncode] >> 4], 1).reshape(-1)[:n].astype(np.int32)
                    g = np.where(nib >= 8, nib - 16, nib) if signed else nib
                    if n % 2:
                        assert got[ncode - 1] >> 4 == 0
                assert np.array_equal(g, want_codes), (n, C, inner)


@pytest.mark.parametrize("prepared", [False, True])
@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_affine_elem_offset_slices(dtype, prepared, lib):
    """A tensor processed as arbitrary flat slices (elem_offset) == processed whole: the contract behind
    batch / channel-block sharding and host staging."""
    rng = np.random.default_rng(11)
    tag = G.DT_TAG[dtype]
    outer, C, inner = 3, 37, 53
    n = outer * C * inner
    scale = (np.abs(rng.standard_normal(C)) * 0.02 + 0.005).astype(np.float32)
    zp = rng.integers(0, 256, size=C).astype(np.int32)
    x = _rand_x(rng, n, dtype, 2.0)
    want = oracle.fq_affine(G.from_torch(x), tag, scale, zp, C, inner, 0, 255)
    sd, zd = torch.from_numpy(scale).to(DEV), torch.from_numpy(zp).to(DEV)
    cuts = sorted(set([0, n] + [int(c) for c in rng.integers(1, n, size=9)] + [8 * int(c) for c in rng.integers(1, n // 8, size=4)]))
    got = np.empty_like(want)
    for a, b in zip(cuts[:-1], cuts[1:]):
        xs = x[a:b].clone().to(DEV)          # fresh (aligned) allocation holding the slice
        ys = torch.empty_like(xs)
        assert _affine_call(lib, prepared, xs, ys, None, b - a, tag, sd, zd, C, inner, a, 0, 255, 0) == 0
        got[a:b] = G.from_torch(ys)
    assert G.bits_equal(got, want)
    # misaligned views (odd element offsets) take the scalar fallback kernel
    xd = x.to(DEV)
    for a in (1, 3, 5):
        ys = torch.empty(n - a + 1, dtype=xd.dtype, device=DEV)[1:]
        assert _affine_call(lib, prepared, xd[a:], ys, None, n - a, tag, sd, zd, C, inner, a, 0, 255, 0) == 0
        assert G.bits_equal(G.from_torch(ys), want[a:])


@pytest.mark.parametrize("dtype", ["float32", "bfloat16", "float16"])
def test_lut_ragged_sizes(dtype, lib):
    from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
    rng = np.random.default_rng(5)
    tag = G.DT_TAG[dtype]
    lut = np.array(sorted(rng.choice(np.arange(-128, 128), size=16, replace=False)), dtype=np.float32)
    table = lut_search_table(lut, 8, True).to(DEV)
    for n in SIZES:
        for (C, inner) in [(1, 1), (3, 1), (5, 7), (4, 8), (2, 4096), (6, 1000)]:
            thr = (np.abs(rng.standard_normal(C)) + 0.05).astype(np.float32)
            x = _rand_x(rng, n, dtype, 0.6)
            xd = x.to(DEV)
            y = torch.empty(n, dtype=torch.float32, device=DEV)
            td = torch.from_numpy(thr).to(DEV)
            rc = lib.mctq_fq_lut(_vp(xd), _vp(y), None, n, tag, _vp(table), 16, _vp(td), C, inner, 0,
                                 float(np.float32(1e-8)), 0, _stream())
            assert rc == 0
            torch.cuda.synchronize()
            want = oracle.fq_lut(G.from_torch(x), tag, lut, thr, C, inner, 8, True, 1e-8)
            assert G.bits_equal(y.cpu().numpy(), want), (n, C, inner, G.mismatch_report(y.cpu().numpy(), want))


@pytest.mark.parametrize("search", ["shuffle", "shared"])
def test_lut_all_table_sizes_and_searches(search, lib):
    """K = 1 .. 256 centroids (every padded search depth), values and indices: tables of <= 32 entries take the
    warp-shuffle search, larger ones the shared-memory search."""
    from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
    rng = np.random.default_rng(9)
    n = 50000
    x = _rand_x(rng, n, "float32", 0.5)
    xd = x.to(DEV)
    thr = np.array([0.9, 0.013, 2.0], dtype=np.float32)
    td = torch.from_numpy(thr).to(DEV)
    for K in ((1, 2, 3, 5, 16, 17) if search == "shuffle" else (64, 100, 256)):
        lut = rng.choice(np.arange(-128, 128), size=K, replace=False).astype(np.float32)   # unsorted on purpose
        table = lut_search_table(lut, 8, True).to(DEV)
        want, want_idx = oracle.fq_lut(x.numpy(), oracle.F32, lut, thr, 3, 5, 8, True, 1e-8, want_idx=True)
        y = torch.empty(n, dtype=torch.float32, device=DEV)
        idx = torch.empty(n, dtype=torch.uint8, device=DEV)
        rc = lib.mctq_fq_lut(_vp(xd), _vp(y), _vp(idx), n, 0, _vp(table), K, _vp(td), 3, 5, 0, float(np.float32(1e-8)), 1, _stream())
        assert rc == 0
        assert G.bits_equal(y.cpu().numpy(), want), K
        assert np.array_equal(idx.cpu().numpy().astype(np.int32), want_idx), K


def test_division_selftest(lib):
    """The 5-operation correctly-rounded division of the LUT kernels == __fdiv_rn on 2^31 (x, d) pairs."""
    bad = torch.zeros(1, dtype=torch.int64, device=DEV)
    assert lib.mctq_selftest_division(1 << 31, 0x1234, _vp(bad), _stream()) == 0
    torch.cuda.synchronize()
    assert int(bad.item()) == 0


def test_rint_variant_and_wide_ranges(lib):
    """8- to 24-bit ranges == oracle.  Ranges of 2^21 codes and more take the rint-based variant: 21 and 22 bits pin the
    switch (kFastRangeLimit) from both sides."""
    rng = np.random.default_rng(3)
    n = 70001
    x = _rand_x(rng, n, "float32", 3.0)
    xd = x.to(DEV)
    for bits in (8, 16, 21, 22, 24):
        qmin, qmax = -(2 ** (bits - 1)), 2 ** (bits - 1) - 1
        scale = np.array([8.0 / 2 ** (bits - 1)], dtype=np.float32)
        zp = np.zeros(1, np.int32)
        y = torch.empty_like(xd)
        rc = lib.mctq_fq_affine_scalar(_vp(xd), _vp(y), None, n, 0, float(scale[0]), 0, qmin, qmax, 0, _stream())
        assert rc == 0
        want = oracle.fq_affine(x.numpy(), 0, scale, zp, 1, 1, qmin, qmax)
        assert G.bits_equal(y.cpu().numpy(), want), bits


def test_dequant_roundtrip(lib):
    """codes -> mctq_dequant_affine == fake-quant values (f32), int8 and packed int4, signed and unsigned."""
    rng = np.random.default_rng(12)
    C, inner, outer = 11, 24, 5
    n = C * inner * outer
    x = _rand_x(rng, n, "float32", 1.0).to(DEV)
    for bits, signed, mode in ((8, True, 1), (8, False, 1), (4, True, 2), (4, False, 2)):
        qmin, qmax = (-(2 ** (bits - 1)), 2 ** (bits - 1) - 1) if signed else (0, 2 ** bits - 1)
        scale = torch.from_numpy((np.abs(rng.standard_normal(C)) * 0.1 + 0.01).astype(np.float32)).to(DEV)
        zp = torch.from_numpy((np.zeros(C) if signed else rng.integers(0, qmax + 1, size=C)).astype(np.int32)).to(DEV)
        y = torch.empty_like(x)
        codes = torch.empty(n if mode == 1 else (n + 1) // 2, dtype=torch.uint8, device=DEV)
        assert lib.mctq_fq_affine(_vp(x), _vp(y), _vp(codes), n, 0, _vp(scale), _vp(zp), C, inner, 0, qmin, qmax, mode, _stream()) == 0
        back = torch.empty_like(x)
        assert lib.mctq_dequant_affine(_vp(codes), mode, int(signed), _vp(back), n, _vp(scale), _vp(zp), C, inner, 0, _stream()) == 0
        assert torch.equal(back.view(torch.int32), y.view(torch.int32))
        # codes-only mode (y == NULL)
        codes2 = torch.empty_like(codes)
        assert lib.mctq_fq_affine(_vp(x), None, _vp(codes2), n, 0, _vp(scale), _vp(zp), C, inner, 0, qmin, qmax, mode, _stream()) == 0
        assert torch.equal(codes, codes2)


def _dequant_vec_widths(fn):
    """Vector widths (template argument V) of the dequant_affine_vec_kernel launches fn() makes, from the profiler."""
    import re
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    widths = set()
    for e in prof.key_averages():
        m = (re.search(r"dequant_affine_vec_kernel<\s*\d+\s*,\s*\d+\s*,\s*(\d+)\s*>", e.key)
             or re.search(r"dequant_affine_vec_kernelILi\d+ELi\d+ELi(\d+)E", e.key))
        if m:
            widths.add(int(m.group(1)))
    return widths


@pytest.mark.parametrize("bits,signed", [(8, True), (8, False), (4, True), (4, False)])
def test_dequant_vector_variants(bits, signed, lib):
    """The streaming dequant kernel in every (code mode, channel mode, vector width) combination, ragged sizes included:
    per-tensor, rows that are multiples of 8 / 4, odd rows.  Per-channel int4 rows of 8 take 8-code vectors with 256-bit
    stores, everything else 4-code vectors; the shapes reach both.  codes -> dequant == fake-quant values bit for bit."""
    rng = np.random.default_rng(77 + bits + int(signed))
    mode = 1 if bits == 8 else 2
    qmin, qmax = (-(2 ** (bits - 1)), 2 ** (bits - 1) - 1) if signed else (0, 2 ** bits - 1)
    launches = []
    for (C, inner, outer, tail) in ((1, 1, 70001, 0), (13, 64, 37, 0), (7, 12, 211, 0), (5, 9, 333, 0), (3, 4096, 3, 0), (6, 8, 1000, 5),
                                 (11, 3, 500, 0), (4, 1, 1000, 0), (3, 5, 2001, 2), (9, 4097, 2, 0)):
        n_full = C * inner * outer
        n = n_full - tail                                     # a flat prefix (ragged last vector)
        x = _rand_x(rng, n, "float32", 1.0).to(DEV)
        scale = torch.from_numpy((np.abs(rng.standard_normal(C)) * 0.1 + 0.01).astype(np.float32)).to(DEV)
        zp = torch.from_numpy((np.zeros(C) if signed else rng.integers(0, qmax + 1, size=C)).astype(np.int32)).to(DEV)
        y = torch.empty_like(x)
        codes = torch.empty(n if mode == 1 else (n + 1) // 2, dtype=torch.uint8, device=DEV)
        assert lib.mctq_fq_affine(_vp(x), _vp(y), _vp(codes), n, 0, _vp(scale), _vp(zp), C, inner, 0, qmin, qmax, mode, _stream()) == 0
        back = torch.full((n + 16,), 7.0, device=DEV)
        launches.append(lambda codes=codes, back=back, n=n, scale=scale, zp=zp, C=C, inner=inner:
                        lib.mctq_dequant_affine(_vp(codes), mode, int(signed), _vp(back), n, _vp(scale), _vp(zp), C, inner, 0, _stream()))
        assert launches[-1]() == 0
        assert torch.equal(back[:n].view(torch.int32), y.view(torch.int32)), (C, inner)
        assert (back[n:] == 7.0).all()
    assert _dequant_vec_widths(lambda: [f() for f in launches]) == ({4, 8} if bits == 4 else {4})


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_prepared_lut_wide_vectors_match_narrow(dtype, Q, lib):
    """2-byte inputs: the 8-element / 256-bit-store variant of the prepared LUT kernel == the 4-element variant (taken for
    an output 16 bytes past a 32-byte boundary) == the oracle, values and indices (int8, packed int4), ragged tails,
    per-channel and per-tensor."""
    from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
    rng = np.random.default_rng(5)
    lut = [float(v) for v in sorted(rng.choice(np.arange(-128, 128), size=16, replace=False))]
    table = lut_search_table(np.asarray(lut, np.float32), 8, True)
    tag = 1 if dtype == torch.bfloat16 else 2
    for shape, per_channel in (((37, 264), True), ((3, 8200), True), ((70003,), False)):
        x = torch.from_numpy((rng.standard_normal(shape) * 0.03).astype(np.float32)).to(dtype).to(DEV)
        if per_channel:
            thr = [float(v) + 1e-3 for v in x.float().abs().amax(1)]
            q = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, thr, True, 0, 2)
        else:
            thr = [0.11]
            q = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, thr, False)
        thr_t = torch.tensor(thr, dtype=torch.float32, device=DEV)
        n = x.numel()
        C, inner = (shape[0], shape[1]) if per_channel else (1, 1)
        wide = (q(x.clone()), torch.ops.mctq.lut_indices(x, table, 16, thr_t, per_channel, 0, 1e-8, 1),
                torch.ops.mctq.lut_indices(x, table, 16, thr_t, per_channel, 0, 1e-8, 2))
        nb = lib.mctq_lut_prepared_bytes(16, 8, 1, C)
        blob = torch.empty(nb, dtype=torch.uint8, device=DEV)
        assert lib.mctq_lut_prepare(_vp(table), 16, _vp(thr_t), C, float(np.float32(1e-8)), 0, 1.0, 1.0, 0, _vp(blob), nb, _stream()) == 0
        narrow = []
        for idx_mode in (1, 2):
            y = torch.empty(n + 8, dtype=torch.float32, device=DEV)[4:4 + n]
            assert y.data_ptr() % 32 == 16
            idx = torch.empty(n if idx_mode == 1 else (n + 1) // 2, dtype=torch.uint8, device=DEV)
            assert lib.mctq_fq_lut_prepared(_vp(x), _vp(y), _vp(idx), n, tag, _vp(blob), 16, 8, 1, C, inner, 0, idx_mode, _stream()) == 0
            narrow.append((y.reshape(shape), idx))
        torch.cuda.synchronize()
        assert torch.equal(narrow[0][0], narrow[1][0])
        outs = [wide, (narrow[0][0], narrow[0][1].reshape(shape), narrow[1][1])]
        for a, b in zip(outs[0], outs[1]):
            assert torch.equal(a, b)
        xb = x.cpu().contiguous().view(torch.int16).numpy().view(np.uint16)
        want, want_idx = oracle.fq_lut(xb, oracle.BF16 if dtype == torch.bfloat16 else oracle.F16, np.asarray(lut, np.float32),
                                       np.asarray(thr, np.float64).astype(np.float32), C, inner, 8, True, 1e-8, want_idx=True)
        assert np.array_equal(outs[1][0].cpu().numpy().view(np.uint32), np.asarray(want).reshape(shape).view(np.uint32))
        # sorted centroid list: the kernel emits the sorted position directly (identity permutation flag in the blob)
        assert np.array_equal(outs[1][1].cpu().numpy().reshape(-1).astype(np.int32), np.asarray(want_idx).reshape(-1))
        i4 = outs[1][2].cpu().numpy()
        un = np.stack([i4 & 0xF, i4 >> 4], 1).reshape(-1)[:x.numel()].astype(np.int32)
        assert np.array_equal(un, np.asarray(want_idx).reshape(-1))


def test_bad_arguments(lib):
    x = torch.zeros(16, device=DEV)
    y = torch.empty_like(x)
    s = torch.ones(1, device=DEV)
    z = torch.zeros(1, dtype=torch.int32, device=DEV)
    assert lib.mctq_fq_affine(_vp(x), _vp(y), None, 16, 7, _vp(s), _vp(z), 1, 1, 0, 0, 255, 0, None) == -2     # dtype
    assert lib.mctq_fq_affine(_vp(x), _vp(y), None, 16, 0, _vp(s), _vp(z), 1, 1, 0, 5, 2, 0, None) == -3       # qmin > qmax
    assert lib.mctq_fq_affine(_vp(x), _vp(y), None, -1, 0, _vp(s), _vp(z), 1, 1, 0, 0, 255, 0, None) == -1
    assert lib.mctq_fq_affine(_vp(x), _vp(y), _vp(y), 16, 0, _vp(s), _vp(z), 1, 1, 0, 0, 1023, 1, None) == -3  # codes do not fit
    assert lib.mctq_fq_affine(_vp(x), _vp(y), None, 0, 0, _vp(s), _vp(z), 1, 1, 0, 0, 255, 0, None) == 0       # empty is fine
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------- large tensors
def test_large_tensor_properties(Q):
    """BASELINE-scale tensors: oracle on sampled windows + size-independent properties (idempotence, code
    range, checksum agreement between two independent launches)."""
    g = torch.Generator(device=DEV).manual_seed(1234)
    n = (1 << 28) + 12345                                        # 1 GiB of f32 (+ ragged tail)
    x = torch.empty(n, device=DEV).uniform_(-50, 50, generator=g)
    q = Q.ActivationSymmetricInferableQuantizer(8, [4.0], True)
    y = q(x)
    y2 = q(y)
    assert torch.equal(y.view(torch.int32), y2.view(torch.int32))            # idempotent
    codes = torch.round(y / (4.0 / 128))
    assert codes.min().item() >= -128 and codes.max().item() <= 127
    scale = np.array([4.0 / 128], dtype=np.float32)
    for start in (0, 4096 * 777 + 3, n - 100000):
        xs = x[start:start + 100000].cpu().numpy()
        want = oracle.fq_affine(xs, 0, scale, np.zeros(1, np.int32), 1, 1, -128, 127)
        assert G.bits_equal(y[start:start + 100000].cpu().numpy(), want)
    del y2, codes
    # per-channel on a Llama-shaped matrix, bf16, channel axis 0 and 1
    W = torch.empty(4096, 11008, device=DEV).normal_(0, 0.02, generator=g).bfloat16()
    for axis in (0, 1):
        thr = W.float().abs().amax(dim=1 - axis).cpu().numpy().astype(np.float64)
        qw = Q.WeightsSymmetricInferableQuantizer(8, [float(t) for t in thr], True, axis)
        yw = qw(W)
        rows = slice(1000, 1016)
        C, inner = (4096, 11008) if axis == 0 else (11008, 1)
        sub = W[rows].contiguous()
        sc = (thr / 128).astype(np.float32)
        if axis == 0:
            want = oracle.fq_affine(G.from_torch(sub), oracle.BF16, sc[rows], np.zeros(16, np.int32), 16, inner, -128, 127)
        else:
            want = oracle.fq_affine(G.from_torch(sub), oracle.BF16, sc, np.zeros(C, np.int32), C, 1, -128, 127)
        assert G.bits_equal(G.from_torch(yw[rows]), want)


def test_index_space_beyond_32_bits(lib):
    """More than 2^32 bytes and more than 2^31 elements in one call (bf16): tail of the tensor is correct."""
    n = (1 << 31) + (1 << 20) + 7
    x = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    x[:1 << 20].normal_(0, 2)
    x[-(1 << 20):].normal_(0, 2)
    y = torch.empty_like(x)
    C, inner = 3, 1 << 29
    scale = torch.tensor([0.05, 0.01, 0.2], device=DEV)
    zp = torch.zeros(3, dtype=torch.int32, device=DEV)
    assert lib.mctq_fq_affine(_vp(x), _vp(y), None, n, 1, _vp(scale), _vp(zp), C, inner, 0, -128, 127, 0, _stream()) == 0
    torch.cuda.synchronize()
    tail = 1 << 20
    # channel of element i is (i / 2^29) % 3: the tail starts in row 4 (channel 1)
    i0 = n - tail
    ch = ((np.arange(i0, n, dtype=np.int64) // inner) % C)
    sc = scale.cpu().numpy()
    xt = G.from_torch(x[-tail:])
    want = np.empty(tail, dtype=np.uint16)
    for c in range(3):
        m = ch == c
        if m.any():
            want[m] = oracle.fq_affine(xt[m], oracle.BF16, sc[c:c + 1], np.zeros(1, np.int32), 1, 1, -128, 127)
    assert G.bits_equal(G.from_torch(y[-tail:]), want)
    xh = G.from_torch(x[:tail])
    want_h = oracle.fq_affine(xh, oracle.BF16, sc[0:1], np.zeros(1, np.int32), 1, 1, -128, 127)
    assert G.bits_equal(G.from_torch(y[:tail]), want_h)


# ------------------------------------------------------------------------------------------- layouts, host path, multi
def test_dense_permuted_layouts_keep_strides(Q):
    rng = np.random.default_rng(21)
    x = torch.from_numpy(rng.standard_normal((4, 6, 5, 7)).astype(np.float32)).to(DEV)
    thr = [float(v) for v in np.abs(rng.standard_normal(6)) + 0.1]
    q = Q.WeightsSymmetricInferableQuantizer(4, thr, True, 1)
    ref = q(x.clone())
    xcl = x.clone().contiguous(memory_format=torch.channels_last)
    ycl = q(xcl)
    assert ycl.stride() == xcl.stride()
    assert torch.equal(ycl, ref)
    xt = x.clone().permute(3, 1, 0, 2)                     # arbitrary dense permutation, channel axis now 1
    yt = q(xt)
    assert torch.equal(yt, ref.permute(3, 1, 0, 2))
    xs = x.clone()[:, :, ::2]                               # genuinely strided: falls back to a contiguous copy
    assert torch.equal(q(xs), ref[:, :, ::2])
    a = Q.ActivationUniformInferableQuantizer(8, [-1.0], [2.3])
    assert torch.equal(a(xcl), a(x))
    assert a(xcl).stride() == xcl.stride()


@pytest.mark.parametrize("name", ["w_sym_b8_pc_6x5x3x3_ax0", "w_uni_b4_pc_4x7x3x5_ax1", "a_uni_b8_straddle", "a_sym_b8_s_bfloat16_allbits",
                                  "wl_sym_lut16_pc_6x40_ax0", "al_s_l16_t4.0", "al_u_t0.0625_float16_allbits", "w_pot_b8_pt"])
def test_host_tensor_path_matches_reference_fixture(name, Q):
    """CPU tensors are streamed through the GPU (mctq_fq_*_host): same bits, result lands in host memory."""
    case = G.get_case(name)
    q = getattr(Q, case["cls"])(**case["args"])
    x = G.to_torch(case["x"], case["x_dtype"], "cpu")
    y = q(x)
    assert y.device.type == "cpu"
    assert G.bits_equal(G.from_torch(y), case["y"])
    y = q(x.pin_memory())
    assert G.bits_equal(G.from_torch(y), case["y"])


def test_host_path_multi_chunk(Q):
    """A host tensor larger than several staging chunks (per-channel, ragged rows) == device path."""
    g = torch.Generator().manual_seed(5)
    x = torch.empty(37, 1 << 20, dtype=torch.float32).normal_(0, 1, generator=g)       # 155 MB, rows not chunk aligned
    thr = [0.5 + 0.1 * i for i in range(37)]
    q = Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)
    y_host = q(x.clone())
    y_dev = q(x.clone().to(DEV))
    assert torch.equal(y_host, y_dev.cpu())
    ql = Q.WeightsLUTSymmetricInferableQuantizer(4, [float(v) for v in range(-128, 128, 16)], thr, True, 0, 2)
    assert torch.equal(ql(x.clone()), ql(x.clone().to(DEV)).cpu())


def test_host_pipeline_deferred_calls(Q, lib):
    """host_pipeline(): calls on pinned host tensors are only enqueued and overlap with each other; every result is
    complete at block exit and equals the device path.  More calls than parameter-ring entries, differing per-channel
    parameters, small (zero-copy) and multi-chunk tensors, LUT and affine mixed, nested scope, explicit wait()."""
    import mct_quantizers_b200 as mctq
    g = torch.Generator().manual_seed(11)
    jobs = []
    for i in range(11):
        rows = 5 + 3 * i
        cols = (1 << 12) if i % 3 else (3 << 19) + 17            # 80 KB .. 70 MB
        x = torch.empty(rows, cols, dtype=torch.float32).normal_(0, 1 + 0.1 * i, generator=g)
        thr = [0.3 + 0.05 * ((7 * i + r) % 13) for r in range(rows)]
        if i % 4 == 1:
            q = Q.WeightsLUTSymmetricInferableQuantizer(4, [float(v) for v in range(-120, 120, 15)], thr, True, 0, 2)
        elif i % 4 == 2:
            q = Q.WeightsUniformInferableQuantizer(8, [-t for t in thr], [1.7 * t for t in thr], True, 0)
        elif i % 4 == 3:
            q = Q.ActivationUniformInferableQuantizer(8, [-1.0 - 0.1 * i], [2.3])
        else:
            q = Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)
        if i == 5:
            x = x.to(torch.bfloat16)
        jobs.append((q, x))
    want = [q(x.clone().to(DEV)).cpu() for q, x in jobs]
    pinned = [x.clone().pin_memory() for _, x in jobs]
    before = lib.mctq_launch_count()
    with mctq.host_pipeline() as hp:
        outs = [q(xp) for (q, _), xp in zip(jobs[:6], pinned[:6])]
        hp.wait()
        assert all(torch.equal(o, w) for o, w in zip(outs, want[:6]))
        with mctq.host_pipeline():                               # nested scope: waits at its own exit, stays deferred
            outs.append(jobs[6][0](pinned[6]))
        assert torch.equal(outs[6], want[6])
        outs += [q(xp) for (q, _), xp in zip(jobs[7:], pinned[7:])]
    assert lib.mctq_launch_count() - before >= len(jobs)
    for k, (o, w) in enumerate(zip(outs, want)):
        assert o.device.type == "cpu" and o.is_pinned() and torch.equal(o, w), k
    for xp, (_, x) in zip(pinned, jobs):
        assert torch.equal(xp, x)                                # inputs untouched
    # outside the block the calls synchronise again
    assert torch.equal(jobs[0][0](pinned[0]), want[0])
    # pageable tensors inside a block work too (their copies are synchronous by nature)
    with mctq.host_pipeline():
        o = jobs[2][0](jobs[2][1].clone())
    assert torch.equal(o, want[2])


def test_whole_model_single_launch(Q, lib):
    """quantize_model_weights: every affine weight quantizer of a model in ONE kernel == per-layer calls."""
    import mct_quantizers_b200 as mctq
    torch.manual_seed(0)
    layers = [torch.nn.Conv2d(3, 16, 3), torch.nn.Conv2d(16, 32, 3, groups=16), torch.nn.Conv2d(32, 8, 1),
              torch.nn.Linear(40, 10)]
    wrapped = []
    for i, layer in enumerate(layers):
        w = layer.weight.detach()
        C = w.shape[0]
        if i % 2 == 0:
            thr = [float(v) for v in w.abs().flatten(1).amax(1)]
            qz = Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)
        else:
            lo = [float(v) for v in w.flatten(1).amin(1) - 0.01]
            hi = [float(v) for v in w.flatten(1).amax(1) + 0.01]
            qz = Q.WeightsUniformInferableQuantizer(8, lo, hi, True, 0)
        wrapped.append(mctq.PytorchQuantizationWrapper(layer, {'weight': qz}))
    model = torch.nn.Sequential(*wrapped).to(DEV)
    before = lib.mctq_launch_count()
    fused = mctq.quantize_model_weights(model)
    assert lib.mctq_launch_count() - before == 1
    for name, mod in model.named_children():
        per_layer = mod.get_quantized_weights()
        assert torch.equal(per_layer['weight'], fused[name]['weight'])
    for mod in model.children():
        assert mod.quantize_weights_batched().keys() == {'weight'}


def test_whole_model_lut_single_launch(Q, lib):
    """WeightPlan / quantize_model_weights with LUT weight quantizers: all of them in ONE mctq_fq_lut_prepared_multi
    launch (next to the one launch of the affine quantizers) == the per-layer calls, bit for bit.  Mixed table:
    f32 / bf16 / f16 weights, rows that are multiples of 8 (wide vectors), multiples of 4, odd (straddling vectors),
    per-tensor, ragged tile tails, different centroid lists and bit widths, a POT quantizer."""
    import mct_quantizers_b200 as mctq
    from mct_quantizers_b200.pytorch.model_quantization import WeightPlan
    rng = np.random.default_rng(33)
    lut16 = [float(v) for v in sorted(rng.choice(np.arange(-128, 128), size=16, replace=False))]
    lut8 = [float(v) for v in sorted(rng.choice(np.arange(-32, 32), size=8, replace=False))]
    specs = [((24, 520), torch.float32, lut16, 8, True), ((40, 64), torch.bfloat16, lut16, 8, True),
             ((6, 8200), torch.float16, lut8, 6, True), ((33, 27), torch.float32, lut8, 6, True),
             ((5, 4100), torch.bfloat16, lut16, 8, True), ((12, 3, 3, 3), torch.float32, lut16, 8, True),
             ((17, 1001), torch.float16, lut16, 8, False), ((3, 100000), torch.bfloat16, lut16, 8, True)]
    triples = []
    for k, (shape, dt, lut, bw, per_channel) in enumerate(specs):
        w = torch.from_numpy(rng.standard_normal(shape).astype(np.float32) * 0.05).to(dt).to(DEV)
        if per_channel:
            thr = [float(v) + 1e-3 for v in w.float().abs().flatten(1).amax(1)]
            q = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, thr, True, 0, len(shape), bw)
        elif k % 2:
            q = Q.WeightsLUTPOTInferableQuantizer(4, lut, [0.25], False, None, None, bw)
        else:
            q = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, [0.21], False, None, None, bw)
        triples.append((f"w{k}", w, q))
    # one affine tensor and one tensor the plan must leave to its own call (channel axis mismatch -> per-layer error path is
    # not exercised here; a user-defined callable quantizer is)
    wa = torch.randn(16, 33, device=DEV)
    triples.append(("affine", wa, Q.WeightsSymmetricInferableQuantizer(8, [float(v) for v in wa.abs().amax(1)], True, 0)))
    plan = WeightPlan(triples)
    assert plan.lut_plan is not None and plan.lut_plan.n_desc == len(specs) and plan.plan is not None and not plan.other
    before = lib.mctq_launch_count()
    outs = plan.run()
    # one affine launch + one LUT launch per kernel variant (this table is deliberately mixed: 7 variants for 8 tensors)
    assert lib.mctq_launch_count() - before == 1 + plan.lut_plan.n_launches and plan.lut_plan.n_launches <= 7
    same = [(f"s{k}", torch.randn(16 + k, 520, device=DEV) * 0.05) for k in range(5)]        # one variant -> ONE launch
    plan_same = WeightPlan([(n, w, Q.WeightsLUTSymmetricInferableQuantizer(4, lut16, [float(v) + 1e-3 for v in w.abs().amax(1)], True, 0, 2))
                            for n, w in same])
    before = lib.mctq_launch_count()
    plan_same.run()
    assert lib.mctq_launch_count() - before == 1 and plan_same.lut_plan.n_launches == 1
    for (name, w, q), y in zip(triples, outs):
        want = q(w.clone())
        assert y.dtype == want.dtype and y.shape == want.shape and torch.equal(y, want), name
    # run() again after changing a weight in place: outputs are refreshed, buffers reused
    ptrs = [y.data_ptr() for y in outs]
    triples[0][1].mul_(0.5)
    outs2 = plan.run()
    assert [y.data_ptr() for y in outs2] == ptrs
    assert torch.equal(outs2[0], triples[0][2](triples[0][1].clone()))
    # through the wrappers of a model
    lin = torch.nn.Linear(64, 40).to(DEV)
    thr = [float(v) + 1e-3 for v in lin.weight.detach().abs().amax(1)]
    wr = mctq.PytorchQuantizationWrapper(lin, {'weight': Q.WeightsLUTSymmetricInferableQuantizer(4, lut16, thr, True, 0, 2)})
    model = torch.nn.Sequential(wr).to(DEV)
    fused = mctq.quantize_model_weights(model)
    assert torch.equal(fused['0']['weight'], wr.get_quantized_weights()['weight'])


def test_weight_plan_under_cuda_graph(Q, lib):
    """WeightPlan.run() (one affine launch + one LUT launch per kernel variant; the LUT plans travel as kernel parameters) can be
    captured in a CUDA graph; a replay re-quantizes the CURRENT contents of the weights into the same output buffers."""
    from mct_quantizers_b200.pytorch.model_quantization import WeightPlan
    rng = np.random.default_rng(8)
    lut = [float(v) for v in sorted(rng.choice(np.arange(-128, 128), size=16, replace=False))]
    w1 = torch.randn(48, 256, device=DEV) * 0.05
    w2 = (torch.randn(16, 3, 3, 3, device=DEV) * 0.05).bfloat16()
    w3 = torch.randn(32, 72, device=DEV)
    q1 = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, [float(v) + 1e-3 for v in w1.abs().amax(1)], True, 0, 2)
    q2 = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, [0.2] * 16, True, 0, 4)
    q3 = Q.WeightsSymmetricInferableQuantizer(8, [float(v) for v in w3.abs().amax(1)], True, 0)
    plan = WeightPlan([("a", w1, q1), ("b", w2, q2), ("c", w3, q3)])
    plan.run()                                               # warm-up outside the capture (shared-memory attributes, caches)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            outs = plan.run()
    torch.cuda.current_stream().wait_stream(side)
    for w in (w1, w2, w3):
        w.mul_(0.7)                                          # new weight values, same storage
    graph.replay()
    torch.cuda.synchronize()
    for (w, q), y in zip(((w1, q1), (w2, q2), (w3, q3)), outs):
        assert torch.equal(y, q(w.clone()))


def test_first_lut_call_inside_a_graph_capture(Q):
    """A LUT quantizer whose FIRST call happens while a CUDA graph is being captured: the one-off table preparation
    (which synchronises) is postponed, the generic kernel is captured instead; replays and later eager calls agree."""
    rng = np.random.default_rng(9)
    lut = [float(v) for v in rng.choice(np.arange(-128, 128), size=16, replace=False)]
    w = torch.randn(24, 136, device=DEV) * 0.05
    x = torch.randn(4, 3000, device=DEV).half()
    qw = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, [float(v) + 1e-3 for v in w.abs().amax(1)], True, 0, 2)
    qa = Q.ActivationLutPOTInferableQuantizer(4, lut, [2.0], True)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            yw, ya = qw(w), qa(x)
    torch.cuda.current_stream().wait_stream(side)
    w.mul_(0.9)
    x.mul_(1.1)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(yw, qw(w.clone())) and torch.equal(ya, qa(x.clone()))      # eager calls: prepared kernels


def test_lut_multi_plan_rejects_what_it_cannot_run(Q, lib):
    """Tensors outside the prepared path (a centroid list too dense for the coarse cell table of a 14-bit grid, misaligned
    views) stay on their own call."""
    from mct_quantizers_b200.pytorch.model_quantization import WeightPlan
    lut = [-2000.0, -2.0, -1.0, 0.0, 1.0, 2.0, 1000.0, 2000.0]              # four thresholds inside one cell of the coarse table
    w = torch.randn(8, 256, device=DEV)
    q_wide = Q.WeightsLUTSymmetricInferableQuantizer(3, lut, [1.0] * 8, True, 0, 2, 14)
    base = torch.randn(8 * 256 + 1, device=DEV)
    w_mis = base[1:].view(8, 256)                                       # 4-byte aligned only
    q_ok = Q.WeightsLUTSymmetricInferableQuantizer(4, [float(v) for v in range(-128, 128, 16)], [1.0] * 8, True, 0, 2)
    plan = WeightPlan([("wide", w, q_wide), ("misaligned", w_mis, q_ok), ("ok", w, q_ok)])
    assert plan.lut_plan is not None and plan.lut_plan.n_desc == 1 and len(plan.other) == 2
    outs = plan.run()
    assert torch.equal(outs[0], q_wide(w.clone())) and torch.equal(outs[1], q_ok(w_mis.clone())) and torch.equal(outs[2], q_ok(w.clone()))


@pytest.mark.parametrize("dtype", ["float32", "bfloat16", "float16"])
def test_multi_tensor_kernel_vs_oracle(dtype, lib):
    """mctq_fq_affine_multi over a mixed descriptor table: rows that are / are not multiples of 4, ragged tails,
    per-tensor entries, int8 codes, a misaligned view -- every tensor bit-equal to the oracle."""
    import ctypes
    from mct_quantizers_b200 import _native
    rng = np.random.default_rng(21)
    tag = G.DT_TAG[dtype]
    specs = [(1, 1, 5), (1, 1, 4099), (16, 27, 16 * 27), (32, 9, 32 * 9), (8, 64, 8 * 64 * 3), (5, 4, 5 * 4 * 103),
             (64, 576, 64 * 576), (3, 2048, 3 * 2048 + 0), (7, 12, 7 * 12 * 11), (1, 1, 2048), (6, 1, 6 * 500)]
    keep, descs, wants = [], (_native.MctqTensorDesc * len(specs))(), []
    for k, (C, inner, n) in enumerate(specs):
        signed = k % 2 == 0
        qmin, qmax = (-128, 127) if signed else (0, 255)
        scale = (np.abs(rng.standard_normal(C)) * 0.03 + 0.004).astype(np.float32)
        zp = np.zeros(C, np.int32) if signed else rng.integers(0, 256, size=C).astype(np.int32)
        x = _rand_x(rng, n, dtype, 1.0)
        off = 1 if k == 5 else 0                                   # one misaligned view
        xd_full = torch.empty(n + off, dtype=x.dtype, device=DEV)
        xd = xd_full[off:]
        xd.copy_(x)
        y = torch.empty(n + off, dtype=x.dtype, device=DEV)[off:]
        codes = torch.full((n + 8,), 0x5A, dtype=torch.uint8, device=DEV) if k % 3 == 0 else None
        sd, zd = torch.from_numpy(scale).to(DEV), torch.from_numpy(zp).to(DEV)
        keep += [xd_full, xd, y, codes, sd, zd]
        d = descs[k]
        d.x, d.y, d.codes, d.scale, d.zp = xd.data_ptr(), y.data_ptr(), codes.data_ptr() if codes is not None else None, sd.data_ptr(), zd.data_ptr()
        d.n, d.C, d.inner, d.qmin, d.qmax, d.dtype, d.code_mode = n, C, inner, qmin, qmax, tag, 1 if codes is not None else 0
        want_y, want_codes = oracle.fq_affine(G.from_torch(x), tag, scale, zp, C, inner, qmin, qmax, want_codes=True)
        wants.append((y, codes, want_y, want_codes, signed, n))
    starts = (ctypes.c_int32 * (len(specs) + 1))()
    total = lib.mctq_multi_plan(ctypes.cast(descs, ctypes.c_void_p), len(specs), ctypes.cast(starts, ctypes.c_void_p))
    assert total > 0
    descs_dev = torch.frombuffer(bytearray(bytes(descs)), dtype=torch.uint8).to(DEV)
    starts_dev = torch.frombuffer(bytearray(bytes(starts)), dtype=torch.uint8).to(DEV)
    assert lib.mctq_fq_affine_multi(_vp(descs_dev), _vp(starts_dev), len(specs), total, _stream()) == 0
    torch.cuda.synchronize()
    for k, (y, codes, want_y, want_codes, signed, n) in enumerate(wants):
        got = G.from_torch(y)
        assert G.bits_equal(got, want_y), (k, specs[k], G.mismatch_report(got, want_y))
        if codes is not None:
            c = codes.cpu().numpy()
            assert (c[n:] == 0x5A).all()
            g = c[:n].view(np.int8).astype(np.int32) if signed else c[:n].astype(np.int32)
            assert np.array_equal(g, want_codes), (k, specs[k])


def test_model_weight_plan_hoists_weight_quantization(Q, lib):
    """plan_model_weights: one launch for all wrappers, forwards inside the plan launch nothing of ours for weights and
    give the per-layer path's result bit for bit; positional (constant) weights are covered too."""
    import mct_quantizers_b200 as mctq
    torch.manual_seed(3)

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            convs = [torch.nn.Conv2d(3, 8, 3, padding=1), torch.nn.Conv2d(8, 8, 3, padding=1, groups=8), torch.nn.Conv2d(8, 4, 1)]
            self.layers = torch.nn.ModuleList()
            for c in convs:
                thr = [float(v) for v in c.weight.detach().abs().flatten(1).amax(1)]
                self.layers.append(mctq.PytorchQuantizationWrapper(c, {'weight': Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)}))
            const = torch.randn(4, 1, 1)
            self.sub = mctq.PytorchQuantizationWrapper(torch.sub, {1: Q.WeightsUniformInferableQuantizer(8, [-2.0], [2.0], False)}, {1: const})

        def forward(self, x):
            for layer in self.layers:
                x = layer(x)
            return self.sub(x)

    model = Net().to(DEV).eval()
    x = torch.randn(2, 3, 16, 16, device=DEV)
    with torch.no_grad():
        want = model(x)
        c0 = lib.mctq_launch_count()
        model(x)
        per_layer_launches = lib.mctq_launch_count() - c0
        assert per_layer_launches == 4
        plan = mctq.plan_model_weights(model)
        c0 = lib.mctq_launch_count()
        with plan:
            assert lib.mctq_launch_count() - c0 == 1            # refresh(): one multi-tensor launch
            got = model(x)
            got2 = model(x)
            assert lib.mctq_launch_count() - c0 == 1            # the forwards launched no weight kernels
        assert torch.equal(got.view(torch.int32), want.view(torch.int32)) and torch.equal(got2.view(torch.int32), want.view(torch.int32))
        c0 = lib.mctq_launch_count()
        again = model(x)                                        # plan left: per-layer path is back
        assert lib.mctq_launch_count() - c0 == per_layer_launches
        assert torch.equal(again.view(torch.int32), want.view(torch.int32))


@pytest.mark.parametrize("bw", [12, 14, 16])
@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_wide_lut_grids_run_on_the_prepared_path(Q, bw, dtype):
    """Grids of more than 10 bits: sparse centroid lists are served by the prepared kernels (cell table coarser than the
    integer grid), values and packed 4-bit indices bit-equal to the oracle on a matrix large enough for the xy-record /
    wide-vector variants; a list with neighbouring integers is refused by mctq_lut_prepare and runs on the generic kernel."""
    from mct_quantizers_b200 import ops
    rng = np.random.default_rng(bw)
    lo, hi = -2 ** (bw - 1), 2 ** (bw - 1) - 1
    lut = sorted(set(int(v) for v in rng.integers(lo, hi, size=16)) | {0})[:16]
    while len(lut) < 16:
        lut.append(lut[-1] + 7)
    lut = [float(v) for v in lut if lo <= v <= hi]
    C, L = 96, 4096
    thr = [float(np.float32(v)) for v in rng.uniform(0.1, 4.0, C)]
    w = torch.from_numpy(rng.standard_normal((C, L)).astype(np.float32)).to(DEV).to(G.TORCH_DT[dtype])
    # plant points around every centroid midpoint of channel 0 and the last channel
    for c in (0, C - 1):
        mids = (np.asarray(lut[:-1]) + np.asarray(lut[1:])) / 2 / 2.0 ** (bw - 1) * (np.float32(thr[c]) + np.float32(1e-8))
        pts = np.concatenate([np.nextafter(mids.astype(np.float32), np.float32(s)) for s in (-np.inf, np.inf)] + [mids.astype(np.float32)])
        w[c, :pts.size] = torch.from_numpy(pts).to(w.dtype).to(DEV)
    n0 = len(ops._LUT_PREPARED)
    q = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, thr, True, 0, 2, bw)
    y = q(w)
    new = [v for v in list(ops._LUT_PREPARED.values())[n0:]]
    assert new and new[-1][1] is not None, "sparse list on a wide grid must be prepared"
    want, want_idx = oracle.fq_lut(G.from_torch(w), G.DT_TAG[dtype], np.asarray(lut, np.float32), np.asarray(thr, np.float64).astype(np.float32),
                                   C, L, bw, True, 1e-8, want_idx=True)
    assert G.bits_equal(y.cpu().numpy(), np.asarray(want).reshape(y.shape))
    from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
    table = lut_search_table(np.asarray(lut, np.float32), bw, True)
    idx4 = torch.ops.mctq.lut_indices(w, table, len(lut), torch.tensor(thr, device=DEV), True, 0, 1e-8, 2).cpu().numpy()
    un = np.stack([idx4 & 0xF, idx4 >> 4], 1).reshape(-1)[:w.numel()].astype(np.int32)
    assert np.array_equal(un, np.asarray(want_idx).reshape(-1))
    # dense list: refused by the prepared path, still exact
    dense = [float(v) for v in (lo, -3, -2, -1, 0, 1, 900, hi)]           # five neighbouring integers
    qd = Q.WeightsLUTSymmetricInferableQuantizer(3, dense, thr, True, 0, 2, bw)
    n1 = len(ops._LUT_PREPARED)
    yd = qd(w)
    newd = list(ops._LUT_PREPARED.values())[n1:]
    # 12 bits: one cell per grid step is still possible (valid for every integer list); beyond that the cells are wider
    assert newd and (newd[-1][1] is None) == (bw > 12), "dense list on a 14- / 16-bit grid must fall back to the generic kernel"
    wantd = oracle.fq_lut(G.from_torch(w), G.DT_TAG[dtype], np.asarray(dense, np.float32), np.asarray(thr, np.float64).astype(np.float32),
                          C, L, bw, True, 1e-8)
    assert G.bits_equal(yd.cpu().numpy(), np.asarray(wantd).reshape(yd.shape))
