"""Packed weights against an independent decoder of the code wire format (include/mctq.h, MCTQ_PACK_*).

The decoder below restates the layout in numpy: it shares no code with csrc/mctq_common.cuh, so a decode error that
mctq_unpack.cu and mctq_packed_linear.cu would share cannot hide.  It is checked on the CPU against the oracle's
fake-quant output and the golden LUT fixtures, then used as the reference for
  - every kernel variant of the unpack launch (kind x output dtype x channel mode x vector width x argument capacity),
    with outputs written into guarded views of one poisoned buffer;
  - the packed linear at the edges of its geometry (rows per CTA, m tiles, split-K segments, the element-wise path),
    with guarded inputs / outputs and non-finite inputs;
  - tensors of more than 2^31 elements;
  - chains of dependent launches under private_stream()."""
import ctypes
from collections import namedtuple

import numpy as np
import pytest
import torch

import golden_util as G
import oracle
from mct_quantizers_b200 import _native, ops
from test_packed_weights import LUT_CASES, dequant_lut_reference

I8, I4, LU8, LI4 = _native.PACK_AFFINE_I8, _native.PACK_AFFINE_I4, _native.PACK_LUT_U8, _native.PACK_LUT_I4
LUT_KINDS = (LU8, LI4)
INT4_KINDS = (I4, LI4)
DT = {torch.float32: _native.F32, torch.bfloat16: _native.BF16, torch.float16: _native.F16}
KIND_DTYPES = [(k, dt) for k in (I8, I4) for dt in (torch.float32, torch.bfloat16, torch.float16)] + [(k, torch.float32) for k in LUT_KINDS]
U_OUT = {torch.float32: 2.0 ** -24, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
HALF_SUBNORMAL = {torch.float32: 2.0 ** -150, torch.bfloat16: 2.0 ** -134, torch.float16: 2.0 ** -25}


# --------------------------------------------------------------------------------------------- reference decoder
def code_range(kind, is_signed):
    bits = 4 if kind in INT4_KINDS else 8
    return (-(1 << (bits - 1)), (1 << (bits - 1)) - 1) if is_signed else (0, (1 << bits) - 1)


def pack_codes(q, kind):
    """Integer codes (any sign) -> wire bytes: one byte per element, or two per byte with element 2j in the low nibble
    (the last high nibble of an odd count is padding, left 0 here)."""
    q = np.asarray(q, dtype=np.int64).reshape(-1)
    if kind not in INT4_KINDS:
        return (q & 0xFF).astype(np.uint8)
    u = q & 0xF
    if u.size % 2:
        u = np.append(u, 0)
    return (u[0::2] | (u[1::2] << 4)).astype(np.uint8)


def unpack_codes(buf, kind, is_signed, e0, count, byte0=0):
    """Codes of elements [e0, e0 + count) as int64 from wire bytes `buf`, whose first byte is byte `byte0` of the tensor.
    Rows are not byte-aligned: with an odd row length an int4 row starts in a high nibble."""
    buf = np.asarray(buf, dtype=np.uint8)
    e = np.arange(e0, e0 + count, dtype=np.int64)
    if kind in INT4_KINDS:
        b = buf[(e >> 1) - byte0].astype(np.int64)
        q = np.where(e & 1, b >> 4, b & 0xF)
        return np.where(q >= 8, q - 16, q) if is_signed else q
    q = buf[e - byte0].astype(np.int64)
    return np.where(q >= 128, q - 256, q) if is_signed else q


def lut_quotients_np(lut, bw, signed):
    """q_k = lut_k / 2^(bw - signed) in f32."""
    return np.asarray(lut, dtype=np.float32).reshape(-1) / np.float32(2.0 ** (bw - int(bool(signed))))


def decode(buf, kind, is_signed, dtype, C, inner, scale, zp=None, quot=None, e0=0, count=None, byte0=0):
    """Rebuilt values of elements [e0, e0 + count): f32 array for f32, uint16 bit patterns for bf16 / f16.
    Element i has channel (i / inner) % C.  Affine: (float)(q - zp[c]) * s[c], one f32 rounding, then one rounding to the
    output dtype.  LUT: quot[q] * thr[c] in f32; an index >= K decodes to 0."""
    if count is None:
        count = int(buf.size * (2 if kind in INT4_KINDS else 1)) - e0
    q = unpack_codes(buf, kind, is_signed, e0, count, byte0)
    c = (np.arange(e0, e0 + count, dtype=np.int64) // inner) % C
    scale = np.asarray(scale, dtype=np.float32).reshape(-1)
    if kind in LUT_KINDS:
        table = np.zeros(256, dtype=np.float32)
        quot = np.asarray(quot, dtype=np.float32).reshape(-1)
        table[:quot.size] = quot
        return table[q] * scale[c]
    zp = np.asarray(zp, dtype=np.int32).reshape(-1)
    y = oracle.dequant_affine(q.astype(np.int32), scale[c], zp[c], count, 1)       # per-element parameters
    return y if dtype == torch.float32 else oracle.f32_to_half_bits(y, DT[dtype])


def decoded_f64(buf, kind, is_signed, dtype, C, inner, scale, zp=None, quot=None, e0=0, count=None, byte0=0):
    y = decode(buf, kind, is_signed, dtype, C, inner, scale, zp, quot, e0, count, byte0)
    if y.dtype == np.uint16:
        y = oracle.half_bits_to_f32(y, DT[dtype])
    return y.astype(np.float64)


# --------------------------------------------------------------------------------------------- A: decoder self-test (CPU)
AFFINE_SELF = [((64, 40), 0), ((33, 5), 1), ((7, 3, 3), 1), ((5, 3, 3, 3), 0), ((999,), 0), ((1,), 0), ((17, 9), -1)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("bits", [4, 8])
@pytest.mark.parametrize("is_signed", [True, False])
@pytest.mark.parametrize("per_channel", [True, False])
def test_decoder_matches_the_oracle_fake_quant(dtype, bits, is_signed, per_channel):
    """Codes of the oracle's affine fake-quant, packed by pack_codes and decoded: the same bits as the oracle's y."""
    rng = np.random.default_rng(bits * 7 + int(is_signed) * 3 + int(per_channel))
    kind = I4 if bits == 4 else I8
    qmin, qmax = code_range(kind, is_signed)
    for shape, axis in AFFINE_SELF:
        C, inner = oracle.channel_layout(shape, axis if per_channel else None)
        x = (rng.standard_normal(shape) * 3).astype(np.float32)
        tag = DT[dtype]
        xs = x if tag == oracle.F32 else oracle.f32_to_half_bits(x, tag)
        scale = rng.uniform(0.01, 0.5, C).astype(np.float32)
        zp = rng.integers(qmin, qmax + 1, C).astype(np.int32)
        zp[0] = qmin
        zp[-1] = qmax
        y, codes = oracle.fq_affine(xs, tag, scale, zp, C, inner, qmin, qmax, want_codes=True)
        assert codes.min() >= qmin and codes.max() <= qmax
        buf = pack_codes(codes, kind)
        if codes.size % 2 and kind == I4:
            buf[-1] |= 0xA0                                     # padding nibble: never decoded
        got = decode(buf, kind, is_signed, dtype, C, inner, scale, zp, count=codes.size)
        assert G.bits_equal(got.reshape(y.shape), y), (shape, axis)
        # a window that starts mid-tensor (and in a high nibble) decodes like the whole
        e0 = 3 if codes.size > 8 else 0
        b0 = e0 // 2 if kind == I4 else e0
        win = decode(buf[b0:], kind, is_signed, dtype, C, inner, scale, zp, e0=e0, count=codes.size - e0, byte0=b0)
        assert G.bits_equal(win, got[e0:])


def test_decoder_wire_layout():
    """The layout itself, independently of any oracle: nibble order, sign extension, rows across byte boundaries."""
    buf = np.array([0x21, 0xF8, 0x7A], dtype=np.uint8)
    assert unpack_codes(buf, I4, False, 0, 6).tolist() == [1, 2, 8, 15, 10, 7]
    assert unpack_codes(buf, I4, True, 0, 6).tolist() == [1, 2, -8, -1, -6, 7]
    assert unpack_codes(buf, I8, True, 0, 3).tolist() == [0x21, -8, 0x7A]
    assert unpack_codes(buf, I8, False, 1, 2).tolist() == [0xF8, 0x7A]
    # rows of 3 int4 codes: row 1 starts in the high nibble of byte 1
    y = decode(buf, I4, True, torch.float32, 2, 3, [1.0, 2.0], [0, 1], count=6)
    assert y.tolist() == [1.0, 2.0, -8.0, -4.0, -14.0, 12.0]
    assert pack_codes([1, 2, -8, -1, -6], I4).tolist() == [0x21, 0xF8, 0x0A]
    # LUT: an index >= K decodes to 0
    q = lut_quotients_np([-128, 64], 8, True)
    assert q.tolist() == [-1.0, 0.5]
    assert decode(np.array([0x10, 0x32], np.uint8), LI4, False, torch.float32, 1, 1, [2.0], quot=q).tolist() == [-2.0, 1.0, 0.0, 0.0]


@pytest.mark.parametrize("name", LUT_CASES)
def test_decoder_matches_golden_lut_cases(name):
    """Oracle LUT indices packed into both LUT layouts and decoded: the reference's y, bitwise, and the same values as
    dequant_lut_reference."""
    case = G.get_case(name)
    out = G.oracle_run(case)
    p = out["p"]
    idx = out["idx"].reshape(-1)
    quot = lut_quotients_np(p["lut"], p["bw"], p["signed"])
    want = dequant_lut_reference(idx, p["lut"], p["thr"], p["C"], p["inner"], p["bw"], p["signed"])
    assert G.bits_equal(want.reshape(case["y"].shape), case["y"])
    for kind in ((LU8, LI4) if p["lut"].size <= 16 else (LU8,)):
        buf = pack_codes(idx, kind)
        got = decode(buf, kind, False, torch.float32, p["C"], p["inner"], p["thr"], quot=quot, count=idx.size)
        assert G.bits_equal(got, want), kind


# --------------------------------------------------------------------------------------------- B: unpack variants
Spec = namedtuple("Spec", "kind dtype C inner n misalign")
# (C, inner): per tensor; per channel with rows of a multiple of 4 but not 8; of a multiple of 8; any row length (inner
# 1, 2, 3, 5, 9: the last one is a conv weight [out][in][3][3] quantized on axis 1)
LAYOUTS = [(1, 1), (3, 4), (3, 12), (5, 8), (2, 16), (4, 1), (3, 2), (5, 3), (2, 5), (5, 9)]


def _round_up(v, m):
    return (v + m - 1) // m * m


def _sizes(row, many):
    """Below one vector, exactly one 4- / 8-wide tile, one tile + 1, several tiles with a ragged (odd) tail."""
    cand = [3, 4096, 4097, 8192, 8193, 3 * 8192 + 7] if many else [3, 4096, 8193]
    return sorted({_round_up(v, row) for v in cand})


def _kind_k(kind, i):
    return {LI4: (5, 16, 11), LU8: (100, 256, 17)}[kind][i % 3] if kind in LUT_KINDS else 0


def coverage_plans():
    """Plans (lists of Spec) that together launch every (variant, argument capacity) pair: per
    layout a plan with <= 4 tensors per variant, and one plan with all layouts (> 4 tensors per variant), tile counts
    from 1 to 19 in one variant (a launch holds tensors within 16x of its largest), and more than 64 tensors of one variant.  f32 outputs alternate between
    32-byte and 16-byte (not 32-byte) aligned starts."""
    few = []
    for C, inner in LAYOUTS:
        plan = []
        for kind, dtype in KIND_DTYPES:
            for i, n in enumerate(_sizes(C * inner, False)):
                plan.append(Spec(kind, dtype, C, inner, n, dtype == torch.float32 and i == 1))
        few.append(plan)
    many = []
    for kind, dtype in KIND_DTYPES:
        for C, inner in LAYOUTS:
            for i, n in enumerate(_sizes(C * inner, True)):
                many.append(Spec(kind, dtype, C, inner, n, dtype == torch.float32 and i % 3 == 2 and C > 1))
    many += [Spec(I4, torch.bfloat16, 1, 1, n, False) for n in (15 * 8192 - 3, 16 * 8192, 18 * 8192 + 5)]
    many += [Spec(LI4, torch.float32, 5, 3, 15 * (1 + k % 7), k % 2 == 1) for k in range(70)]
    return few + [many]


def _layout(specs):
    """Byte offsets of the outputs inside one buffer: gaps of 48..80 bytes between them, 32-byte aligned starts, or
    16 mod 32 where misalign is set."""
    offs, cur = [], 64
    for s in specs:
        off = _round_up(cur + 48, 32) + (16 if s.misalign else 0)
        offs.append(off)
        cur = off + s.n * torch.tensor([], dtype=s.dtype).element_size()
    return offs, _round_up(cur + 64, 32)


def _plan_variants(blob, nbytes):
    """(kind, dtype, mode, v, capacity) of every launch of a plan blob: a 64-byte header (n_chunks at offset 8), then
    one block per launch that starts with n_desc, kind, dtype, mode, v as int32."""
    raw = bytes(blob)[:nbytes]
    n_chunks = int(np.frombuffer(raw[8:12], np.int32)[0])
    if n_chunks == 0:
        return []
    stride = (nbytes - 64) // n_chunks
    out = []
    for c in range(n_chunks):
        n_desc, kind, dtype, mode, v = np.frombuffer(raw[64 + c * stride: 64 + c * stride + 20], np.int32).tolist()
        out.append((kind, dtype, mode, v, 4 if n_desc <= 4 else 64))
    return out


def _all_variant_pairs():
    """The (kind, out dtype, mode, V, capacity) launches that mctq_unpack.cu instantiates, no more and no fewer: per tensor
    (mode 0) 4-element vectors for f32 and 8 for 2-byte outputs; rows of a multiple of 4 (mode 1) 4, and 8 for 2-byte
    outputs and f32 int4 codes; other rows (mode 2) 4."""
    want = set()
    for kind, dtype in KIND_DTYPES:
        two_byte = dtype != torch.float32
        modes = [(0, 8 if two_byte else 4), (1, 4), (2, 4)] + ([(1, 8)] if two_byte or kind in INT4_KINDS else [])
        for mode, v in modes:
            for cap in (4, 64):
                want.add((kind, DT[dtype], mode, v, cap))
    assert len(want) == 60
    return want


def _fake_descs(specs):
    offs, _ = _layout(specs)
    ds = []
    for s, off in zip(specs, offs):
        d = _native.MctqPackedDesc()
        d.codes, d.y, d.n, d.C, d.inner = 0x7f0000000000, 0x7f1000000000 + off, s.n, s.C, s.inner
        d.kind, d.is_signed, d.y_dtype, d.K = s.kind, 1, DT[s.dtype], _kind_k(s.kind, 0) or 16
        d.scale = 0x7f2000000000
        d.zp, d.lut_quotients = (None, 0x7f4000000000) if s.kind in LUT_KINDS else (0x7f3000000000, None)
        ds.append(d)
    return ds


def test_unpack_variant_selection_covers_every_kernel():
    """Host half of the coverage check (no GPU): the plans of coverage_plans(), compiled from descriptors with fake device
    pointers, launch exactly the 60 (variant, capacity) pairs the library instantiates; a 16-byte but not 32-byte aligned
    f32 output never takes 8-element vectors."""
    lib = _native.load()

    def plan_variants(specs):
        ds = _fake_descs(specs)
        arr = (_native.MctqPackedDesc * len(ds))(*ds)
        p = ctypes.cast(arr, ctypes.c_void_p)
        nb = lib.mctq_unpack_plan_bytes(p, len(ds))
        assert nb > 0
        buf = (ctypes.c_uint8 * nb)()
        assert lib.mctq_unpack_plan(p, len(ds), ctypes.cast(buf, ctypes.c_void_p), nb) > 0
        return _plan_variants(buf, nb)

    seen = set()
    for specs in coverage_plans():
        seen |= set(plan_variants(specs))
    # a misaligned f32 output alone: 4-element vectors, also for per-channel int4 rows of 8
    mis = plan_variants([Spec(k, torch.float32, C, inner, 8200, True) for k in (I8, LI4) for C, inner in ((1, 1), (5, 8))])
    assert all(v == 4 for _, _, _, v, _ in mis)
    seen |= set(mis)
    want = _all_variant_pairs()
    assert seen == want, (sorted(want - seen), sorted(seen - want))


def _unpack_data(spec, rng, idx):
    """Codes (numpy bytes) and parameters for one tensor: every byte value in every position of the first 2048 bytes,
    random bytes after them, per-channel zero points at both ends of the code range, LUT indices >= K, a nonzero
    padding nibble after an odd int4 tensor."""
    kind = spec.kind
    nb = spec.n if kind not in INT4_KINDS else (spec.n + 1) // 2
    codes = rng.integers(0, 256, nb, dtype=np.uint8)
    j = np.arange(min(nb, 2048))
    codes[:j.size] = ((j // 8) + 37 * (j % 8) + idx) % 256
    if kind in INT4_KINDS and spec.n % 2:
        codes[-1] = (codes[-1] & 0x0F) | 0xB0
    is_signed = kind not in LUT_KINDS and idx % 2 == 0
    C = spec.C
    if kind in LUT_KINDS:
        K = _kind_k(kind, idx)
        scale = rng.uniform(0.25, 4.0, C).astype(np.float32)
        quot = lut_quotients_np(rng.integers(-128, 128, K), 8, True)
        return codes, False, scale, None, quot
    lo, hi = code_range(kind, is_signed)
    scale = (rng.uniform(0.5, 2.0, C) * 2.0 ** rng.integers(-12, 4, C)).astype(np.float32)
    zp = rng.integers(lo, hi + 1, C).astype(np.int32)
    zp[0], zp[-1] = (lo, hi) if idx % 4 < 2 else (hi, lo)
    return codes, is_signed, scale, zp, None


def _np_bits(t):
    t = t.detach().contiguous().cpu()
    return t.view(torch.int32).numpy().view(np.uint32) if t.element_size() == 4 else t.view(torch.int16).numpy().view(np.uint16)


def _run_guarded_unpack(specs, rng):
    """Build and run one UnpackPlan whose outputs are views of poisoned buffers (one per dtype); check every output
    against the decoder and every byte outside the outputs.  Returns the (variant, capacity) pairs of its launches."""
    dev = "cuda"
    items, outputs, refs, bufs = [], [], [], {}
    offs_all = {}
    for dtype in {s.dtype for s in specs}:
        sub = [s for s in specs if s.dtype == dtype]
        offs, total = _layout(sub)
        bufs[dtype] = torch.full((total,), 0xFF, dtype=torch.uint8, device=dev)
        offs_all[dtype] = iter(offs)
    covered = {dt: np.zeros(b.numel(), bool) for dt, b in bufs.items()}
    for k, s in enumerate(specs):
        codes, is_signed, scale, zp, quot = _unpack_data(s, rng, k)
        off = next(offs_all[s.dtype])
        esz = torch.tensor([], dtype=s.dtype).element_size()
        y = bufs[s.dtype][off: off + s.n * esz].view(s.dtype)
        covered[s.dtype][off: off + s.n * esz] = True
        if s.C > 1 and s.C * s.inner == 45:
            y = y.view(-1, 5, 3, 3)                                 # a conv weight quantized on axis 1
        items.append((torch.from_numpy(codes).to(dev), s.kind, is_signed, s.dtype, tuple(y.shape), None, s.C, s.inner,
                      torch.from_numpy(scale).to(dev), None if zp is None else torch.from_numpy(zp).to(dev),
                      None if quot is None else torch.from_numpy(quot).to(dev)))
        outputs.append(y)
        refs.append(decode(codes, s.kind, is_signed, s.dtype, s.C, s.inner, scale, zp, quot, count=s.n))
    plan = ops.UnpackPlan(items, outputs=outputs)
    launched = _plan_variants(plan._plan_host, plan._plan_nb)
    got = plan.run()
    assert all(a is b for a, b in zip(got, outputs))
    torch.cuda.synchronize()
    for k, (s, y, ref) in enumerate(zip(specs, outputs, refs)):
        g = _np_bits(y).reshape(-1)
        r = ref.view(np.uint32) if ref.dtype == np.float32 else ref
        if not np.array_equal(g, r):
            bad = np.flatnonzero(g != r)
            raise AssertionError(f"tensor {k} {s}: {bad.size} elements differ, first at {bad[:5].tolist()}")
    for dtype, buf in bufs.items():
        host = buf.cpu().numpy()
        guard = host[~covered[dtype]]
        assert np.all(guard == 0xFF), (dtype, int(np.count_nonzero(guard != 0xFF)))
    return launched


@pytest.mark.gpu
def test_unpack_every_variant_against_the_decoder():
    """All 30 kernel variants, each launched with <= 4 and with > 4 tensors, at every size class and channel layout, with
    outputs in guarded views; the launched (variant, capacity) pairs are read from the plan blobs and must be exactly the
    60 the library instantiates."""
    rng = np.random.default_rng(2024)
    seen = set()
    for specs in coverage_plans():
        seen |= set(_run_guarded_unpack(specs, rng))
    names = {I8: "affine_i8", I4: "affine_i4", LU8: "lut_u8", LI4: "lut_i4"}
    dnames = {0: "f32", 1: "bf16", 2: "f16"}
    print("\nlaunched unpack variants (kind, out, mode, V, capacity):")
    for kind, dt, mode, v, cap in sorted(seen):
        print(f"  {names[kind]:9s} {dnames[dt]:4s} mode {mode} V={v} cap {cap:2d}")
    want = _all_variant_pairs()
    assert seen == want, (sorted(want - seen), sorted(seen - want))


# --------------------------------------------------------------------------------------------- B: beyond 2^31 elements
def _big_unpack(kind, C, inner, n):
    g = torch.Generator(device="cuda").manual_seed(n % 1000)
    nb = (n + 1) // 2
    codes = torch.randint(0, 256, (nb,), dtype=torch.uint8, device="cuda", generator=g)
    rng = np.random.default_rng(C)
    scale = (rng.uniform(0.5, 2.0, C) * 2.0 ** -3).astype(np.float32)
    zp = np.arange(-3, -3 + C, dtype=np.int32)
    item = (codes, kind, True, torch.bfloat16, (n,), None, C, inner, torch.from_numpy(scale).cuda(), torch.from_numpy(zp).cuda(), None)
    plan = ops.UnpackPlan([item])
    y = plan.run()[0]
    torch.cuda.synchronize()
    windows = [(0, 4096), ((1 << 31) - 5000, 10001), (n - 6001, 6001)]
    for e0, cnt in windows:
        e0 -= e0 % 2
        b0 = e0 // 2
        buf = codes[b0: b0 + (cnt + 3) // 2].cpu().numpy()
        want = decode(buf, kind, True, torch.bfloat16, C, inner, scale, zp, e0=e0, count=min(cnt, n - e0), byte0=b0)
        got = _np_bits(y[e0: e0 + want.size])
        assert np.array_equal(got, want), (C, inner, e0, int(np.count_nonzero(got != want)))
    del y, plan, codes, item
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_unpack_beyond_2_31_elements():
    """int4 per-channel weights of more than 2^31 elements take the 64-bit channel walk: any row length (inner 3, odd n)
    and rows of a multiple of 8, bf16 out; windows at the start, around element 2^31 and at the end."""
    _big_unpack(I4, 7, 3, 21 * 102261127)                          # 2147483667 elements, mode 2
    _big_unpack(I4, 5, 8, 40 * 53687092)                           # 2147483680 elements, mode 1, 8-element vectors


# --------------------------------------------------------------------------------------------- C: packed linear
def _lin_data(kind, dtype, N, K, per_channel, is_signed, rng, exact=True, lut_k=None, scale_pow=None):
    """Packed weight [N][K] (numpy) with a nonzero padding nibble after odd int4 weights and LUT indices >= K.  exact:
    power-of-two scales / thresholds and LUT values on the 8-bit grid, so that every product and partial sum of the
    test inputs is exact in f32."""
    n = N * K
    nb = n if kind not in INT4_KINDS else (n + 1) // 2
    codes = rng.integers(0, 256, nb, dtype=np.uint8)
    if kind in INT4_KINDS and n % 2:
        codes[-1] = (codes[-1] & 0x0F) | 0xD0
    C = N if per_channel else 1
    if exact:
        scale = (2.0 ** rng.integers(-2, 2, C)).astype(np.float32)
    else:
        scale = (rng.uniform(0.5, 2.0, C) * 2.0 ** -6).astype(np.float32)
    if scale_pow is not None:
        scale[:] = np.float32(2.0 ** scale_pow)
    if kind in LUT_KINDS:
        K_lut = lut_k or (11 if kind == LI4 else 200)
        quot = lut_quotients_np(rng.integers(-128, 128, K_lut), 8, True)
        return codes, False, scale, None, quot
    lo, hi = code_range(kind, is_signed)
    zp = rng.integers(lo, hi + 1, C).astype(np.int32)
    zp[0] = lo
    zp[-1] = hi
    return codes, is_signed, scale, zp, None


def _dev(a, dtype=None):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _weight(data, kind, dtype, N, K):
    codes, is_signed, scale, zp, quot = data
    C = scale.size
    return decoded_f64(codes, kind, is_signed, dtype, C, K if C > 1 else 1, scale, zp, quot, count=N * K).reshape(N, K)


def _x(rng, shape, dtype, exact=True):
    if exact:
        x = rng.integers(-2, 3, shape).astype(np.float32) * np.float32(0.25)
    else:
        x = rng.standard_normal(shape).astype(np.float32)
    return torch.from_numpy(x).to("cuda", dtype)


def _linear(x, data, kind, N, bias=None):
    codes, is_signed, scale, zp, quot = data
    return torch.ops.mctq.packed_linear(x, _dev(codes), kind, is_signed, N, _dev(scale), _dev(zp), _dev(quot), bias)


def _ref(x, w, bias, elementwise=False):
    x64 = x.detach().double().cpu().numpy().reshape(-1, x.shape[-1])
    if elementwise:            # IEEE products of every pair (0 * inf = NaN), whatever the BLAS does with zeros
        y = (x64[:, None, :] * w[None, :, :]).sum(-1)
    else:
        y = x64 @ w.T
    mag = np.abs(x64) @ np.abs(w).T if not elementwise else None
    if bias is not None:
        b = bias.double().cpu().numpy()
        y = y + b
        mag = mag + np.abs(b) if mag is not None else None
    return y, mag


def _assert_exact(y, x, w, bias, what):
    want, _ = _ref(x, w, bias)
    want_t = torch.from_numpy(want).to(y.dtype).reshape(y.shape)
    got = _np_bits(y)
    ref = _np_bits(want_t)
    if not np.array_equal(got, ref):
        bad = np.argwhere(got.reshape(want.shape) != ref.reshape(want.shape))
        raise AssertionError(f"{what}: {len(bad)} outputs differ, first (row, col) {bad[:4].tolist()}")


def _within_bound(y, x, w, bias):
    want, mag = _ref(x, w, bias)
    K = x.shape[-1]
    got = y.double().cpu().numpy().reshape(want.shape)
    lim = (K + 3) * 2.0 ** -24 * mag * 1.01 + U_OUT[y.dtype] * np.abs(want) + (K + 2) * 2.0 ** -149 + HALF_SUBNORMAL[y.dtype]
    err = np.abs(got - want)
    return bool(np.all(err <= lim)), float(np.max(err - lim))


def _k_values(kind):
    """Around one vector of codes per lane (16 int4 / 8 int8 elements) and around 64 vectors per row (both split-K
    segments of a warp pair full)."""
    return [1, 15, 16, 17, 1008, 1024, 1040, 4095, 11008] if kind in INT4_KINDS else [1, 7, 8, 9, 504, 512, 520, 4095, 11008]


def _exact_shapes(kind):
    shapes = [(M, 9, 33) for M in (1, 2, 3, 4, 5, 7, 8, 9, 16, 17, 100)]              # rows of x: m tiles of 1, 2, 4, 8
    shapes += [(3, N, 64) for N in (1, 7, 8, 9, 15, 16, 17, 4097)]                       # rows of W around 8 / 16 per CTA
    shapes += [(2, 17, K) for K in _k_values(kind)]
    shapes += [(9, 4097, 1040 if kind in INT4_KINDS else 520), (5, 16, 11008)]
    return shapes


SIGNED_CASES = [(k, dt, s) for k, dt in KIND_DTYPES for s in ((True, False) if k not in LUT_KINDS else (False,))]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype,is_signed", SIGNED_CASES)
@pytest.mark.parametrize("per_channel", [True, False])
@pytest.mark.parametrize("with_bias", [True, False])
def test_linear_exact_against_the_decoder(kind, dtype, is_signed, per_channel, with_bias):
    """Exactly representable data: the output equals the f64 product with the decoder's weight, rounded once."""
    rng = np.random.default_rng(kind * 100 + DT[dtype] * 10 + 4 * is_signed + 2 * per_channel + with_bias)
    for M, N, K in _exact_shapes(kind):
        data = _lin_data(kind, dtype, N, K, per_channel, is_signed, rng)
        x = _x(rng, (M, K), dtype)
        bias = _x(rng, (N,), dtype) * 4 if with_bias else None
        y = _linear(x, data, kind, N, bias)
        assert y.shape == (M, N) and y.dtype == dtype
        _assert_exact(y, x, _weight(data, kind, dtype, N, K), bias, (M, N, K))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", KIND_DTYPES)
def test_linear_more_m_tiles_than_the_grid(kind, dtype):
    """8 * 65535 + 9 rows: more m tiles than the grid has in y, so CTAs loop over several tiles."""
    rng = np.random.default_rng(kind + 10 * DT[dtype])
    M, N, K = 8 * 65535 + 9, 9, 17
    data = _lin_data(kind, dtype, N, K, True, True, rng)
    x = _x(rng, (M, K), dtype)
    bias = _x(rng, (N,), dtype)
    _assert_exact(_linear(x, data, kind, N, bias), x, _weight(data, kind, dtype, N, K), bias, "M = 8 * 65535 + 9")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", KIND_DTYPES)
def test_linear_fast_and_elementwise_paths_agree(kind, dtype):
    """At an aligned in_features, a misaligned x (4-byte offset) or misaligned codes (1-byte offset) take the element-wise
    path: its bits equal the aligned call's."""
    rng = np.random.default_rng(7 + kind)
    epv = 16 if kind in INT4_KINDS else 8
    for M, N, K in ((1, 17, epv), (3, 33, 64 * epv), (8, 9, 4096), (2, 40, 11008)):
        data = _lin_data(kind, dtype, N, K, True, True, rng, exact=False)
        codes, is_signed, scale, zp, quot = data
        x = _x(rng, (M, K), dtype, exact=False)
        bias = _x(rng, (N,), dtype, exact=False)
        args = (kind, is_signed, N, _dev(scale), _dev(zp), _dev(quot), bias)
        aligned = torch.ops.mctq.packed_linear(x, _dev(codes), *args)
        esz = x.element_size()
        xbuf = torch.empty(M * K + 16, dtype=dtype, device="cuda")
        xo = xbuf[4 // esz: 4 // esz + M * K].view(M, K)
        xo.copy_(x)
        cbuf = torch.empty(codes.size + 16, dtype=torch.uint8, device="cuda")
        co = cbuf[1: 1 + codes.size]
        co.copy_(_dev(codes))
        assert xo.data_ptr() % 16 == 4 and co.data_ptr() % 16 == 1
        for xa, ca in ((xo, _dev(codes)), (x, co), (xo, co)):
            got = torch.ops.mctq.packed_linear(xa, ca, *args)
            assert np.array_equal(_np_bits(got), _np_bits(aligned)), (M, N, K, xa is xo, ca is co)
        ok, worst = _within_bound(aligned, x, _weight(data, kind, dtype, N, K), bias)
        assert ok, (M, N, K, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", KIND_DTYPES)
def test_linear_error_bound_on_random_data(kind, dtype):
    """Random data, few output rows and long rows (a split of K across CTAs would change these first), and subnormal x."""
    rng = np.random.default_rng(11 + kind + DT[dtype])
    for M, N, K in ((1, 10, 11008), (4, 10, 11008), (1, 1, 16384), (3, 1, 16384), (8, 4097, 1040), (2, 33, 4095)):
        for per_channel in (True, False):
            data = _lin_data(kind, dtype, N, K, per_channel, True, rng, exact=False)
            x = _x(rng, (M, K), dtype, exact=False)
            bias = _x(rng, (N,), dtype, exact=False)
            ok, worst = _within_bound(_linear(x, data, kind, N, bias), x, _weight(data, kind, dtype, N, K), bias)
            assert ok, (M, N, K, per_channel, worst)
    # subnormal inputs (and results)
    tiny = {torch.float32: 2.0 ** -135, torch.bfloat16: 2.0 ** -135, torch.float16: 2.0 ** -20}[dtype]
    for M, N, K in ((3, 17, 1040), (2, 9, 33)):
        data = _lin_data(kind, dtype, N, K, True, True, rng, exact=False)
        x = (_x(rng, (M, K), torch.float32, exact=False) * tiny).to(dtype)
        assert bool((x != 0).any()) and bool((x.float().abs() < (2.0 ** -126 if dtype != torch.float16 else 2.0 ** -14)).all())
        ok, worst = _within_bound(_linear(x, data, kind, N), x, _weight(data, kind, dtype, N, K), None)
        assert ok, ("subnormal", M, N, K, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", KIND_DTYPES)
def test_linear_guard_bands(kind, dtype):
    """The C ABI with y and bias inside NaN-poisoned buffers and x followed by NaN rows: every guard keeps its bits, no NaN
    reaches y, and y is exact.  Odd int4 weights carry a nonzero padding nibble; LUT indices go up to 15 / 255 with
    K = 5 / 100."""
    lib = _native.load()
    rng = np.random.default_rng(3 + kind)
    GAP = 37
    for M, N, K in ((3, 17, 33), (8, 9, 1040), (5, 33, 15), (1, 7, 4097), (2, 16, 64)):
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
        rc = lib.mctq_packed_linear(pl._desc_ptr, N, K, xbuf.data_ptr(), DT[dtype], M, bbuf[GAP:].data_ptr(),
                                    ybuf[GAP:].data_ptr(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        torch.cuda.synchronize()
        after = _np_bits(ybuf)
        assert np.array_equal(after[:GAP], before[0][:GAP]) and np.array_equal(after[GAP + M * N:], before[0][GAP + M * N:]), (M, N, K)
        assert np.array_equal(_np_bits(bbuf), before[1]) and np.array_equal(_np_bits(xbuf), before[2])
        y = ybuf[GAP: GAP + M * N].view(M, N)
        assert not bool(torch.isnan(y).any()), (M, N, K)
        _assert_exact(y, x, _weight(data, kind, dtype, N, K), bias, ("guarded", M, N, K))


def _same_pattern(y, want, what):
    got = y.double().cpu().numpy().reshape(want.shape)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (what, "NaN pattern")
    inf = np.isinf(want)
    assert np.array_equal(np.isinf(got), inf) and np.array_equal(got[inf], want[inf]), (what, "inf pattern")
    fin = np.isfinite(want)
    want_t = torch.from_numpy(np.where(fin, want, 0.0)).to(y.dtype).double().numpy()
    assert np.array_equal(got[fin], want_t[fin]), (what, "finite values")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dtype", KIND_DTYPES)
def test_linear_non_finite_inputs(kind, dtype):
    """NaN / +-inf in x reach exactly the outputs the f64 product gives them (NaN where 0 * inf or inf - inf, the signed
    infinity elsewhere); other rows stay exact.  f16 weights that round to +-inf do the same."""
    rng = np.random.default_rng(5 + kind)
    for M, N, K in ((4, 33, 1040), (4, 17, 33)):
        data = _lin_data(kind, dtype, N, K, True, True, rng)
        w = _weight(data, kind, dtype, N, K)
        x = _x(rng, (M, K), dtype)
        x[1, 5] = float("nan")
        x[2, 7] = float("inf")
        x[3, 11] = float("-inf")
        x[3, K - 2] = float("inf")
        bias = _x(rng, (N,), dtype)
        want, _ = _ref(x, w, bias, elementwise=True)
        _same_pattern(_linear(x, data, kind, N, bias), want, (M, N, K))
    if dtype == torch.float16 and kind not in LUT_KINDS:
        M, N, K = 3, 24, 64
        data = _lin_data(kind, dtype, N, K, True, False, rng)
        data[2][::3] = 2.0 ** 12 if kind == I8 else 2.0 ** 13         # (q - zp) * s beyond 65504 in some rows
        w = _weight(data, kind, dtype, N, K)
        assert np.isinf(w).any() and np.isfinite(w).any()
        x = _x(rng, (M, K), dtype)
        want, _ = _ref(x, w, None, elementwise=True)
        _same_pattern(_linear(x, data, kind, N), want, "f16 weights at +-inf")


@pytest.mark.gpu
def test_linear_beyond_2_31_weight_elements():
    """One int4 weight of 65539 x 32768 (> 2^31 elements) at one row of x: rows around element 2^31 and the last rows."""
    N, K = 65539, 32768
    g = torch.Generator(device="cuda").manual_seed(5)
    codes = torch.randint(0, 256, (N * K // 2,), dtype=torch.uint8, device="cuda", generator=g)
    rng = np.random.default_rng(9)
    scale = (rng.uniform(0.5, 2.0, N) * 2.0 ** -6).astype(np.float32)
    zp = rng.integers(-8, 8, N).astype(np.int32)
    x = _x(rng, (1, K), torch.float32, exact=False)
    y = torch.ops.mctq.packed_linear(x, codes, I4, True, N, _dev(scale), _dev(zp), None, None)
    rows = [0, 1, 65533, 65534, 65535, 65536, 65537, 65538]       # element 2^31 is the first of row 65536
    for r in rows:
        buf = codes[r * K // 2: (r + 1) * K // 2].cpu().numpy()
        w = decoded_f64(buf, I4, True, torch.float32, N, K, scale, zp, e0=r * K, count=K, byte0=r * K // 2).reshape(1, K)
        ok, worst = _within_bound(y[:, r:r + 1], x, w, None)
        assert ok, (r, worst)
    del codes, y
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_linear_f32_scale_factoring_envelope():
    """f32 affine weights apply the scale after the row sum: |x| up to 1e30 with |q - zp| up to 255 stays within the
    error bound (the sum before the scale stays below FLT_MAX)."""
    rng = np.random.default_rng(13)
    for kind in (I8, I4):
        for M, N, K in ((2, 64, 4096), (1, 9, 1040)):
            data = _lin_data(kind, torch.float32, N, K, True, False, rng, exact=False)
            data[3][:] = 0 if kind == I4 else np.where(np.arange(N) % 2, 0, 255)
            x = torch.from_numpy((rng.uniform(-1, 1, (M, K)) * 1e30).astype(np.float32)).cuda()
            x[0, :8] = 1e30
            y = _linear(x, data, kind, N)
            assert bool(torch.isfinite(y).all())
            ok, worst = _within_bound(y, x, _weight(data, kind, torch.float32, N, K), None)
            assert ok, (kind, M, N, K, worst)


# --------------------------------------------------------------------------------------------- D: dependent launches
@pytest.mark.gpu
def test_packed_kernels_under_private_stream_orders():
    """Chains of this library's launches through the C ABI under the opt-in overlap orders (key 3 = 2, 3) give the bits of
    the default order: fake-quant writes x -> packed linear reads it; a scalar fake-quant reads y -> a second packed
    linear; fake-quant emits int8 codes into the buffer a PackedLinear and an UnpackPlan read; fake-quant overwrites the x
    that was just read."""
    lib = _native.load()
    dev = "cuda"
    N, K, M, N2 = 4096, 4096, 8, 2048
    gen = torch.Generator(device=dev).manual_seed(21)
    w_src = torch.empty(N, K, device=dev).uniform_(-1, 1, generator=gen)
    x_src = [torch.empty(M, K, device=dev).uniform_(-4, 4, generator=gen) for _ in range(2)]
    big_src = torch.empty(48 << 20, device=dev).uniform_(-4, 4, generator=gen)
    wscale = torch.full((N,), 1.0 / 127, device=dev)
    wzp = torch.zeros(N, dtype=torch.int32, device=dev)
    codes = torch.zeros(N * K, dtype=torch.uint8, device=dev)
    pl = ops.PackedLinear(codes, I8, True, torch.float32, N, K, wscale, wzp, None)
    c2 = torch.randint(0, 256, (N2 * N,), dtype=torch.uint8, device=dev, generator=gen)
    pl2 = ops.PackedLinear(c2, I8, True, torch.float32, N2, N, torch.full((N2,), 2.0 ** -9, device=dev),
                           torch.zeros(N2, dtype=torch.int32, device=dev), None)
    w_out = torch.empty(N, K, device=dev)
    plan = ops.UnpackPlan([(codes, I8, True, torch.float32, (N, K), None, N, K, wscale, wzp, None)], outputs=[w_out])
    x, y, y2, z, big = (torch.empty(M, K, device=dev), torch.empty(M, N, device=dev), torch.empty(M, N, device=dev),
                        torch.empty(M, N2, device=dev), torch.empty(48 << 20, device=dev))
    one = torch.ones(1, device=dev)
    zero = torch.zeros(1, dtype=torch.int32, device=dev)
    vp = ctypes.c_void_p

    def st():
        return vp(torch.cuda.current_stream().cuda_stream)

    def fq(src, dst, codes_out=None, C=1, inner=1, s=one, zp=zero, qmin=0, qmax=255):
        n = src.numel()
        assert lib.mctq_fq_affine(vp(src.data_ptr()), vp(dst.data_ptr()) if dst is not None else None,
                                  vp(codes_out.data_ptr()) if codes_out is not None else None, n, 0, vp(s.data_ptr()),
                                  vp(zp.data_ptr()), C, inner, 0, qmin, qmax, 1 if codes_out is not None else 0, st()) == 0

    def linear(p, xin, out, m, n_out, k):
        assert lib.mctq_packed_linear(p._desc_ptr, n_out, k, vp(xin.data_ptr()), 0, m, None, vp(out.data_ptr()), st()) == 0

    xs, s_big = torch.full((1,), 0.05, device=dev), (torch.full((1,), 0.03, device=dev), torch.full((1,), 0.07, device=dev))

    def sequence():
        codes.zero_()
        for t in (x, y, y2, z, w_out, big):
            t.fill_(float("nan"))
        torch.cuda.synchronize()
        fq(big_src, big, s=s_big[0])              # a large predecessor
        fq(w_src, None, codes_out=codes, C=N, inner=K, s=wscale, zp=wzp, qmin=-128, qmax=127)   # codes of W
        fq(x_src[0], x, s=xs)                                               # writes x
        linear(pl, x, y, M, N, K)                                                 # reads x and the codes
        assert lib.mctq_unpack_multi(ctypes.cast(plan._plan_host, vp), st()) == 0  # reads the codes
        assert lib.mctq_fq_affine_scalar(vp(y.data_ptr()), vp(y2.data_ptr()), None, M * N, 0, 0.125, 128, 0, 255, 0, st()) == 0
        linear(pl2, y2, z, M, N2, N)                                              # reads the scalar fake-quant's output
        fq(x_src[1], y2, s=xs)                                              # overwrites the x just read
        fq(x_src[1], x, s=xs)
        fq(big_src, big, s=s_big[1])
        torch.cuda.synchronize()
        return [t.clone() for t in (codes, x, y, y2, z, w_out, big)]

    want = sequence()
    assert not any(bool(torch.isnan(t.float()).any()) for t in want)
    wq = decoded_f64(want[0].cpu().numpy(), I8, True, torch.float32, N, K, wscale.cpu().numpy(), wzp.cpu().numpy(), count=N * K)
    assert np.array_equal(want[5].cpu().numpy().reshape(-1), wq.astype(np.float32))
    for mode in (2, 3):
        prev = lib.mctq_set_tuning(3, mode)
        try:
            for _ in range(3):
                for a, b in zip(want, sequence()):
                    assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), mode
        finally:
            lib.mctq_set_tuning(3, prev)
