"""Host-side robustness of the CUDA path: inference tensors, stale launch plans, in-place parameter edits, reuse and
fallbacks of the whole-model plans, wide ranges in the fused holder.  Every result is compared with the per-layer call
and / or the oracle."""
import numpy as np
import pytest
import torch

import golden_util as G
import oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def Q():
    from mct_quantizers_b200.pytorch import quantizers
    return quantizers


def _oracle_sym(w, thr, bits=8):
    C = w.shape[0]
    sc = (np.asarray(thr, np.float64) / 2 ** (bits - 1)).astype(np.float32)
    return oracle.fq_affine(G.from_torch(w), {torch.float32: oracle.F32, torch.bfloat16: oracle.BF16, torch.float16: oracle.F16}[w.dtype],
                            sc, np.zeros(C, np.int32), C, w[0].numel(), -2 ** (bits - 1), 2 ** (bits - 1) - 1)


def test_quantizers_built_and_run_under_inference_mode(Q):
    """Inference tensors carry no version counter: cache keys must not touch `_version` (a per-channel weight call used
    to raise 'Inference tensors do not track version counter')."""
    rng = np.random.default_rng(0)
    with torch.inference_mode():
        w = torch.from_numpy(rng.standard_normal((24, 40)).astype(np.float32)).to(DEV)
        thr = [float(v) for v in w.abs().amax(1)]
        q = Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)
        assert q.scales.is_inference()
        y = q(w)
        lut = [-8.0, -3.0, 0.0, 1.0, 5.0, 7.0]
        ql = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, thr, True, 0, 2, 4)
        yl = ql(w)
        qa = Q.ActivationUniformInferableQuantizer(8, [-1.0], [2.0])
        ya = qa(w)
    assert G.bits_equal(y.cpu().numpy(), np.asarray(_oracle_sym(w, thr)).reshape(y.shape))
    want = oracle.fq_lut(w.cpu().numpy(), oracle.F32, np.asarray(lut, np.float32), np.asarray(thr, np.float64).astype(np.float32),
                         24, 40, 4, True, 1e-8)
    assert G.bits_equal(yl.cpu().numpy(), np.asarray(want).reshape(yl.shape))
    assert ya.shape == w.shape
    # parameters created under inference mode, used outside it, and (when there is a second GPU) on another device
    y2 = q(w.clone())
    assert torch.equal(y2, y)
    if torch.cuda.device_count() > 1:
        with torch.inference_mode():
            y3 = q(w.to("cuda:1"))
        assert torch.equal(y3.cpu(), y.cpu())


def test_weight_plan_follows_moved_and_converted_weights(Q):
    """WeightPlan / ModelWeightPlan capture pointers: after .half(), a re-assigned parameter or new storage the plan must
    rebuild instead of quantizing the stale storage."""
    import mct_quantizers_b200 as mctq
    from mct_quantizers_b200.pytorch.model_quantization import plan_model_weights
    torch.manual_seed(0)
    convs = [torch.nn.Conv2d(8, 16, 3), torch.nn.Conv2d(16, 8, 1)]
    wrappers = []
    for c in convs:
        thr = [float(v) for v in c.weight.detach().abs().flatten(1).amax(1)]
        wrappers.append(mctq.PytorchQuantizationWrapper(c, {'weight': Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)}))
    model = torch.nn.Sequential(*wrappers).to(DEV)
    plan = plan_model_weights(model)
    plan.enable()

    def installed():
        return [w.layer.weight.detach().clone() for w in wrappers]

    def per_layer():
        return [w.get_quantized_weights()['weight'] for w in wrappers]

    for got, want in zip(installed(), per_layer()):
        assert torch.equal(got, want)
    # 1. new values in new storage (what load_state_dict / an optimizer step into fresh tensors does)
    with torch.no_grad():
        for w in wrappers:
            for _, p, _ in w.get_weights_vars():
                p.data = (p.data * 0.5).clone()
    plan.refresh()
    for got, want in zip(installed(), per_layer()):
        assert torch.equal(got, want)
    # 2. dtype conversion of the whole model
    model.half()
    plan.refresh()
    for got, want, w in zip(installed(), per_layer(), wrappers):
        assert got.dtype == torch.float16 and torch.equal(got, want)
        p = w.get_weights_vars()[0][1]
        thr = [float(v) for v in w.get_weights_vars()[0][2].threshold_np]
        assert G.bits_equal(G.from_torch(got).reshape(-1), np.asarray(_oracle_sym(p.detach(), thr)).reshape(-1))
    plan.disable()


def test_weight_plan_fallbacks_and_reuse(Q):
    from mct_quantizers_b200.pytorch.model_quantization import WeightPlan
    rng = np.random.default_rng(1)
    w_dense = torch.from_numpy(rng.standard_normal((16, 32)).astype(np.float32)).to(DEV)
    w_view = torch.from_numpy(rng.standard_normal((16, 64)).astype(np.float32)).to(DEV)[:, ::2]      # not dense
    w_reuse = torch.from_numpy(rng.standard_normal((16, 32)).astype(np.float32)).to(DEV)
    thr = lambda w: [float(v) for v in w.abs().amax(1)]  # noqa: E731
    q1 = Q.WeightsSymmetricInferableQuantizer(8, thr(w_dense), True, 0)
    q2 = Q.WeightsSymmetricInferableQuantizer(8, thr(w_view), True, 0)
    q3 = Q.WeightsSymmetricInferableQuantizer(8, thr(w_reuse), True, 0)
    q3.enable_reuse_quantizer()
    plan = WeightPlan([("a", w_dense, q1), ("b", w_view, q2), ("c", w_reuse, q3)])
    assert plan.plan is not None and plan.plan.n_desc == 1 and len(plan.other) == 2      # view and reuse -> per-quantizer calls
    y = plan.run()
    assert torch.equal(y[0], q1(w_dense)) and torch.equal(y[1], q2(w_view.contiguous()).reshape(y[1].shape))
    first = y[2]
    w_reuse.mul_(0.25)
    again = plan.run()[2]
    assert again is first                                  # the reuse contract: later calls return the first output object
    q3.disable_reuse_quantizer()
    fresh = plan.run()[2]                                  # flag change -> plan rebuilt, tensor back in the fused launch
    assert not torch.equal(fresh, first) and torch.equal(fresh, q3(w_reuse))
    if torch.cuda.device_count() > 1:
        w_far = w_dense.to("cuda:1")
        plan2 = WeightPlan([("a", w_dense, q1), ("far", w_far, q1)])
        ya, yf = plan2.run()
        assert yf.device == w_far.device and torch.equal(ya.cpu(), yf.cpu())


def test_inplace_parameter_edits_are_noticed(Q):
    rng = np.random.default_rng(2)
    w = torch.from_numpy((rng.standard_normal((12, 264)) * 0.05).astype(np.float32)).to(DEV)
    thr = [float(v) for v in w.abs().amax(1)]
    lut = [float(v) for v in sorted(rng.choice(np.arange(-128, 128), size=16, replace=False))]
    ql = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, thr, True, 0, 2)
    qs = Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)
    y0, s0 = ql(w), qs(w)
    ql._threshold_torch.mul_(2.0)                           # in place: same data_ptr, new version
    qs.scales.mul_(2.0)
    y1, s1 = ql(w), qs(w)
    thr2 = (np.asarray(thr, np.float64).astype(np.float32) * np.float32(2.0))
    want = oracle.fq_lut(w.cpu().numpy(), oracle.F32, np.asarray(lut, np.float32), thr2, 12, 264, 8, True, 1e-8)
    assert G.bits_equal(y1.cpu().numpy(), np.asarray(want).reshape(y1.shape))
    assert not torch.equal(y0, y1)
    sc = (np.asarray(thr, np.float64) / 128).astype(np.float32) * np.float32(2.0)
    want_s = oracle.fq_affine(w.cpu().numpy(), oracle.F32, sc, np.zeros(12, np.int32), 12, 264, -128, 127)
    assert G.bits_equal(s1.cpu().numpy(), np.asarray(want_s).reshape(s1.shape)) and not torch.equal(s0, s1)


def test_fused_holder_wide_range_falls_back(Q):
    import mct_quantizers_b200 as mctq
    q = Q.ActivationSymmetricInferableQuantizer(23, [4.0], True)           # 2^23 codes: outside the fused kernel's fast rounding
    fh = mctq.PytorchFusedActivationQuantizationHolder(q, "relu")
    x = torch.randn(5000, device=DEV) * 3
    y = fh(x)
    assert torch.equal(y, q(torch.relu(x)))


def test_activation_plan_matches_per_holder_calls_and_oracle(Q):
    """One launch over many per-tensor sites (mctq_fq_affine_scalar_multi) == the holders called one by one == the oracle:
    mixed dtypes, ragged sizes, a channels_last tensor, more sites than one launch holds (64), a 23-bit range (rint path),
    a LUT holder and a misaligned view (both fall back to their own call); the plan rebuilds when an input moves."""
    import mct_quantizers_b200 as mctq
    rng = np.random.default_rng(3)
    quants = [Q.ActivationUniformInferableQuantizer(8, [-1.3], [2.9]), Q.ActivationSymmetricInferableQuantizer(8, [3.7], True),
              Q.ActivationPOTInferableQuantizer(4, [2.0], False), Q.ActivationSymmetricInferableQuantizer(23, [4.0], True)]
    pairs = []
    sizes = [1, 7, 2048, 2049, 4097, 70001, 8192 * 3 + 5]
    for k in range(70):
        dt = (torch.float32, torch.bfloat16, torch.float16)[k % 3]
        n = sizes[k % len(sizes)]
        x = torch.from_numpy((rng.standard_normal(n) * 2).astype(np.float32)).to(dt).to(DEV)
        pairs.append((mctq.PytorchActivationQuantizationHolder(quants[k % 4]), x))
    cl = torch.randn(2, 8, 5, 6, device=DEV).contiguous(memory_format=torch.channels_last)
    pairs.append((quants[0], cl))
    lut_q = Q.ActivationLutPOTInferableQuantizer(4, [-8.0, -3.0, 0.0, 1.0, 5.0, 7.0], [4.0], True)
    pairs.append((lut_q, torch.randn(300, device=DEV)))
    pairs.append((quants[1], torch.randn(1001, device=DEV)[1:]))              # 4-byte aligned view
    plan = mctq.ActivationPlan(pairs)
    assert len(plan.other) == 2 and len(plan._plans) == 1 and plan._plans[0][1].n_sites == 71
    ys = plan.run()
    torch.cuda.synchronize()
    for (h, x), y in zip(pairs, ys):
        want = h(x)
        assert y.dtype == want.dtype and y.shape == want.shape and y.stride() == want.stride()
        assert torch.equal(y.view(torch.int32) if y.dtype == torch.float32 else y.view(torch.int16),
                           want.view(torch.int32) if y.dtype == torch.float32 else want.view(torch.int16))
    q = quants[0]
    x, y = pairs[4][1], ys[4]
    want = oracle.fq_affine(G.from_torch(x), oracle.BF16, np.array([q.scale], np.float64).astype(np.float32),
                            np.array([q.zero_point], np.int32), 1, 1, 0, 255)
    assert G.bits_equal(G.from_torch(y), np.asarray(want).reshape(-1))
    # a moved input: same values in new storage -> rebuilt plan, same result; edited values -> new result
    old = pairs[5][1]
    plan.pairs[5] = (plan.pairs[5][0], old.clone() * 0.5)
    y5 = plan.run()[5]
    assert torch.equal(y5, pairs[5][0](old * 0.5))
    assert mctq.quantize_activations(pairs[:3])[2].shape == pairs[2][1].shape


def test_activation_plan_c_abi_argument_errors():
    import ctypes
    from mct_quantizers_b200 import _native
    lib = _native.load()
    x = torch.zeros(64, device=DEV)
    y = torch.empty_like(x)
    d = (_native.MctqSiteDesc * 1)()
    d[0].x, d[0].y, d[0].n, d[0].dtype, d[0].scale, d[0].zp, d[0].qmin, d[0].qmax = x.data_ptr(), y.data_ptr(), 64, 0, 0.5, 0, -128, 127
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.mctq_fq_affine_scalar_multi(ctypes.cast(d, ctypes.c_void_p), 1, st) == 0
    d[0].dtype = 9
    assert lib.mctq_fq_affine_scalar_multi(ctypes.cast(d, ctypes.c_void_p), 1, st) == -2
    d[0].dtype, d[0].qmin = 0, 300
    assert lib.mctq_fq_affine_scalar_multi(ctypes.cast(d, ctypes.c_void_p), 1, st) == -3
    d[0].qmin, d[0].x = -128, x.data_ptr() + 4
    assert lib.mctq_fq_affine_scalar_multi(ctypes.cast(d, ctypes.c_void_p), 1, st) == -1
    assert lib.mctq_fq_affine_scalar_multi(None, 0, st) == 0
    torch.cuda.synchronize()


def test_private_stream_early_order_keeps_dependent_chains_correct(Q):
    """Opt-in early order (loads before griddepcontrol.wait): independent back-to-back calls and chains in which every call
    consumes the previous call's output give the same bits as the default order."""
    import mct_quantizers_b200 as mctq
    from mct_quantizers_b200 import _native
    g = torch.Generator(device=DEV).manual_seed(7)
    xs = [torch.empty(1 << 22, device=DEV).uniform_(-6, 6, generator=g) for _ in range(6)]
    qs = [Q.ActivationUniformInferableQuantizer(8, [-1.0 - 0.1 * k], [2.0 + 0.3 * k]) for k in range(6)]

    def chain():
        outs = []
        for x in xs:                                   # independent inputs (early order applies) ...
            y = x
            for q in qs:                               # ... each followed by a chain: input = previous output (late order)
                y = q(y)
            outs.append(y)
        fh = mctq.PytorchFusedActivationQuantizationHolder(qs[0], "add_relu")
        outs.append(fh(outs[0], outs[1]))
        return outs

    want = chain()
    torch.cuda.synchronize()
    with mctq.private_stream():
        assert _native.load().mctq_set_tuning(3, 3) == 3
        got = chain()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):                     # a stream the library has not seen: first launch falls back to the late order
            s.wait_stream(torch.cuda.current_stream())
            got2 = chain()
        s.synchronize()
    assert _native.load().mctq_set_tuning(3, 1) == 1   # restored on exit
    torch.cuda.synchronize()
    for a, b, c in zip(want, got, got2):
        assert torch.equal(a, b) and torch.equal(a, c)


def test_code_emission_and_dequant_accept_host_tensors(Q):
    """quantize_affine_channel / dequantize_affine / lut_indices / the producer-fused op on HOST tensors: computed on the GPU
    (copied up, codes copied back), same bits as the device call and the oracle."""
    from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
    rng = np.random.default_rng(9)
    w = torch.from_numpy(rng.standard_normal((12, 40)).astype(np.float32))
    thr = w.abs().amax(1)
    scale = (thr / 128).float()
    zp = torch.zeros(12, dtype=torch.int32)
    codes_h, y_h = torch.ops.mctq.quantize_affine_channel(w, scale, zp, 0, -128, 127, 1, True)
    codes_d, y_d = torch.ops.mctq.quantize_affine_channel(w.to(DEV), scale.to(DEV), zp.to(DEV), 0, -128, 127, 1, True)
    assert not codes_h.is_cuda and not y_h.is_cuda
    assert torch.equal(codes_h, codes_d.cpu()) and torch.equal(y_h, y_d.cpu())
    want, want_codes = oracle.fq_affine(w.numpy(), oracle.F32, scale.numpy(), zp.numpy(), 12, 40, -128, 127, want_codes=True)
    assert G.bits_equal(y_h.numpy(), np.asarray(want).reshape(y_h.shape))
    assert np.array_equal(codes_h.numpy().astype(np.int32).reshape(-1), np.asarray(want_codes).reshape(-1))
    back = torch.ops.mctq.dequantize_affine(codes_h, 1, True, list(w.shape), scale, zp, 0)
    assert not back.is_cuda and torch.equal(back, y_h)
    lut = [float(v) for v in sorted(rng.choice(np.arange(-128, 128), size=16, replace=False))]
    table = lut_search_table(np.asarray(lut, np.float32), 8, True)
    i_h = torch.ops.mctq.lut_indices(w, table, 16, thr.float(), True, 0, 1e-8, 2)
    i_d = torch.ops.mctq.lut_indices(w.to(DEV), table, 16, thr.float().to(DEV), True, 0, 1e-8, 2)
    assert not i_h.is_cuda and torch.equal(i_h, i_d.cpu())
    f_h = torch.ops.mctq.fq_affine_scalar_pre(w, None, 1, 0.02, 0, 0, 255)
    assert not f_h.is_cuda and torch.equal(f_h, torch.ops.mctq.fq_affine_scalar_pre(w.to(DEV), None, 1, 0.02, 0, 0, 255).cpu())


def test_private_stream_orders_respect_every_hazard_between_own_launches():
    """Opt-in overlap (orders "early" / "free"): sequences with read-after-write, write-after-read and write-after-write
    hazards between consecutive launches of the library give the bits of the default order.  Large tensors, so that
    consecutive kernels really could overlap."""
    import ctypes
    from mct_quantizers_b200 import _native
    lib = _native.load()
    n = 48 << 20
    g = torch.Generator(device=DEV).manual_seed(11)
    src = [torch.empty(n, device=DEV).uniform_(-4, 4, generator=g) for _ in range(3)]
    st = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731

    def fq(a, b, scale, m=n):
        assert lib.mctq_fq_affine_scalar(ctypes.c_void_p(a.data_ptr()), ctypes.c_void_p(b.data_ptr()), None, m, 0, scale, 3, 0, 255, 0, st()) == 0

    def sequence():
        x, z, u = (t.clone() for t in src)
        y, w, v = torch.empty(n, device=DEV), torch.empty(n, device=DEV), torch.empty(n, device=DEV)
        torch.cuda.synchronize()
        fq(x, y, 0.031)              # A
        fq(z, x, 0.017)              # B writes A's input            (write-after-read)
        fq(x, w, 0.023)              # C reads B's output            (read-after-write)
        fq(u, w[: n // 2], 0.011, n // 2)   # D overwrites half of C's output (write-after-write)
        fq(u, v, 0.05)               # E, F, G: independent of everything in flight -> may run without waiting
        fq(z, y, 0.04)               # (y was A's output: A has long finished being relevant, but the range check must hold)
        fq(v, u, 0.02)               # reads E's output, writes E's input
        for k in range(6):           # a run of independent launches: every third one must wait again
            fq(src[k % 3], [y, w, v][k % 3], 0.01 * (k + 1))
        torch.cuda.synchronize()
        return [t.clone() for t in (x, y, w, v, u)]

    want = sequence()
    for mode in (2, 3):
        prev = lib.mctq_set_tuning(3, mode)
        try:
            for _ in range(3):
                got = sequence()
                for a, b in zip(want, got):
                    assert torch.equal(a, b), mode
        finally:
            lib.mctq_set_tuning(3, prev)


def test_activation_quantizers_cut_the_autograd_graph_like_the_reference(Q):
    """The reference runs torch.fake_quantize_per_tensor_affine under `with torch.no_grad():`
    (activation_symmetric_inferable_quantizer.py:112, activation_uniform_inferable_quantizer.py:123), so its
    activation quantizers return tensors that do NOT require grad even when the input does; the weights quantizers
    clear `requires_grad` on their input (weights_symmetric_inferable_quantizer.py:138).  Same here, through the holder
    (CUDA tensor: lean launch; torch.ops path: FakeTensor-visible operator)."""
    from mct_quantizers_b200.pytorch.activation_quantization_holder import PytorchActivationQuantizationHolder
    x = torch.randn(4, 33, device=DEV, requires_grad=True)
    for q in (Q.ActivationSymmetricInferableQuantizer(8, [4.0], True), Q.ActivationPOTInferableQuantizer(8, [2.0], False),
              Q.ActivationUniformInferableQuantizer(8, [-1.0], [2.3]),
              Q.ActivationLutPOTInferableQuantizer(4, [-8.0, -2.0, 0.0, 3.0, 7.0], [2.0], True, 4, 1e-8)):
        y = PytorchActivationQuantizationHolder(q)(x * 1.0)
        assert not y.requires_grad and y.grad_fn is None
    w = torch.nn.Parameter(torch.randn(8, 16, device=DEV))
    yw = Q.WeightsSymmetricInferableQuantizer(8, [1.0] * 8, True, 0)(w)
    assert not yw.requires_grad and not w.requires_grad


@pytest.mark.parametrize("pdl_mode", [1, 2, 3])
def test_tables_staged_before_the_wait_never_see_a_blob_being_prepared(Q, pdl_mode):
    """Kernels stage their prepared parameter tables BEFORE the dependent-launch wait unless the blob was written by a
    prepare call still in flight on the stream (mctq_host.cu, plan_launch).  Worst case for that rule: a long launch keeps
    the GPU busy, a NEW quantizer is prepared (the allocator tends to hand out the address of the blob freed one
    iteration earlier) and used at once -- a kernel that read the blob too early would see the previous iteration's
    thresholds."""
    from mct_quantizers_b200 import _native
    lib = _native.load()
    rng = np.random.default_rng(5)
    busy = torch.empty(96 << 20, device=DEV).uniform_(-4, 4)
    qa = Q.ActivationUniformInferableQuantizer(8, [-1.0], [2.0])
    C, L = 256, 8192
    w = torch.from_numpy(rng.standard_normal((C, L)).astype(np.float32)).to(DEV)
    wb = w.to(torch.bfloat16)
    lut = [-8.0, -5.0, -3.0, -1.0, 0.0, 1.0, 2.0, 4.0, 6.0, 7.0]
    prev = lib.mctq_set_tuning(3, pdl_mode)
    try:
        for it in range(6):
            thr = [float(v) for v in rng.uniform(0.5, 4.0, C)]
            qa(busy)                                                     # ~100 us of work in front of the prepare
            qs = Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)
            ys = qs(w)
            ys2 = qs(w)                                                  # second use: tables staged early
            qa(busy)
            ql = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, thr, True, 0, 2, 4)
            yl = ql(wb)
            yl2 = ql(wb)
            torch.cuda.synchronize()
            want_s = _oracle_sym(w, thr)
            assert G.bits_equal(ys.cpu().numpy(), np.asarray(want_s).reshape(ys.shape)), it
            assert torch.equal(ys, ys2)
            want_l = oracle.fq_lut(G.from_torch(wb), oracle.BF16, np.asarray(lut, np.float32), np.asarray(thr, np.float64).astype(np.float32),
                                   C, L, 4, True, 1e-8)
            assert G.bits_equal(yl.cpu().numpy(), np.asarray(want_l).reshape(yl.shape)), it
            assert torch.equal(yl, yl2)
            del qs, ql
    finally:
        lib.mctq_set_tuning(3, prev)


def test_nvtx_ranges_can_be_switched_on():
    """mctq_set_tuning key 9: NVTX ranges around the C-ABI entry points (no profiler attached here: the calls must be
    harmless and the results unchanged)."""
    from mct_quantizers_b200 import _native
    lib = _native.load()
    x = torch.randn(1 << 16, device=DEV)
    q = __import__("mct_quantizers_b200.pytorch.quantizers", fromlist=["x"]).ActivationUniformInferableQuantizer(8, [-1.0], [2.0])
    want = q(x)
    prev = lib.mctq_set_tuning(9, 1)
    try:
        assert prev == 0
        assert torch.equal(q(x), want)
    finally:
        assert lib.mctq_set_tuning(9, prev) == 1


def test_lut_outputs_follow_the_reference_in_shape_and_strides(Q):
    """Two things the differential fuzzer (tools/differential_fuzz.py, against the unmodified reference on the B200) found:
    the reference's eager LUT composition (argmin + gather) returns a ROW-MAJOR tensor whatever the input's strides (the
    affine quantizers keep the input's strides, like ATen), and a 0-dim input of a per-tensor LUT weights quantizer comes
    back 1-D because the result is multiplied by the threshold tensor of shape (1,)."""
    lut = [-8.0, -3.0, 0.0, 2.0, 7.0]
    x = torch.randn(4, 6, 5, 3, device=DEV).contiguous(memory_format=torch.channels_last)
    qa = Q.ActivationLutPOTInferableQuantizer(4, lut, [2.0], True, 4)
    ya = qa(x)
    assert ya.is_contiguous() and torch.equal(ya, qa(x.contiguous()))
    qw = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, [1.5], False, None, None, 4)
    yw = qw(x.clone())
    assert yw.is_contiguous() and torch.equal(yw, qw(x.contiguous()))
    xt = torch.randn(7, 12, device=DEV).t()
    qc = Q.WeightsLUTSymmetricInferableQuantizer(4, lut, [1.0 + 0.1 * k for k in range(12)], True, 0, 2, 4)
    yc = qc(xt.clone())
    assert yc.is_contiguous() and torch.equal(yc, qc(xt.contiguous()))
    # affine: strides preserved
    qs = Q.ActivationSymmetricInferableQuantizer(8, [4.0], True)
    assert qs(x).stride() == x.stride()
    # 0-dim
    s = torch.tensor(0.7, device=DEV)
    assert qw(s.clone()).shape == (1,) and qa(s).shape == () and qs(s).shape == ()


def test_concurrent_threads_on_their_own_streams(Q):
    """Four Python threads, each on its own CUDA stream, hammer the same quantizer objects (ctypes releases the GIL inside
    the native calls, so launches, the per-stream dependent-launch bookkeeping and the prepared-parameter caches really
    run concurrently): every result equals the single-threaded one."""
    import threading
    rng = np.random.default_rng(77)
    w = torch.from_numpy(rng.standard_normal((48, 1024)).astype(np.float32)).to(DEV)
    x = torch.from_numpy(rng.standard_normal((8, 3, 64, 64)).astype(np.float32)).to(DEV)
    thr = [float(v) for v in w.abs().amax(1)]
    qs = [Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0),
          Q.WeightsLUTSymmetricInferableQuantizer(4, [-100.0, -30.0, -8.0, 0.0, 5.0, 21.0, 77.0, 127.0], thr, True, 0, 2),
          Q.ActivationUniformInferableQuantizer(8, [-1.0], [2.5]),
          Q.ActivationLutPOTInferableQuantizer(4, [-8.0, -3.0, 0.0, 2.0, 7.0], [2.0], True, 4)]
    ins = [w, w, x, x]
    want = [q(t.clone()) for q, t in zip(qs, ins)]
    torch.cuda.synchronize()
    errors = []

    def work(k):
        try:
            st = torch.cuda.Stream()
            with torch.cuda.stream(st):
                for it in range(150):
                    j = (it + k) % len(qs)
                    y = qs[j](ins[j])
                    if it % 10 == 0:
                        st.synchronize()
                        if not torch.equal(y, want[j]):
                            errors.append((k, it, j))
            st.synchronize()
        except Exception as e:          # noqa: BLE001
            errors.append((k, repr(e)))

    threads = [threading.Thread(target=work, args=(k,)) for k in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:5]
