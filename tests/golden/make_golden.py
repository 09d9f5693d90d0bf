#!/usr/bin/env python
"""Generate the golden fixtures in this directory by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference, CPU torch):

    python tests/golden/make_golden.py

It imports ``mct_quantizers`` 1.6.0 from /root/reference, instantiates each of the nine PyTorch
inferable quantizers over a grid of constructor arguments, feeds seeded inputs (random, special
values and a boundary-dense set: every rounding tie (k + 1/2) * scale +- {0..3} ulp, every LUT
mid-point +- {0..3} ulp, all 2^16 bit patterns for half-precision per-tensor cases) and stores
inputs, outputs and the constructor-derived parameters.  The reference has no golden vectors of its
own (SURVEY.md 8c), so these fixtures are what pins the oracle and the CUDA path.

Outputs: golden_v1.npz, golden_v1_2.npz, ... (arrays, each file below 1 MB) + golden_v1.json (manifest,
which lists the archives).  Half-precision tensors are stored as uint16 bit patterns; the all-bit-pattern
inputs are not stored, tests/golden_util.py regenerates them.  The reference cannot travel to the GPU box; the fixtures do.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gen_common import *  # noqa: E402,F401,F403  (Q, torch, arrays, manifest, helpers)
from gen_common import Q, torch, manifest, add_case, affine_channel_input, build_tensor, all_finite_half_patterns, \
    lut_channel_input, save, TORCH_DT  # noqa: E402

rng = np.random.default_rng(20261017)

# ----------------------------------------------------------------------------------- affine: weights
W_SHAPES = [((6, 5, 3, 3), 0), ((4, 7, 3, 5), 1), ((3, 4, 9, 5), 2), ((2, 5, 4, 11), 3), ((16, 24), 0), ((24, 16), 1),
            ((10,), 0)]


def rand_thresholds(C, pot=False):
    if pot:
        return [float(2.0 ** int(e)) for e in rng.integers(-5, 4, size=C)]
    return [float(v) for v in np.abs(rng.normal(0, 1.5, size=C)) + 0.05]


for cls_name, pot in (("WeightsSymmetricInferableQuantizer", False), ("WeightsPOTInferableQuantizer", True)):
    for bits in (2, 3, 4, 8):
        for shape, axis in W_SHAPES:
            if bits in (3,) and len(shape) != 4:
                continue
            C = shape[axis]
            thr = rand_thresholds(C, pot)
            scales = (np.asarray(thr) / 2 ** (bits - 1)).astype(np.float32)
            L = int(np.prod(shape)) // C
            L_gen = max(L, 1)
            vecs = [affine_channel_input(rng, scales[c], 0, -2 ** (bits - 1), 2 ** (bits - 1) - 1, L_gen) for c in range(C)]
            x = torch.from_numpy(build_tensor(vecs, shape, axis))
            add_case(f"w_{'pot' if pot else 'sym'}_b{bits}_pc_{'x'.join(map(str, shape))}_ax{axis}", cls_name,
                     dict(num_bits=bits, threshold=thr, per_channel=True, channel_axis=axis), x)
        # per-tensor (tensor qparams path)
        thr = rand_thresholds(1, pot)
        sc = np.float32(thr[0] / 2 ** (bits - 1))
        v = affine_channel_input(rng, sc, 0, -2 ** (bits - 1), 2 ** (bits - 1) - 1, 4096)
        add_case(f"w_{'pot' if pot else 'sym'}_b{bits}_pt", cls_name,
                 dict(num_bits=bits, threshold=thr, per_channel=False), torch.from_numpy(v.reshape(4, 8, 128)))

# half-precision weights (f32 scales, bf16/f16 data; reference accepts them, SURVEY 8a-a3)
for dt in ("bfloat16", "float16"):
    shape, axis, bits = (6, 5, 3, 3), 0, 8
    thr = rand_thresholds(shape[axis])
    scales = (np.asarray(thr) / 2 ** (bits - 1)).astype(np.float32)
    vecs = [affine_channel_input(rng, scales[c], 0, -128, 127, 45) for c in range(shape[axis])]
    x = torch.from_numpy(build_tensor(vecs, shape, axis)).to(TORCH_DT[dt])
    add_case(f"w_sym_b8_pc_{dt}", "WeightsSymmetricInferableQuantizer",
             dict(num_bits=bits, threshold=thr, per_channel=True, channel_axis=axis), x)
    x = all_finite_half_patterns(dt)
    add_case(f"w_sym_b4_pt_{dt}_allbits", "WeightsSymmetricInferableQuantizer",
             dict(num_bits=4, threshold=[1.7], per_channel=False), x, x_gen="all_finite_half_patterns")

# uniform weights: straddling, strictly positive, strictly negative ranges (range fixing) + zp truncation
for bits in (2, 4, 8):
    for shape, axis in W_SHAPES[:5]:
        C = shape[axis]
        lo = rng.normal(-1.0, 1.0, size=C)
        hi = lo + np.abs(rng.normal(0, 2.0, size=C)) + 0.1
        if C >= 3:
            lo[0], hi[0] = 0.3, 2.1       # min > 0  -> (0, max)
            lo[1], hi[1] = -2.5, -0.4     # max < 0  -> (min, 0)
        min_range, max_range = [float(v) for v in lo], [float(v) for v in hi]
        probe = Q.WeightsUniformInferableQuantizer(bits, min_range, max_range, True, axis)
        sc, zp = probe.scales.numpy(), probe.zero_points.numpy()
        L = int(np.prod(shape)) // C
        vecs = [affine_channel_input(rng, sc[c], int(zp[c]), 0, 2 ** bits - 1, L) for c in range(C)]
        x = torch.from_numpy(build_tensor(vecs, shape, axis))
        add_case(f"w_uni_b{bits}_pc_{'x'.join(map(str, shape))}_ax{axis}", "WeightsUniformInferableQuantizer",
                 dict(num_bits=bits, min_range=min_range, max_range=max_range, per_channel=True, channel_axis=axis), x)
    for tag, (a, b) in {"straddle": (-1.3, 2.45), "pos": (0.2, 3.0), "neg": (-4.0, -0.5)}.items():
        probe = Q.WeightsUniformInferableQuantizer(bits, [a], [b], False)
        v = affine_channel_input(rng, probe.scales.numpy()[0], int(probe.zero_points.numpy()[0]), 0, 2 ** bits - 1, 4096)
        add_case(f"w_uni_b{bits}_pt_{tag}", "WeightsUniformInferableQuantizer",
                 dict(num_bits=bits, min_range=[a], max_range=[b], per_channel=False), torch.from_numpy(v.reshape(64, 64)))

# ------------------------------------------------------------------------------- affine: activations
for cls_name, thr_list in (("ActivationSymmetricInferableQuantizer", [3.7, 0.61]), ("ActivationPOTInferableQuantizer", [4.0, 0.125])):
    for signed in (True, False):
        for bits in (2, 4, 8):
            for thr in thr_list:
                if signed:
                    sc, qmin, qmax = np.float32(thr / 2 ** (bits - 1)), -2 ** (bits - 1), 2 ** (bits - 1) - 1
                else:
                    sc, qmin, qmax = np.float32(thr / 2 ** bits), 0, 2 ** bits - 1
                v = affine_channel_input(rng, sc, 0, qmin, qmax, 6000)
                tag = f"a_{'pot' if 'POT' in cls_name else 'sym'}_b{bits}_{'s' if signed else 'u'}_t{thr}"
                add_case(tag, cls_name, dict(num_bits=bits, threshold=[thr], signed=signed),
                         torch.from_numpy(v.reshape(2, 3, 10, 100)))
for dt in ("bfloat16", "float16"):
    x = all_finite_half_patterns(dt)
    add_case(f"a_sym_b8_s_{dt}_allbits", "ActivationSymmetricInferableQuantizer", dict(num_bits=8, threshold=[3.7], signed=True), x,
             x_gen="all_finite_half_patterns")
    add_case(f"a_pot_b8_u_{dt}_allbits", "ActivationPOTInferableQuantizer", dict(num_bits=8, threshold=[4.0], signed=False), x,
             x_gen="all_finite_half_patterns")
    add_case(f"a_uni_b8_{dt}_allbits", "ActivationUniformInferableQuantizer", dict(num_bits=8, min_range=[-1.0], max_range=[2.3]), x,
             x_gen="all_finite_half_patterns")

for bits in (2, 4, 7, 8):
    for tag, (a, b) in {"straddle": (-1.0, 2.3), "sym4": (-4.0, 4.0), "pos": (0.25, 6.0), "neg": (-3.0, -0.7)}.items():
        probe = Q.ActivationUniformInferableQuantizer(bits, [a], [b])
        v = affine_channel_input(rng, np.float32(probe.scale), probe.zero_point, 0, 2 ** bits - 1, 6000)
        add_case(f"a_uni_b{bits}_{tag}", "ActivationUniformInferableQuantizer",
                 dict(num_bits=bits, min_range=[a], max_range=[b]), torch.from_numpy(v.reshape(4, 1500)))

# ------------------------------------------------------------------------------------------- LUT
LUT16 = [float(v) for v in sorted(rng.choice(np.arange(-128, 128), size=16, replace=False))]
LUT16_UNSORTED_DUP = [25.0, -100.0, 0.0, 25.0, 127.0, -128.0, 64.0, -7.0, -100.0, 3.0, 4.0, 90.0, -64.0, -33.0, 12.0, 0.0]
LUT4 = [-25.0, 0.0, 25.0, 100.0]
LUT32 = [float(v) for v in rng.permutation(np.arange(-128, 128, 8))]
LUT64 = [float(v) for v in rng.permutation(np.arange(-128, 128, 4))]
LUT_U16 = [float(v) for v in sorted(rng.choice(np.arange(0, 256), size=16, replace=False))]


for cls_name, pot in (("WeightsLUTSymmetricInferableQuantizer", False), ("WeightsLUTPOTInferableQuantizer", True)):
    for lut_name, lut, bits in (("lut16", LUT16, 4), ("lut16dup", LUT16_UNSORTED_DUP, 4), ("lut4", LUT4, 2),
                                ("lut32", LUT32, 5), ("lut64", LUT64, 6)):
        for shape, axis in (((6, 40), 0), ((33, 5), 1), ((4, 3, 2, 30), 1), ((2, 30, 3, 3), 3), ((5, 3, 16, 2), 0)):
            if lut_name in ("lut32", "lut64", "lut4") and len(shape) != 2:
                continue
            C = shape[axis]
            thr = rand_thresholds(C, pot)
            if not pot:
                thr[0] = 0.013      # < 0.25: eps perturbs the divisor
            L = int(np.prod(shape)) // C
            vecs = [lut_channel_input(rng, lut, thr[c], 8, True, L) for c in range(C)]
            x = torch.from_numpy(build_tensor(vecs, shape, axis))
            args = dict(num_bits=bits, lut_values=lut, threshold=thr, per_channel=True, channel_axis=axis,
                        input_rank=len(shape))
            thr_t = torch.tensor(thr, dtype=torch.float32).reshape([-1 if i == axis else 1 for i in range(len(shape))])
            add_case(f"wl_{'pot' if pot else 'sym'}_{lut_name}_pc_{'x'.join(map(str, shape))}_ax{axis}", cls_name, args, x,
                     lut_info=dict(threshold=thr_t, bw=8, signed=True, eps=1e-8))
        thr = rand_thresholds(1, pot)
        v = lut_channel_input(rng, lut, thr[0], 8, True, 3000)
        add_case(f"wl_{'pot' if pot else 'sym'}_{lut_name}_pt", cls_name,
                 dict(num_bits=bits, lut_values=lut, threshold=thr, per_channel=False), torch.from_numpy(v.reshape(30, 100)),
                 lut_info=dict(threshold=torch.tensor(thr, dtype=torch.float32), bw=8, signed=True, eps=1e-8))

# non-default lut_values_bitwidth / eps, half-precision weights (output stays f32)
thr = rand_thresholds(6)
vecs = [lut_channel_input(rng, [-8.0, -3.0, 0.0, 7.0], thr[c], 4, True, 200, eps=1e-3) for c in range(6)]
add_case("wl_sym_bw4_eps1e-3", "WeightsLUTSymmetricInferableQuantizer",
         dict(num_bits=2, lut_values=[-8.0, -3.0, 0.0, 7.0], threshold=thr, per_channel=True, channel_axis=0, input_rank=2,
              lut_values_bitwidth=4, eps=1e-3), torch.from_numpy(build_tensor(vecs, (6, 200), 0)),
         lut_info=dict(threshold=torch.tensor(thr, dtype=torch.float32).reshape(-1, 1), bw=4, signed=True, eps=1e-3))
for dt in ("bfloat16", "float16"):
    thr = rand_thresholds(5)
    vecs = [lut_channel_input(rng, LUT16, thr[c], 8, True, 600) for c in range(5)]
    x = torch.from_numpy(build_tensor(vecs, (5, 600), 0)).to(TORCH_DT[dt])
    add_case(f"wl_sym_lut16_pc_{dt}", "WeightsLUTSymmetricInferableQuantizer",
             dict(num_bits=4, lut_values=LUT16, threshold=thr, per_channel=True, channel_axis=0, input_rank=2), x,
             lut_info=dict(threshold=torch.tensor(thr, dtype=torch.float32).reshape(-1, 1), bw=8, signed=True, eps=1e-8))

for signed, lut in ((True, LUT16), (True, LUT16_UNSORTED_DUP), (False, LUT_U16)):
    for thr in (4.0, 0.125, 0.0625, 32.0):
        v = lut_channel_input(rng, lut, thr, 8, signed, 6000)
        add_case(f"al_{'s' if signed else 'u'}_{'dup' if lut is LUT16_UNSORTED_DUP else 'l16'}_t{thr}",
                 "ActivationLutPOTInferableQuantizer",
                 dict(num_bits=4, lut_values=lut, threshold=[thr], signed=signed), torch.from_numpy(v.reshape(6, 10, 100)),
                 lut_info=dict(threshold=thr, bw=8, signed=signed, eps=1e-8))
for dt in ("bfloat16", "float16"):
    x = all_finite_half_patterns(dt)
    for signed, lut in ((True, LUT16), (False, LUT_U16)):
        for thr in (4.0, 0.0625):
            add_case(f"al_{'s' if signed else 'u'}_t{thr}_{dt}_allbits", "ActivationLutPOTInferableQuantizer",
                     dict(num_bits=4, lut_values=lut, threshold=[thr], signed=signed), x,
                     lut_info=dict(threshold=thr, bw=8, signed=signed, eps=1e-8), x_gen="all_finite_half_patterns")

# range-fix constants asserted by the reference's own tests (test_fln_activation_quantizer_holder.py:42-45)
q = Q.ActivationUniformInferableQuantizer(7, [-4.0], [4.0])
manifest["range_fix_known_answers"] = {"num_bits": 7, "min": -4.0, "max": 4.0, "min_range": q.min_range,
                                       "max_range": q.max_range, "scale": q.scale, "zero_point": q.zero_point}

save("golden_v1")
