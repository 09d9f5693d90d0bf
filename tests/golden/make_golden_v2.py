#!/usr/bin/env python
"""Second batch of golden fixtures from the UNMODIFIED reference (build container only, CPU torch):

    python tests/golden/make_golden_v2.py        ->  golden_v2.npz + golden_v2.json

Cases the first batch (make_golden.py) does not have, chosen after the kernel variants that exist by the end of round 1:
half-precision uniform weights (per-channel zero points with bf16 / f16 data), 16-bit quantizers (65536 levels), channel-
innermost per-channel layouts with channel counts that are / are not multiples of 4 (f32 and half precision: the 8-byte
vector variant), rows that are multiples of 8 / of 4 / odd for half-precision LUT weights (8-element vectors with 256-bit
stores vs 4-element vectors vs straddling vectors), LUT grids other than 8 bit (6 and 10) with table sizes that are not
powers of two, sorted and unsorted centroid lists (index emission with and without the identity shortcut).
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gen_common import Q, torch, manifest, add_case, affine_channel_input, build_tensor, all_finite_half_patterns, \
    lut_channel_input, save, TORCH_DT  # noqa: E402

rng = np.random.default_rng(20261018)


def narrow(x, dt):
    """f32 tensor -> dtype `dt`; values that overflow to +-inf when narrowed (3e9, 1e6 in f16) become 0: non-finite inputs
    are outside the parity contract (the reference's per-channel CPU path maps +inf to qmin through an int64 overflow,
    SURVEY 8a hazard 3)."""
    y = x.to(TORCH_DT[dt])
    return torch.where(torch.isfinite(y), y, torch.zeros_like(y))


def thresholds(C, pot=False):
    if pot:
        return [float(2.0 ** int(e)) for e in rng.integers(-5, 4, size=C)]
    return [float(v) for v in np.abs(rng.normal(0, 1.5, size=C)) + 0.05]


def uniform_ranges(C):
    lo = rng.normal(-1.0, 1.0, size=C)
    hi = lo + np.abs(rng.normal(0, 2.0, size=C)) + 0.1
    if C >= 3:
        lo[0], hi[0] = 0.3, 2.1
        lo[1], hi[1] = -2.5, -0.4
    return [float(v) for v in lo], [float(v) for v in hi]


# ---- uniform weights on half-precision data, per-channel (non-zero zero points) and per-tensor over all bit patterns
for dt in ("bfloat16", "float16"):
    for shape, axis in (((6, 5, 3, 3), 0), ((24, 16), 1), ((12, 64), 0)):
        C = shape[axis]
        lo, hi = uniform_ranges(C)
        probe = Q.WeightsUniformInferableQuantizer(8, lo, hi, True, axis)
        sc, zp = probe.scales.numpy(), probe.zero_points.numpy()
        L = int(np.prod(shape)) // C
        vecs = [affine_channel_input(rng, sc[c], int(zp[c]), 0, 255, L) for c in range(C)]
        x = narrow(torch.from_numpy(build_tensor(vecs, shape, axis)), dt)
        add_case(f"w_uni_b8_pc_{'x'.join(map(str, shape))}_ax{axis}_{dt}", "WeightsUniformInferableQuantizer",
                 dict(num_bits=8, min_range=lo, max_range=hi, per_channel=True, channel_axis=axis), x)
    add_case(f"w_uni_b4_pt_{dt}_allbits", "WeightsUniformInferableQuantizer",
             dict(num_bits=4, min_range=[-0.7], max_range=[1.9], per_channel=False), all_finite_half_patterns(dt),
             x_gen="all_finite_half_patterns")

# ---- 16-bit quantizers
thr = thresholds(5)
scales = (np.asarray(thr) / 2 ** 15).astype(np.float32)
vecs = [affine_channel_input(rng, scales[c], 0, -32768, 32767, 1200) for c in range(5)]
add_case("w_sym_b16_pc_5x1200_ax0", "WeightsSymmetricInferableQuantizer",
         dict(num_bits=16, threshold=thr, per_channel=True, channel_axis=0), torch.from_numpy(build_tensor(vecs, (5, 1200), 0)))
probe = Q.ActivationUniformInferableQuantizer(16, [-1.0], [2.3])
v = affine_channel_input(rng, np.float32(probe.scale), probe.zero_point, 0, 65535, 8000)
add_case("a_uni_b16_straddle", "ActivationUniformInferableQuantizer", dict(num_bits=16, min_range=[-1.0], max_range=[2.3]),
         torch.from_numpy(v.reshape(8, 1000)))
v = affine_channel_input(rng, np.float32(4.0 / 2 ** 15), 0, -32768, 32767, 8000)
add_case("a_pot_b16_s_t4.0", "ActivationPOTInferableQuantizer", dict(num_bits=16, threshold=[4.0], signed=True),
         torch.from_numpy(v.reshape(8, 1000)))

# ---- channel-innermost per-channel layouts
for dt in ("float32", "bfloat16", "float16"):
    for shape in ((50, 64), (37, 12), (200, 3), (9, 7, 10)):
        axis = len(shape) - 1
        C = shape[axis]
        L = int(np.prod(shape)) // C
        thr = thresholds(C)
        scales = (np.asarray(thr) / 128).astype(np.float32)
        vecs = [affine_channel_input(rng, scales[c], 0, -128, 127, L) for c in range(C)]
        x = narrow(torch.from_numpy(build_tensor(vecs, shape, axis)), dt)
        add_case(f"w_sym_b8_pc_{'x'.join(map(str, shape))}_last_{dt}", "WeightsSymmetricInferableQuantizer",
                 dict(num_bits=8, threshold=thr, per_channel=True, channel_axis=axis), x)
    shape, axis = (40, 16), 1
    lo, hi = uniform_ranges(16)
    probe = Q.WeightsUniformInferableQuantizer(8, lo, hi, True, axis)
    sc, zp = probe.scales.numpy(), probe.zero_points.numpy()
    vecs = [affine_channel_input(rng, sc[c], int(zp[c]), 0, 255, 40) for c in range(16)]
    x = narrow(torch.from_numpy(build_tensor(vecs, shape, axis)), dt)
    add_case(f"w_uni_b8_pc_40x16_last_{dt}", "WeightsUniformInferableQuantizer",
             dict(num_bits=8, min_range=lo, max_range=hi, per_channel=True, channel_axis=axis), x)

# ---- LUT weights: row lengths x dtypes, grids other than 8 bit, table sizes that are not powers of two
LUT16_SORTED = [float(v) for v in sorted(rng.choice(np.arange(-128, 128), size=16, replace=False))]
LUT16_UNSORTED = [float(v) for v in rng.permutation(LUT16_SORTED)]
LUT5_BW6 = [-32.0, -9.0, 0.0, 14.0, 31.0]
LUT11_BW10 = [float(v) for v in sorted(rng.choice(np.arange(-512, 512), size=11, replace=False))]
for dt in ("float32", "bfloat16", "float16"):
    for shape in ((7, 264), (7, 44), (9, 27), (3, 8200)):
        for lut_name, lut in (("sorted", LUT16_SORTED), ("unsorted", LUT16_UNSORTED)):
            if lut_name == "unsorted" and shape != (7, 264):
                continue
            C = shape[0]
            thr = thresholds(C)
            vecs = [lut_channel_input(rng, lut, thr[c], 8, True, shape[1]) for c in range(C)]
            x = narrow(torch.from_numpy(build_tensor(vecs, shape, 0)), dt)
            add_case(f"wl_sym_{lut_name}_pc_{shape[0]}x{shape[1]}_{dt}", "WeightsLUTSymmetricInferableQuantizer",
                     dict(num_bits=4, lut_values=lut, threshold=thr, per_channel=True, channel_axis=0, input_rank=2), x,
                     lut_info=dict(threshold=torch.tensor(thr, dtype=torch.float32).reshape(-1, 1), bw=8, signed=True, eps=1e-8))
for lut_name, lut, bits, bw in (("lut5_bw6", LUT5_BW6, 3, 6), ("lut11_bw10", LUT11_BW10, 4, 10)):
    for pot in (False, True):
        thr = thresholds(6, pot)
        vecs = [lut_channel_input(rng, lut, thr[c], bw, True, 400) for c in range(6)]
        add_case(f"wl_{'pot' if pot else 'sym'}_{lut_name}_pc_6x400", "WeightsLUTPOTInferableQuantizer" if pot else "WeightsLUTSymmetricInferableQuantizer",
                 dict(num_bits=bits, lut_values=lut, threshold=thr, per_channel=True, channel_axis=0, input_rank=2, lut_values_bitwidth=bw),
                 torch.from_numpy(build_tensor(vecs, (6, 400), 0)),
                 lut_info=dict(threshold=torch.tensor(thr, dtype=torch.float32).reshape(-1, 1), bw=bw, signed=True, eps=1e-8))

# ---- LUT activations on a 6-bit grid, signed and unsigned, 7 centroids
for signed, lut in ((True, [-32.0, -20.0, -3.0, 0.0, 5.0, 17.0, 31.0]), (False, [0.0, 3.0, 9.0, 20.0, 33.0, 50.0, 63.0])):
    for thr in (2.0, 0.125):
        v = lut_channel_input(rng, lut, thr, 6, signed, 4000)
        add_case(f"al_{'s' if signed else 'u'}_lut7_bw6_t{thr}", "ActivationLutPOTInferableQuantizer",
                 dict(num_bits=3, lut_values=lut, threshold=[thr], signed=signed, lut_values_bitwidth=6),
                 torch.from_numpy(v.reshape(4, 1000)), lut_info=dict(threshold=thr, bw=6, signed=signed, eps=1e-8))
        for dt in ("bfloat16", "float16"):
            add_case(f"al_{'s' if signed else 'u'}_lut7_bw6_t{thr}_{dt}", "ActivationLutPOTInferableQuantizer",
                     dict(num_bits=3, lut_values=lut, threshold=[thr], signed=signed, lut_values_bitwidth=6),
                     narrow(torch.from_numpy(v.reshape(4, 1000)), dt), lut_info=dict(threshold=thr, bw=6, signed=signed, eps=1e-8))

save("golden_v2")
