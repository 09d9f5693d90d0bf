"""Load the golden fixtures (generated from the unmodified reference by tests/golden/make_golden.py)
and run the CPU oracle on a fixture case.  Shared by the CPU and GPU test suites."""
import json
import os
from functools import lru_cache

import numpy as np
import torch

import oracle
from oracle import torch_cpu_port as port

HERE = os.path.dirname(os.path.abspath(__file__))
DT_TAG = {"float32": oracle.F32, "bfloat16": oracle.BF16, "float16": oracle.F16}
TORCH_DT = {"float32": torch.float32, "bfloat16": torch.bfloat16, "float16": torch.float16}


class _Arrays:
    """Read-only view over the arrays of several .npz batches (case names are unique across batches)."""

    def __init__(self, files):
        self._files = files

    def __getitem__(self, key):
        for f in self._files:
            if key in f.files:
                return f[key]
        raise KeyError(key)


@lru_cache(maxsize=1)
def _load():
    """golden_v1 (make_golden.py) + golden_v2 (make_golden_v2.py) + golden_v3 (make_golden_v3.py): one manifest, one array lookup."""
    manifest, files = None, []
    for stem in ("golden_v1", "golden_v2", "golden_v3"):
        with open(os.path.join(HERE, "golden", stem + ".json")) as f:
            m = json.load(f)
        if manifest is None:
            manifest = m
        else:
            manifest["cases"] = manifest["cases"] + m["cases"]
        files += [np.load(os.path.join(HERE, "golden", a)) for a in m.get("archives", [stem + ".npz"])]
    names = [c["name"] for c in manifest["cases"]]
    assert len(names) == len(set(names)), "duplicate golden case names"
    return manifest, _Arrays(files)


def manifest():
    return _load()[0]


def case_names():
    return [c["name"] for c in manifest()["cases"]]


def all_finite_half_patterns(dtype_name):
    """Every finite bfloat16 / float16 value as uint16 bit patterns, in increasing bit order: the input of the `_allbits`
    cases, which the fixtures do not store (tests/golden/gen_common.py, `x_gen`)."""
    bits = np.arange(1 << 16, dtype=np.uint32).astype(np.uint16)
    exponent = np.uint16(0x7F80 if dtype_name == "bfloat16" else 0x7C00)
    return bits[(bits & exponent) != exponent]


def get_case(name):
    m, arrays = _load()
    for c in m["cases"]:
        if c["name"] == name:
            out = dict(c)
            gen = c.get("x_gen")
            out["x"] = all_finite_half_patterns(c["x_dtype"]) if gen == "all_finite_half_patterns" else arrays[f"{name}/x"]
            out["y"] = arrays[f"{name}/y"]
            out["idx"] = arrays[f"{name}/idx"] if c.get("has_idx") else None
            out["p"] = {k: arrays[f"{name}/p/{k}"] for k, v in c["params"].items() if v["kind"] in ("tensor", "ndarray")}
            return out
    raise KeyError(name)


def to_torch(arr, dtype_name, device="cpu"):
    """Stored ndarray (uint16 bits for half types) -> torch tensor of the named dtype."""
    if dtype_name in ("bfloat16", "float16"):
        t = torch.from_numpy(arr.view(np.int16).copy()).view(TORCH_DT[dtype_name])
    else:
        t = torch.from_numpy(arr.copy())
    return t.to(device)


def from_torch(t):
    t = t.detach().cpu().contiguous()
    if t.dtype in (torch.bfloat16, torch.float16):
        return t.view(torch.int16).numpy().view(np.uint16)
    return t.numpy()


def derive_params(case):
    """Constructor args -> dict(kind, scale[C], zp[C], C, inner, qmin, qmax, ...) through the oracle's
    restatement of the reference's constructor math (oracle/torch_cpu_port.py)."""
    cls, a, shape = case["cls"], case["args"], case["shape"]
    if cls in ("WeightsSymmetricInferableQuantizer", "WeightsPOTInferableQuantizer"):
        scales, zps, qmin, qmax = port.weights_symmetric_qparams(a["threshold"], a["num_bits"])
        C, inner = oracle.channel_layout(shape, a.get("channel_axis") if a["per_channel"] else None)
        return dict(kind="affine", scale=scales.numpy(), zp=zps.numpy(), C=C, inner=inner, qmin=qmin, qmax=qmax)
    if cls == "WeightsUniformInferableQuantizer":
        lo, hi, scales, zps, qmin, qmax = port.weights_uniform_qparams(a["min_range"], a["max_range"], a["num_bits"])
        C, inner = oracle.channel_layout(shape, a.get("channel_axis") if a["per_channel"] else None)
        return dict(kind="affine", scale=scales.numpy(), zp=zps.numpy(), C=C, inner=inner, qmin=qmin, qmax=qmax,
                    min_range=lo.numpy(), max_range=hi.numpy())
    if cls in ("ActivationSymmetricInferableQuantizer", "ActivationPOTInferableQuantizer"):
        scales, qmin, qmax = port.symmetric_qparams(a["threshold"], a["num_bits"], a["signed"])
        s32 = np.array([float(scales[0])], dtype=np.float64).astype(np.float32)   # double -> float inside ATen
        return dict(kind="affine", scale=s32, zp=np.zeros(1, np.int32), C=1, inner=1, qmin=qmin, qmax=qmax,
                    scale_py=float(scales[0]))
    if cls == "ActivationUniformInferableQuantizer":
        lo, hi, scale, zp, qmin, qmax = port.activation_uniform_qparams(a["min_range"], a["max_range"], a["num_bits"])
        return dict(kind="affine", scale=np.array([scale], dtype=np.float64).astype(np.float32),
                    zp=np.array([zp], np.int32), C=1, inner=1, qmin=qmin, qmax=qmax,
                    scale_py=scale, zp_py=zp, min_range=lo, max_range=hi)
    if cls in ("WeightsLUTSymmetricInferableQuantizer", "WeightsLUTPOTInferableQuantizer"):
        C, inner = oracle.channel_layout(shape, a.get("channel_axis") if a["per_channel"] else None)
        return dict(kind="lut", lut=np.asarray(a["lut_values"], np.float32), thr=np.asarray(a["threshold"], np.float64).astype(np.float32),
                    C=C, inner=inner, bw=a.get("lut_values_bitwidth", 8), signed=True, eps=a.get("eps", 1e-8), act=False)
    if cls == "ActivationLutPOTInferableQuantizer":
        return dict(kind="lut", lut=np.asarray(a["lut_values"], np.float32), thr=float(a["threshold"][0]), C=1, inner=1,
                    bw=a.get("lut_values_bitwidth", 8), signed=a["signed"], eps=a.get("eps", 1e-8), act=True)
    raise KeyError(cls)


def oracle_run(case, x=None):
    """Run the C restatement on the case's input (or on `x`, same storage convention)."""
    p = derive_params(case)
    x = case["x"] if x is None else x
    tag = DT_TAG[case["x_dtype"]]
    if p["kind"] == "affine":
        y, codes = oracle.fq_affine(x, tag, p["scale"], p["zp"], p["C"], p["inner"], p["qmin"], p["qmax"], want_codes=True)
        return dict(y=y, codes=codes, p=p)
    y, idx = oracle.fq_lut(x, tag, p["lut"], p["thr"], p["C"], p["inner"], p["bw"], p["signed"], p["eps"],
                           activation_mode=p["act"], want_idx=True)
    return dict(y=y, idx=idx, p=p)


def bits_equal(a, b):
    """Bitwise equality of two same-dtype arrays (distinguishes -0.0 from +0.0, compares NaN payloads)."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    if a.dtype == np.float32:
        return bool(np.array_equal(a.view(np.uint32), b.view(np.uint32)))
    return bool(np.array_equal(a, b))


def mismatch_report(a, b, x=None, limit=5):
    a, b = np.ascontiguousarray(a).reshape(-1), np.ascontiguousarray(b).reshape(-1)
    va = a.view(np.uint32) if a.dtype == np.float32 else a
    vb = b.view(np.uint32) if b.dtype == np.float32 else b
    bad = np.nonzero(va != vb)[0]
    lines = [f"{bad.size} / {a.size} mismatches"]
    for i in bad[:limit]:
        xs = "" if x is None else f" x={np.ascontiguousarray(x).reshape(-1)[i]!r}"
        lines.append(f"  [{i}] got={a[i]!r} want={b[i]!r}{xs}")
    return "\n".join(lines)
