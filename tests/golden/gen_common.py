"""Helpers shared by the golden-fixture generators (make_golden.py, make_golden_v2.py): they import the UNMODIFIED
reference from /root/reference, run it on CPU torch and collect inputs / outputs / constructor-derived parameters.
Build container only."""
import json
import os
import sys
import warnings
import zlib

import numpy as np

REF = os.environ.get("MCTQ_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
warnings.filterwarnings("ignore", category=SyntaxWarning)

import torch  # noqa: E402

import mct_quantizers  # noqa: E402
from mct_quantizers.pytorch import quantizers as Q  # noqa: E402
from mct_quantizers.pytorch.quantizer_utils import int_quantization_with_threshold  # noqa: E402

assert mct_quantizers.__version__ == "1.6.0"
assert not torch.cuda.is_available(), "fixtures must come from the reference's CPU path"

HERE = os.path.dirname(os.path.abspath(__file__))
TORCH_DT = {"float32": torch.float32, "bfloat16": torch.bfloat16, "float16": torch.float16}

arrays = {}
manifest = {"reference_version": mct_quantizers.__version__, "torch": torch.__version__,
            "numpy": np.__version__, "cases": []}


def store(t):
    """torch tensor -> ndarray (half types as uint16 bit patterns)."""
    t = t.detach().cpu().contiguous()
    if t.dtype in (torch.bfloat16, torch.float16):
        return t.view(torch.int16).numpy().view(np.uint16).copy()
    return t.numpy().copy()


def ulp_neighbourhood(v, k=3):
    """v (f32 array) -> all values within +-k ulp of each entry."""
    v = np.asarray(v, dtype=np.float32)
    bits = v.view(np.int32).astype(np.int64)
    # map to a monotone integer line so that stepping crosses zero correctly
    mono = np.where(bits < 0, -(bits & 0x7fffffff), bits)
    out = []
    for d in range(-k, k + 1):
        m = mono + d
        b = np.where(m < 0, (-m) | 0x80000000, m).astype(np.uint32)
        out.append(b.view(np.float32))
    return np.concatenate(out)


SPECIALS = np.array([0.0, -0.0, 1e-30, -1e-30, 1e-8, -1e-8, 1e6, -1e6, 3e9, -3e9, 0.5, -0.5, 1.0, -1.0],
                    dtype=np.float32)


def affine_channel_input(rng, scale, zp, qmin, qmax, L):
    """1-D f32 vector of length L for one channel: ties +- ulps first, then specials, then random."""
    ks = np.arange(qmin - 2, qmax + 2, dtype=np.float64)
    ties = ((ks + 0.5 - zp) * np.float64(scale)).astype(np.float32)
    # also the reciprocal-side ties: x such that x * (1/s) is a tie
    inv = np.float32(1.0) / np.float32(scale)
    ties2 = ((ks + 0.5 - zp) / np.float64(inv)).astype(np.float32)
    dense = np.concatenate([ulp_neighbourhood(ties), ulp_neighbourhood(ties2, 1), SPECIALS])
    if dense.size > L // 2:
        dense = rng.choice(dense, size=L // 2, replace=False)
    span = (qmax - qmin + 1) * float(scale)
    lo = (qmin - zp) * float(scale)
    n_rand = L - dense.size
    r1 = rng.uniform(lo - 0.2 * span, lo + 1.2 * span, size=n_rand // 2)
    r2 = rng.normal(0.0, 0.35 * span, size=n_rand - n_rand // 2)
    v = np.concatenate([dense, r1.astype(np.float32), r2.astype(np.float32)]).astype(np.float32)
    rng.shuffle(v)
    return v


def build_tensor(per_channel_vectors, shape, channel_axis):
    """[C, L] -> tensor of `shape` whose `channel_axis` indexes C."""
    C = shape[channel_axis]
    rest = [s for i, s in enumerate(shape) if i != channel_axis]
    a = np.asarray(per_channel_vectors, dtype=np.float32).reshape([C] + rest)
    return np.ascontiguousarray(np.moveaxis(a, 0, channel_axis))


def all_finite_half_patterns(dtype):
    bits = np.arange(0, 1 << 16, dtype=np.uint16)
    t = torch.from_numpy(bits.view(np.int16)).view(TORCH_DT[dtype])
    keep = torch.isfinite(t.float())
    return t[keep]


def add_case(name, cls_name, args, x, extra_params=None, lut_info=None, x_gen=None):
    """`x_gen`: name of the generator in tests/golden_util.py that reproduces `x` exactly (e.g. "all_finite_half_patterns");
    the input is then not stored, only what the reference computed from it."""
    cls = getattr(Q, cls_name)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        q = cls(**args)
    x_in = x.clone()
    y = q(x_in)
    case = {"name": name, "cls": cls_name, "args": args, "shape": list(x.shape),
            "x_dtype": str(x.dtype).replace("torch.", ""), "y_dtype": str(y.dtype).replace("torch.", ""),
            "params": {}}
    if x_gen is None:
        arrays[f"{name}/x"] = store(x)
    else:
        case["x_gen"] = x_gen
    arrays[f"{name}/y"] = store(y)
    # constructor-derived parameters (what the host side of the replacement must reproduce bit-for-bit)
    for attr in ("scales", "zero_points", "min_range", "max_range", "scale", "zero_point",
                 "adjusted_min_range_np", "adjusted_max_range_np", "threshold_np",
                 "min_quantized_domain", "max_quantized_domain"):
        if hasattr(q, attr):
            v = getattr(q, attr)
            if isinstance(v, torch.Tensor):
                arrays[f"{name}/p/{attr}"] = store(v)
                case["params"][attr] = {"kind": "tensor", "dtype": str(v.dtype).replace("torch.", "")}
            elif isinstance(v, np.ndarray) or isinstance(v, np.generic):
                arrays[f"{name}/p/{attr}"] = np.asarray(v)
                case["params"][attr] = {"kind": "ndarray", "dtype": str(np.asarray(v).dtype)}
            else:
                case["params"][attr] = {"kind": type(v).__name__, "value": v,
                                        "hex": float(v).hex() if isinstance(v, float) else None}
    if lut_info is not None:
        # LUT assignment re-derived with the reference's own helper, exactly as its tests do
        # (tests/pytorch_tests/quantizers_tests/test_weights_lut_inferable_quantizer.py:77-87)
        thr = lut_info["threshold"]
        t = int_quantization_with_threshold(x.clone(), n_bits=lut_info["bw"], signed=lut_info["signed"],
                                            threshold=thr, eps=lut_info["eps"]).unsqueeze(-1)
        lutv = torch.tensor(args["lut_values"], dtype=torch.float32)
        idx = torch.argmin(torch.abs(t - lutv.reshape([1] * (t.dim() - 1) + [-1])), dim=-1)
        arrays[f"{name}/idx"] = idx.numpy().astype(np.int32)
        case["has_idx"] = True
    manifest["cases"].append(case)
    return q


def lut_channel_input(rng, lut, thr, bw, signed, L, eps=1e-8):
    """1-D f32 vector: x whose normalised value sits on / around every centroid mid-point and the clip bounds."""
    lutv = np.unique(np.asarray(lut, dtype=np.float64))
    mult = 2.0 ** (bw - int(signed))
    mids = (lutv[:-1] + lutv[1:]) / 2.0
    lo, hi = (-2.0 ** (bw - 1), 2.0 ** (bw - 1) - 1) if signed else (0.0, 2.0 ** bw - 1)
    pts = np.concatenate([mids, lutv, [lo, hi, lo - 1, hi + 1, 0.0]])
    d = np.float64(np.float32(thr) + np.float32(eps))
    xs = (pts / mult * d).astype(np.float32)
    dense = np.concatenate([ulp_neighbourhood(xs), SPECIALS[:8]])
    if dense.size > L // 2:
        dense = rng.choice(dense, size=L // 2, replace=False)
    n_rand = L - dense.size
    r = rng.normal(0, 0.5 * thr, size=n_rand).astype(np.float32)
    if not signed:
        r = np.abs(r)
    v = np.concatenate([dense, r]).astype(np.float32)
    rng.shuffle(v)
    return v


MAX_ARCHIVE_BYTES = 900_000     # keeps every fixture file below 1 MB


def save(stem):
    """arrays -> stem.npz, stem_2.npz, ... (a new archive whenever the compressed size would pass MAX_ARCHIVE_BYTES; the
    manifest lists them under "archives"), manifest -> stem.json."""
    parts, part, size = [], {}, 0
    for key, a in arrays.items():
        n = len(zlib.compress(np.ascontiguousarray(a).tobytes())) + 256       # + npy header and zip entry
        if part and size + n > MAX_ARCHIVE_BYTES:
            parts.append(part)
            part, size = {}, 0
        part[key] = a
        size += n
    parts.append(part)
    manifest["archives"] = [stem + ".npz"] + [f"{stem}_{k}.npz" for k in range(2, len(parts) + 1)]
    for name, part in zip(manifest["archives"], parts):
        np.savez_compressed(os.path.join(HERE, name), **part)
    with open(os.path.join(HERE, stem + ".json"), "w") as f:
        json.dump(manifest, f, indent=1)
    tot = sum(a.nbytes for a in arrays.values())
    print(f"{len(manifest['cases'])} cases, {len(arrays)} arrays, {tot / 1e6:.1f} MB raw ->",
          [os.path.getsize(os.path.join(HERE, name)) / 1e6 for name in manifest["archives"]], "MB")
