#!/usr/bin/env python
"""Fused packed linear (mctq_packed_linear) against the exact packed path and against resident float weights, on one GPU.

    python tools/packed_linear_bench.py [--json out.json] [--rows 1,2,4,8,16,32,64] [--reps 3]

Workload: Llama-7B's MLP matrices, 32 x (gate 11008x4096, up 11008x4096, down 4096x11008), in three formats
    lut4_f32        4-bit LUT (K = 16) per output channel, f32 weights / activations
    int4_sym_bf16   int4 symmetric per output channel, bf16
    int8_sym_bf16   int8 symmetric per output channel, bf16
Arms, each timed with CUDA events over a sweep of all 96 matrices (2.1 GB of int4 codes, far above the 126 MB L2, so every
sweep streams from HBM):
    fused     ops.PackedLinear: y = x @ W^T straight from the codes
    rebuild   today's exact packed path: ops.UnpackPlan (fresh output) + F.linear
    float     F.linear on the already rebuilt weights, resident in the storage dtype (the best a float model can do)
The arms alternate inside every repetition; the table reports the median over --reps repetitions and the spread.  Bytes are
algorithmic: codes + parameters + M*in*x + M*out*y (fused, float: the float weight instead of the codes), TB/s over 7.7 TB/s
(data sheet) gives the share of the memory bound.  Also reported: the M = 1 sweep as 96 eager fused-mode wrapper forwards
(host time included) and as one CUDA-graph replay, next to the same wrappers on the exact packed path.
The card's name, power limit and SM clock are printed in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import warnings

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mct_quantizers_b200 as mctq  # noqa: E402
from mct_quantizers_b200 import _native, ops  # noqa: E402
from mct_quantizers_b200.pytorch import quantizers as Q  # noqa: E402
from mct_quantizers_b200.pytorch.packed_weights import pack_model_weights  # noqa: E402

SHAPES = [(11008, 4096), (11008, 4096), (4096, 11008)] * 32
HBM_TBPS = 7.7
FORMATS = [("lut4_f32", _native.PACK_LUT_I4, torch.float32), ("int4_sym_bf16", _native.PACK_AFFINE_I4, torch.bfloat16),
           ("int8_sym_bf16", _native.PACK_AFFINE_I8, torch.bfloat16)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def make_items(kind, dtype, seed=0):
    """Random codes and per-channel parameters for the 96 matrices: UnpackPlan items (codes, kind, signed, dtype, shape,
    stride, C, inner, scale, zp, quotients)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    lut = kind in _native.PACK_LUT_KINDS
    quot = ops.lut_quotients(torch.arange(-128, 128, 16, dtype=torch.float32), 8, True).cuda() if lut else None
    items = []
    for out_f, in_f in SHAPES:
        n = out_f * in_f
        codes = torch.randint(0, 256, (_native.packed_code_bytes(kind, n),), dtype=torch.uint8, device="cuda", generator=g)
        if kind == _native.PACK_AFFINE_I4:                  # symmetric int4: codes in [-8, 7], both nibbles
            codes = codes & 0x77
        scale = torch.rand(out_f, device="cuda", generator=g) * 0.01 + 0.005
        zp = None if lut else torch.zeros(out_f, dtype=torch.int32, device="cuda")
        items.append((codes, kind, not lut, dtype, (out_f, in_f), None, out_f, in_f, scale, zp, quot))
    return items


def sweep_events(fn, n=3):
    """Median of n timed sweeps (ms), after one warm-up sweep."""
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def bench_format(name, kind, dtype, rows, reps, out):
    items = make_items(kind, dtype)
    lins = [ops.PackedLinear(c, k, s, dt, sh[0], sh[1], sc, z, q) for c, k, s, dt, sh, _, _, _, sc, z, q in items]
    plans = [ops.UnpackPlan([it], fresh=True) for it in items]
    float_w = ops.UnpackPlan(items).run()                   # resident rebuilt weights in the storage dtype
    esz = torch.tensor([], dtype=dtype).element_size()
    code_bytes = sum(it[0].numel() for it in items)
    param_bytes = sum(it[8].numel() * 4 + (it[9].numel() * 4 if it[9] is not None else 0) for it in items)
    w_bytes = sum(w.numel() * w.element_size() for w in float_w)
    for M in rows:
        xs = {k: torch.randn(M, k, device="cuda").to(dtype) for k in (4096, 11008)}
        arms = {
            "fused": lambda: [lin(xs[lin.in_features]) for lin in lins],
            "rebuild": lambda: [F.linear(xs[p._out_specs[0][0][1]], p.run()[0]) for p in plans],
            "float": lambda: [F.linear(xs[w.shape[1]], w) for w in float_w],
        }
        times = {a: [] for a in arms}
        for _ in range(reps):
            for a, fn in arms.items():
                times[a].append(sweep_events(fn))
        act = sum(M * i * esz + M * o * esz for o, i in SHAPES)
        row = dict(format=name, M=M)
        for a in arms:
            ms = statistics.median(times[a])
            nbytes = (w_bytes if a == "float" else code_bytes + param_bytes) + act
            row[a + "_ms"] = round(ms, 4)
            row[a + "_spread_ms"] = round(max(times[a]) - min(times[a]), 4)
            row[a + "_TBps"] = round(nbytes / ms / 1e9, 3)
            row[a + "_share_of_7.7TBps"] = round(nbytes / ms / 1e9 / HBM_TBPS, 3)
        row["fused_vs_rebuild"] = round(row["rebuild_ms"] / row["fused_ms"], 2)
        row["fused_vs_float"] = round(row["float_ms"] / row["fused_ms"], 2)
        # the fused result against the exact path, at this size (f32 accumulation; reordered sums differ in the last bits)
        y_f, y_r = lins[0](xs[4096]).float(), F.linear(xs[4096], plans[0].run()[0]).float()
        row["max_rel_diff_vs_rebuild"] = float(((y_f - y_r).abs().max() / y_r.abs().max().clamp_min(1e-30)).item())
        out.append(row)
        print(row, flush=True)
    del lins, plans, float_w, items
    torch.cuda.empty_cache()


def lut_q(C):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return Q.WeightsLUTSymmetricInferableQuantizer(4, [float(v) for v in range(-128, 128, 16)],
                                                       [0.02 + 0.0001 * (c % 97) for c in range(C)], True, 0, 2, 8)


def wrapper_rows(out, reps):
    """96 fused-mode LUT f32 wrappers at M = 1: eager forwards (host clock around the sweep + synchronize) and a CUDA-graph
    replay, against the same wrappers on the exact packed path."""
    torch.manual_seed(0)
    mats = []
    for out_f, in_f in SHAPES:
        lin = torch.nn.Linear(in_f, out_f, bias=False, device="cuda")
        torch.nn.init.normal_(lin.weight, std=0.02)
        w = mctq.PytorchQuantizationWrapper(lin, {"weight": lut_q(out_f)})
        pack_model_weights(w, fused_linear=True)
        mats.append(w)
    ops.clear_lut_caches()
    xs = {k: torch.randn(1, k, device="cuda") for k in (4096, 11008)}

    def sweep():
        return [m(xs[m.layer.in_features]) for m in mats]

    def eager_ms():
        sweep()
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            sweep()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        return statistics.median(ts)

    with torch.no_grad():
        res = {}
        for mode in (True, False):
            for m in mats:
                m._packed.fused = mode
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                sweep()
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                sweep()
            key = "fused" if mode else "exact_packed"
            e, gr = [], []
            for _ in range(reps):
                e.append(eager_ms())
                gr.append(sweep_events(graph.replay))
            res[key + "_eager_ms"] = round(statistics.median(e), 4)
            res[key + "_graph_ms"] = round(statistics.median(gr), 4)
            del graph
        row = dict(what="96 LUT f32 wrappers, M = 1, one sweep", **res)
        out.append(row)
        print(row, flush=True)
    del mats
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json")
    ap.add_argument("--rows", default="1,2,4,8,16,32,64")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--formats", default=",".join(f[0] for f in FORMATS))
    ap.add_argument("--no-wrappers", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("packed_linear_bench needs a CUDA device")
    res = dict(card=card(), torch=torch.__version__, rows=[], wrappers=[])
    print(res["card"], flush=True)
    rows = [int(r) for r in a.rows.split(",")]
    with torch.no_grad():
        for name, kind, dtype in FORMATS:
            if name in a.formats.split(","):
                bench_format(name, kind, dtype, rows, a.reps, res["rows"])
    if not a.no_wrappers:
        wrapper_rows(res["wrappers"], a.reps)
    # crossover: the largest M at which fused beats rebuild in every format of a dtype
    for dt in ("f32", "bf16"):
        fr = [r for r in res["rows"] if r["format"].endswith(dt)]
        ok = [M for M in rows if all(r["fused_ms"] < r["rebuild_ms"] for r in fr if r["M"] == M)]
        res["crossover_" + dt] = max((M for M in ok if all(m in ok for m in rows if m <= M)), default=0)
    print({k: v for k, v in res.items() if k.startswith("crossover")}, flush=True)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
