#!/usr/bin/env python
"""Batched packed linear (mctq_packed_linear_batched, tensor cores) against the exact packed path, resident float weights and
the CUDA-core fused kernel, on one GPU.

    python tools/packed_batched_bench.py [--json out.json] [--rows 8,12,16,32,64,128,256] [--reps 3]

Workload and formats of tools/packed_linear_bench.py: Llama-7B's 96 MLP matrices (2.1 GB of int4 codes, far above the
126 MB L2, so every sweep streams from HBM) as 4-bit LUT f32, int4 symmetric bf16 and int8 symmetric bf16, plus int4 / int8
symmetric f32 (the f32 affine kernels, which share FUSED_BATCHED_MAX_ROWS with the LUT).  Arms, timed
with CUDA events over a sweep of all 96 matrices and alternated inside every repetition (median over --reps, and spread):
    batched   ops.PackedLinear.batched: the tensor-core kernel
    rebuild   today's exact packed path: ops.UnpackPlan (fresh output) + F.linear
    float     F.linear on resident rebuilt weights in the storage dtype
    fused     ops.PackedLinear: the CUDA-core kernel of the fused mode
Also per row: the largest relative difference of the batched result to the rebuild path on the first matrix (max |diff| /
max |rebuild|), and the batched arm's share of its binding bound max(code bytes / 7.7 TB/s, MMA FLOPs / 2.25 PFLOP/s), the
FLOPs counting the three bf16 passes of an f32 x.  Data-sheet rates of one B200 at 1000 W; the card's name, power limit and
SM clock are printed in the same run.
"""
import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from mct_quantizers_b200 import _native, ops  # noqa: E402
from mct_quantizers_b200.pytorch.packed_weights import FUSED_LINEAR_MAX_ROWS  # noqa: E402
from packed_linear_bench import FORMATS, HBM_TBPS, SHAPES, card, make_items, sweep_events  # noqa: E402

MMA_TFLOPS = 2250.0
FORMATS = FORMATS + [("int4_sym_f32", _native.PACK_AFFINE_I4, torch.float32),
                     ("int8_sym_f32", _native.PACK_AFFINE_I8, torch.float32)]


def bench_format(name, kind, dtype, rows, reps, out):
    items = make_items(kind, dtype)
    lins = [ops.PackedLinear(c, k, s, dt, sh[0], sh[1], sc, z, q) for c, k, s, dt, sh, _, _, _, sc, z, q in items]
    plans = [ops.UnpackPlan([it], fresh=True) for it in items]
    float_w = ops.UnpackPlan(items).run()
    code_bytes = sum(it[0].numel() for it in items)
    terms = 3 if dtype == torch.float32 else 1
    for M in rows:
        xs = {k: torch.randn(M, k, device="cuda").to(dtype) for k in (4096, 11008)}
        arms = {
            "batched": lambda: [lin.batched(xs[lin.in_features]) for lin in lins],
            "rebuild": lambda: [F.linear(xs[p._out_specs[0][0][1]], p.run()[0]) for p in plans],
            "float": lambda: [F.linear(xs[w.shape[1]], w) for w in float_w],
            "fused": lambda: [lin(xs[lin.in_features]) for lin in lins],
        }
        times = {a: [] for a in arms}
        for _ in range(reps):
            for a, fn in arms.items():
                times[a].append(sweep_events(fn))
        row = dict(format=name, M=M)
        for a in arms:
            row[a + "_ms"] = round(statistics.median(times[a]), 4)
            row[a + "_spread_ms"] = round(max(times[a]) - min(times[a]), 4)
        flops = sum(2.0 * M * o * i for o, i in SHAPES) * terms
        bound_bytes_ms, bound_flops_ms = code_bytes / HBM_TBPS / 1e9, flops / MMA_TFLOPS / 1e9
        row["bound"] = "bytes" if bound_bytes_ms >= bound_flops_ms else "mma"
        row["batched_share_of_bound"] = round(max(bound_bytes_ms, bound_flops_ms) / row["batched_ms"], 3)
        row["batched_vs_rebuild"] = round(row["rebuild_ms"] / row["batched_ms"], 2)
        row["batched_vs_float"] = round(row["float_ms"] / row["batched_ms"], 2)
        row["batched_vs_fused"] = round(row["fused_ms"] / row["batched_ms"], 2)
        y_b, y_r = lins[0].batched(xs[4096]).float(), F.linear(xs[4096], plans[0].run()[0]).float()
        row["max_rel_diff_vs_rebuild"] = float(((y_b - y_r).abs().max() / y_r.abs().max().clamp_min(1e-30)).item())
        out.append(row)
        print(row, flush=True)
    del lins, plans, float_w, items
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json")
    ap.add_argument("--rows", default="8,12,16,32,64,128,256")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--formats", default=",".join(f[0] for f in FORMATS))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("packed_batched_bench needs a CUDA device")
    res = dict(card=card(), torch=torch.__version__, rows=[])
    print(res["card"], flush=True)
    rows = [int(r) for r in a.rows.split(",")]
    with torch.no_grad():
        for name, kind, dtype in FORMATS:
            if name in a.formats.split(","):
                bench_format(name, kind, dtype, rows, a.reps, res["rows"])
    # crossover: the largest M up to which batched beats rebuild at every measured M above the fused kernel's row limit
    # (the rows batched mode serves), in every format of a dtype; 0 when it loses at the first of them
    for dt, tdt in (("f32", torch.float32), ("bf16", torch.bfloat16)):
        fr = [r for r in res["rows"] if r["format"].endswith(dt)]
        served = [M for M in rows if M > FUSED_LINEAR_MAX_ROWS[tdt]]
        ok = [M for M in served if all(r["batched_ms"] < r["rebuild_ms"] for r in fr if r["M"] == M)]
        res["crossover_" + dt] = max((M for M in ok if all(m in ok for m in served if m <= M)), default=0)
    print({k: v for k, v in res.items() if k.startswith("crossover")}, flush=True)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
