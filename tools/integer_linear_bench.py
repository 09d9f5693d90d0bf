#!/usr/bin/env python
"""Integer linear mode (mctq_quantize_rows_i8 + mctq_packed_linear_i8) against the existing packed paths, resident float
weights and cuBLAS int8, on one GPU.

    python tools/integer_linear_bench.py [--json out.json] [--rows 1,4,...] [--reps 3]

Workload: Llama-7B's linear shapes 4096 -> 11008, 11008 -> 4096 and 4096 -> 4096, int8 and int4 symmetric per-channel codes,
x in f32 and bf16.  Each shape is replicated until its codes exceed 300 MB (above the 126 MB L2, so every sweep streams the
weights from HBM).  Arms, timed with CUDA events over a sweep of all copies and alternated inside every repetition (median
over --reps):
    integer   ops.IntegerLinear: row quantizer + integer GEMM (end to end)
    igemm     the integer GEMM alone, on codes quantized once
    packed    the best existing packed path for the dtype: fused kernel up to FUSED_LINEAR_MAX_ROWS, batched kernel up to
              FUSED_BATCHED_MAX_ROWS, else rebuild (UnpackPlan) + F.linear
    float     F.linear on resident float weights of the dtype
    int_mm    torch._int_mm (cuBLAS int8) on the same int8 codes of x and W (M > 16 only; int4 codes widened to int8)
Per row also: igemm's share of its binding bound, max((code + x code + y bytes) / 7.7 TB/s, 2 M N K / 4.5 POPS) (data-sheet
rates of one B200 at 1000 W: HBM3e bandwidth and dense int8 tensor-core rate), and whether the integer arm's output equals
the exact integer reference (f64 code sums on the device, exact below 2^53) bit for bit on the first copy.  The card's name,
power limit and clocks are read in the same run, and the kernel's SASS counts (UTCIMMA, registers, local memory) are recorded.
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from mct_quantizers_b200 import _native, ops  # noqa: E402
from mct_quantizers_b200.pytorch.packed_weights import FUSED_BATCHED_MAX_ROWS, FUSED_LINEAR_MAX_ROWS  # noqa: E402
from packed_linear_bench import HBM_TBPS, card, sweep_events  # noqa: E402

INT8_POPS = 4.5
SHAPES = [(11008, 4096), (4096, 11008), (4096, 4096)]          # (out_features, in_features)
FORMATS = [("int8", _native.PACK_AFFINE_I8), ("int4", _native.PACK_AFFINE_I4)]
X_SCALE, X_ZP = 0.0213, 0                                      # a symmetric 8-bit input quantizer


def sass_counts():
    """UTCIMMA instructions and resource usage of the integer GEMM kernels in libmctq_sm100.so."""
    try:
        sass = subprocess.run(["cuobjdump", "-sass", _native.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
        res = subprocess.run(["cuobjdump", "-res-usage", _native.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}
    out = {}
    for block in sass.split("Function : ")[1:]:
        name = block.split("\n", 1)[0].strip()
        if "packed_igemm_kernel" in name:
            out.setdefault(name, {})["UTCIMMA"] = block.count("UTCIMMA")
    for line, nxt in zip(res.splitlines(), res.splitlines()[1:]):
        if "packed_igemm_kernel" in line:
            name = line.split("Function ")[-1].rstrip(":").strip()
            m = {k: int(v) for k, v in re.findall(r"(REG|STACK|LOCAL|SHARED):(\d+)", nxt)}
            out.setdefault(name, {}).update(m)
    return out


def make_weights(kind, out_f, in_f, copies, g):
    ws = []
    for _ in range(copies):
        n = out_f * in_f
        codes = torch.randint(0, 256, (_native.packed_code_bytes(kind, n),), dtype=torch.uint8, device="cuda", generator=g)
        if kind == _native.PACK_AFFINE_I4:
            codes = codes & 0x77                                # int4: both nibbles in [0, 7] (non-negative signed codes)
        else:
            codes = (codes.view(torch.int8).clamp_(-127, 127)).contiguous()
        scale = torch.rand(out_f, device="cuda", generator=g) * 0.01 + 0.005
        zp = torch.zeros(out_f, dtype=torch.int32, device="cuda")
        ws.append((codes, scale, zp))
    return ws


def reference(lin, qx, qw, bias):
    c = qx.to(torch.float64) @ qw.to(torch.float64).T
    return ((c.to(torch.int64).to(torch.float32) * lin.factor[None, :]) + (bias.float() if bias is not None else 0)
            ).to(lin.dtype)


def bench(shape, fmt, kind, dtype, rows, reps, out, g):
    out_f, in_f = shape
    code_bytes = _native.packed_code_bytes(kind, out_f * in_f)
    copies = max(1, -(-300_000_000 // code_bytes))
    ws = make_weights(kind, out_f, in_f, copies, g)
    ilins = [ops.IntegerLinear(c, kind, True, dtype, out_f, in_f, s, z, X_SCALE, X_ZP, -128, 127) for c, s, z in ws]
    plins = [ops.PackedLinear(c, kind, True, dtype, out_f, in_f, s, z, None) for c, s, z in ws]
    items = [(c, kind, True, dtype, (out_f, in_f), (in_f, 1), out_f, in_f, s, z, None) for c, s, z in ws]
    plans = [ops.UnpackPlan([it], fresh=True) for it in items]
    float_w = ops.UnpackPlan(items).run()
    wq8 = [ops.weight_code_values(c, kind, True, out_f, in_f).to(torch.int8).T.contiguous().T for c, _, _ in ws]
    esz = torch.tensor([], dtype=dtype).element_size()
    for M in rows:
        x = torch.randn(M, in_f, device="cuda", generator=g).to(dtype)
        qx, _ = ilins[0].quantize(x)
        arms = {
            "integer": lambda: [lin(x) for lin in ilins],
            "igemm": lambda: [lin.gemm(qx) for lin in ilins],
            "float": lambda: [F.linear(x, w) for w in float_w],
        }
        if M <= FUSED_LINEAR_MAX_ROWS[dtype]:
            arms["packed"] = lambda: [lin(x) for lin in plins]
        elif M <= FUSED_BATCHED_MAX_ROWS[dtype]:
            arms["packed"] = lambda: [lin.batched(x) for lin in plins]
        else:
            arms["packed"] = lambda: [F.linear(x, p.run()[0]) for p in plans]
        if M > 16:
            arms["int_mm"] = lambda: [torch._int_mm(qx, w.T) for w in wq8]
        times = {a: [] for a in arms}
        for _ in range(reps):
            for a, fn in arms.items():
                times[a].append(sweep_events(fn))
        row = dict(shape=f"{in_f}->{out_f}", format=fmt, x=str(dtype).replace("torch.", ""), M=M, copies=copies)
        for a, ts in times.items():
            row[a + "_ms"] = statistics.median(ts) / copies
            row[a + "_spread"] = (max(ts) - min(ts)) / copies
        t = row["igemm_ms"] * 1e-3
        bytes_ = code_bytes + M * in_f + M * out_f * esz
        ops_ = 2.0 * M * out_f * in_f
        t_hbm, t_ops = bytes_ / (HBM_TBPS * 1e12), ops_ / (INT8_POPS * 1e15)
        row["bound"] = "hbm" if t_hbm >= t_ops else "int8"
        row["igemm_share"] = max(t_hbm, t_ops) / t
        y = ilins[0](x)
        row["bit_exact"] = bool(torch.equal(y, reference(ilins[0], qx, wq8[0], None)))
        print(json.dumps(row), flush=True)
        out.append(row)
    del ilins, plins, plans, float_w, wq8, ws
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json")
    ap.add_argument("--txt")
    ap.add_argument("--rows", default="1,4,8,16,32,64,128,256,1024,4096")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("integer_linear_bench needs a CUDA device")
    res = dict(card=card(), torch=torch.__version__, sass=sass_counts(), rows=[])
    print(res["card"], flush=True)
    print(json.dumps(res["sass"]), flush=True)
    rows = [int(r) for r in a.rows.split(",")]
    g = torch.Generator(device="cuda").manual_seed(0)
    with torch.no_grad():
        for shape in SHAPES:
            for fmt, kind in FORMATS:
                for dtype in (torch.float32, torch.bfloat16):
                    bench(shape, fmt, kind, dtype, rows, a.reps, res["rows"], g)
    res["card_after"] = card()
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    if a.txt:
        arms = ("integer", "igemm", "packed", "float", "int_mm")
        with open(a.txt, "w") as f:
            f.write(f"{res['card']}\n(after: {res['card_after']})\n")
            f.write("per-matrix time in us (median of %d alternated sweeps); igemm share of its binding bound\n" % a.reps)
            f.write("shape        fmt  x        M     " + "".join(f"{x:>10}" for x in arms) + "   share  bound exact\n")
            for r in res["rows"]:
                f.write(f"{r['shape']:<12} {r['format']:<4} {r['x']:<8} {r['M']:<5} " +
                        "".join(f"{r[x + '_ms'] * 1e3:>10.1f}" if x + "_ms" in r else f"{'-':>10}" for x in arms) +
                        f"   {r['igemm_share'] * 100:5.1f}% {r['bound']:>5} {r['bit_exact']}\n")
            f.write("SASS: " + json.dumps(res["sass"]) + "\n")


if __name__ == "__main__":
    main()
