#!/usr/bin/env python
"""Kernel micro-benchmark (GPU box): achieved algorithmic GB/s of each kernel family through the raw C ABI.
CUDA events on the launch stream, buffers rotated so that nothing is L2-resident, median of reps.

    python tools/kbench.py [--mb 1024] [--reps 20] [--what affine,lut,codes]
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mct_quantizers_b200 import _native  # noqa: E402
from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table  # noqa: E402

DT = {"f32": (torch.float32, 0, 4), "bf16": (torch.bfloat16, 1, 2), "f16": (torch.float16, 2, 2)}


def vp(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def timeit(fn, reps, nbuf):
    st = torch.cuda.current_stream()
    for i in range(3):
        fn(i % nbuf)
    torch.cuda.synchronize()
    ts = []
    for i in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn(i % nbuf)
        b.record(st)
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    # the same launch with the queue kept full: 4 launches between two events (what a model's back-to-back calls see; a
    # lone launch pays its own ramp and drain, 2-4 % at 150 us)
    qs = []
    for i in range(max(reps // 4, 3)):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for k in range(4):
            fn((i * 4 + k) % nbuf)
        b.record(st)
        b.synchronize()
        qs.append(a.elapsed_time(b) / 4)
    qs.sort()
    timeit.queued = qs[len(qs) // 2]
    return ts[len(ts) // 2], ts[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mb", type=float, default=1024.0, help="input megabytes per launch")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--what", default="affine,channel,fused,codes,lut,copy")
    ap.add_argument("--dtypes", default="f32,bf16")
    ap.add_argument("--json", default=None)
    ap.add_argument("--tune", default="", help="comma separated key=value pairs for mctq_set_tuning (keys 3, 9)")
    args = ap.parse_args()
    lib = _native.load()
    for kv in filter(None, args.tune.split(",")):
        k, v = kv.split("=")
        assert lib.mctq_set_tuning(int(k), int(v)) >= 0
    dev = torch.device("cuda:0")
    stream = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
    peak = 6457.7
    try:
        peak = json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    rows = []
    what = args.what.split(",")
    nbuf = 3

    def report(name, dt, algo_bytes, med, best):
        gbs = algo_bytes / med / 1e6
        q_ms = getattr(timeit, "queued", med)
        gq = algo_bytes / q_ms / 1e6
        rows.append({"kernel": name, "dtype": dt, "mb_in": args.mb, "median_ms": round(med, 4), "best_ms": round(best, 4),
                     "GBs": round(gbs, 1), "frac_of_copy_peak": round(gbs / peak, 4), "pct_of_8TBs": round(gbs / 80.0, 2),
                     "queued_ms": round(q_ms, 4), "GBs_queued": round(gq, 1), "pct_of_8TBs_queued": round(gq / 80.0, 2)})
        print(f"{name:46s} {dt:5s} {args.mb:8.0f} MB  lone launch {med:8.4f} ms {gbs:8.1f} GB/s {gbs / 80:6.2f}% of 8TB/s | "
              f"4 queued {gq:8.1f} GB/s {gq / peak * 100:6.2f}% of copy peak {gq / 80:6.2f}% of 8TB/s", flush=True)

    for dt in args.dtypes.split(","):
        tdt, tag, es = DT[dt]
        n = int(args.mb * 1e6 / es) // 4096 * 4096
        xs = [torch.empty(n, dtype=tdt, device=dev).uniform_(-50, 50) for _ in range(nbuf)]
        ys = [torch.empty(n, dtype=tdt, device=dev) for _ in range(nbuf)]
        if "copy" in what:
            med, best = timeit(lambda i: ys[i].copy_(xs[i]), args.reps, nbuf)
            report("torch copy_ (reference point)", dt, 2 * n * es, med, best)
        if "affine" in what:
            med, best = timeit(lambda i: lib.mctq_fq_affine_scalar(vp(xs[i]), vp(ys[i]), None, n, tag, 0.03125, 0, -128, 127, 0, stream()),
                               args.reps, nbuf)
            report("affine per-tensor scalar", dt, 2 * n * es, med, best)
            med, best = timeit(lambda i: lib.mctq_fq_affine_scalar(vp(xs[i]), vp(ys[i]), None, n, tag, 0.0129, 77, 0, 255, 0, stream()),
                               args.reps, nbuf)
            report("affine per-tensor uniform zp", dt, 2 * n * es, med, best)
        if "channel" in what:
            for (C, inner, label) in ((4096, 11008, "rows 11008"), (11008, 4096, "rows 4096"), (512, 4608, "conv 512x512x3x3"),
                                      (960, 9, "depthwise inner 9"), (1024, 64, "rows 64"), (256, 16, "convT 4x4 inner 16"),
                                      (768, 1, "channel-last C=768"), (3, 1, "channel-last C=3")):
                sc = torch.rand(C, device=dev) * 0.05 + 0.01
                zp = torch.zeros(C, dtype=torch.int32, device=dev)
                med, best = timeit(lambda i: lib.mctq_fq_affine(vp(xs[i]), vp(ys[i]), None, n, tag, vp(sc), vp(zp), C, inner, 0, -128, 127, 0, stream()),
                                   args.reps, nbuf)
                report(f"affine per-channel {label}", dt, 2 * n * es, med, best)
                nb = lib.mctq_affine_prepared_bytes(C)
                blob = torch.empty(nb, dtype=torch.uint8, device=dev)
                assert lib.mctq_affine_prepare(vp(sc), vp(zp), C, vp(blob), nb, stream()) == 0
                torch.cuda.synchronize()
                fn = lambda i: lib.mctq_fq_affine_prepared(vp(xs[i]), vp(ys[i]), None, n, tag, vp(blob), C, inner, 0, -128, 127, 0, stream())
                assert fn(0) == 0
                med, best = timeit(fn, args.reps, nbuf)
                report(f"affine-prepared per-channel {label}", dt, 2 * n * es, med, best)
        if "fused" in what:
            for pre, label, streams in ((1, "relu", 2), (2, "relu6", 2), (3, "add", 3), (4, "add+relu", 3)):
                fn = lambda i: lib.mctq_fq_affine_scalar_pre(vp(xs[i]), vp(xs[(i + 1) % nbuf]), vp(ys[i]), n, tag, pre, 0.0129, 77, 0, 255, stream())
                assert fn(0) == 0
                med, best = timeit(fn, args.reps, nbuf)
                report(f"fused {label} -> affine per-tensor", dt, streams * n * es, med, best)
        if "codes" in what:
            cs = [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(nbuf)]
            med, best = timeit(lambda i: lib.mctq_fq_affine_scalar(vp(xs[i]), vp(ys[i]), vp(cs[i]), n, tag, 0.03125, 0, -128, 127, 1, stream()), args.reps, nbuf)
            report("affine per-tensor + int8 codes", dt, n * (2 * es + 1), med, best)
            med, best = timeit(lambda i: lib.mctq_fq_affine_scalar(vp(xs[i]), None, vp(cs[i]), n, tag, 0.03125, 0, -128, 127, 1, stream()), args.reps, nbuf)
            report("affine per-tensor int8 codes only", dt, n * (es + 1), med, best)
            med, best = timeit(lambda i: lib.mctq_fq_affine_scalar(vp(xs[i]), vp(ys[i]), vp(cs[i]), n, tag, 0.5, 0, -8, 7, 2, stream()), args.reps, nbuf)
            report("affine per-tensor + int4 codes", dt, n * (2 * es + 0.5), med, best)
            # consumer side of the code wire format: codes -> f32 values (5 / 4.5 algorithmic bytes per element)
            yf32 = [torch.empty(n, dtype=torch.float32, device=dev) for _ in range(nbuf)]
            for (C, inner, label) in ((1, 1, "per-tensor"), (4096, n // 4096 // 8 * 8 or 8, "per-channel long rows"), (960, 9, "per-channel inner 9")):
                sc = torch.rand(C, device=dev) * 0.05 + 0.01
                zp = torch.zeros(C, dtype=torch.int32, device=dev)
                for mode, cb, lab in ((1, 1.0, "int8"), (2, 0.5, "int4")):
                    fn = lambda i: lib.mctq_dequant_affine(vp(cs[i]), mode, 1, vp(yf32[i]), n, vp(sc), vp(zp), C, inner, 0, stream())
                    assert fn(0) == 0
                    med, best = timeit(fn, args.reps, nbuf)
                    report(f"dequant {lab} codes -> f32 {label}", dt, n * (cb + 4), med, best)
            del cs, yf32
        if "lut" in what:
            del ys
            yf = [torch.empty(n, dtype=torch.float32, device=dev) for _ in range(nbuf)]
            rng = np.random.default_rng(0)
            lut = np.array(sorted(rng.choice(np.arange(-128, 128), size=16, replace=False)), dtype=np.float32)
            table = lut_search_table(lut, 8, True).to(dev)
            for x in xs:
                x.normal_(0, 0.02)
            for (C, inner, label) in ((4096, 11008, "rows 11008"), (11008, 4096, "rows 4096"), (1, 1, "per-tensor")):
                thr = torch.rand(C, device=dev) * 0.05 + 0.06
                med, best = timeit(lambda i: lib.mctq_fq_lut(vp(xs[i]), vp(yf[i]), None, n, tag, vp(table), 16, vp(thr), C, inner, 0,
                                                             1e-8, 0, stream()), args.reps, nbuf)
                report(f"lut K=16 weights {label}", dt, n * (es + 4), med, best)
            med, best = timeit(lambda i: lib.mctq_fq_lut_scalar(vp(xs[i]), vp(yf[i]), None, n, tag, vp(table), 16, 0.125, 0.125, int(es == 2), 0, stream()),
                               args.reps, nbuf)
            report("lut K=16 activation scalar", dt, n * (es + 4), med, best)
            # prepared path: per-channel decision tables in the x domain (built once, outside the timed region)
            table_host = lut_search_table(lut, 8, True)
            for (C, inner, label) in ((4096, 11008, "rows 11008"), (11008, 4096, "rows 4096"), (1, 1, "per-tensor"), (65536, 64, "rows 64")):
                thr = torch.rand(C, device=dev) * 0.05 + 0.06
                nb = lib.mctq_lut_prepared_bytes(16, 8, 1, C)
                blob = torch.empty(nb, dtype=torch.uint8, device=dev)
                rc = lib.mctq_lut_prepare(vp(table_host), 16, vp(thr), C, 1e-8, 0, 1.0, 1.0, 0, vp(blob), nb, stream())
                assert rc == 0, rc
                torch.cuda.synchronize()
                for mode, lab in ((0, ""), (2, " + int4 idx")):
                    ib = torch.empty(n // 2 + 8, dtype=torch.uint8, device=dev) if mode else None
                    fn = lambda i: lib.mctq_fq_lut_prepared(vp(xs[i]), vp(yf[i]), vp(ib), n, tag, vp(blob), 16, 8, 1, C, inner, 0, mode, stream())
                    assert fn(0) == 0
                    med, best = timeit(fn, args.reps, nbuf)
                    report(f"lut-prepared K=16 weights {label}{lab}", dt, n * (es + 4 + (0.5 if mode else 0)), med, best)
            del yf
        del xs
        torch.cuda.empty_cache()
    if "gaps" in what:
        # launch-gap experiment: 64 back-to-back launches of a small (64 MB) and a medium (256 MB) tensor, PDL on / off
        for mb in (16, 64, 256):
            n = int(mb * 1e6 / 4) // 4096 * 4096
            xs = [torch.empty(n, device=dev).uniform_(-50, 50) for _ in range(8)]
            ys = [torch.empty(n, device=dev) for _ in range(8)]
            for pdl in (0, 1):
                lib.mctq_set_tuning(3, pdl)
                def burst(_):
                    for k in range(64):
                        lib.mctq_fq_affine_scalar(vp(xs[k % 8]), vp(ys[k % 8]), None, n, 0, 0.0129, 77, 0, 255, 0, stream())
                med, best = timeit(burst, 10, 1)
                gbs = 64 * 8 * n / med / 1e6
                print(f"64 back-to-back launches of {mb} MB f32, PDL={pdl}: {med / 64 * 1e3:8.2f} us per launch  {gbs:8.1f} GB/s", flush=True)
                rows.append({"kernel": f"burst64 {mb}MB pdl={pdl}", "us_per_launch": round(med / 64 * 1e3, 2), "GBs": round(gbs, 1)})
            lib.mctq_set_tuning(3, 1)
            del xs, ys
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"peak_gbs": peak, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
