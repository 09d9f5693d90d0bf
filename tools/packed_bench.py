#!/usr/bin/env python
"""Packed weights (mct_quantizers_b200.pytorch.packed_weights) on one GPU: resident memory, per-forward weight cost and
whole-model forward latency, in one run.

    python tools/packed_bench.py [--json out.json] [--batches 1,32,256] [--reps 50]

  memory     torch.cuda.memory_allocated before / after packing: C1 ResNet-18 and C2 MobileNetV2 (8-bit per-channel
             symmetric weights, wrapped as in tools/model_forward_bench.py), C3 Llama-7B's 96 MLP matrices (32 layers x
             gate / up 11008x4096 and down 4096x11008) as 4-bit LUT (K = 16) weights in f32 and bf16; peak memory of one
             packed forward pass
  weights    per-forward weight cost, CUDA events: per-wrapper unpack (one launch) against per-wrapper fake-quant (the float
             path), and the whole-model unpack launch against WeightPlan's fake-quant launches; algorithmic GB/s counted as
             code bytes read + output bytes written (unpack) and input + output bytes (fake-quant)
  forward    MobileNetV2 / ResNet-18 forward latency (CUDA events, median) at each batch for float wrappers, packed, and
             packed under ModelWeightPlan; logits compared bit for bit with the float model's

The card's name and power limit are part of the output.  The Llama matrices are 96 x 45 M elements (17.3 GB in f32): far
larger than L2, so every timed pass streams from HBM.
"""
import argparse
import copy
import importlib.util
import json
import os
import subprocess
import sys
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mct_quantizers_b200 as mctq  # noqa: E402
from mct_quantizers_b200.pytorch import quantizers as Q  # noqa: E402
from mct_quantizers_b200.pytorch.packed_weights import pack_model_weights  # noqa: E402

MB = 1 << 20


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        out = f"nvidia-smi unavailable ({e})"
    return out


def events_ms(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def tv_model(name):
    import torchvision
    spec = importlib.util.spec_from_file_location("mfb", os.path.join(ROOT, "tools", "model_forward_bench.py"))
    mfb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mfb)
    torch.manual_seed(0)
    return mfb.quantize_model(getattr(torchvision.models, name)(weights=None).eval(), mctq, Q).cuda()


def lut_q(C):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        lut = [float(v) for v in range(-128, 128, 16)]                        # 16 centroids on an 8-bit grid
        thr = [0.02 + 0.0001 * (c % 97) for c in range(C)]
        return Q.WeightsLUTSymmetricInferableQuantizer(4, lut, thr, True, 0, 2, 8)


def llama(dtype):
    torch.manual_seed(0)
    mats = []
    for _ in range(32):
        for out_f, in_f in ((11008, 4096), (11008, 4096), (4096, 11008)):
            lin = torch.nn.Linear(in_f, out_f, bias=False, device="cuda", dtype=dtype)
            torch.nn.init.normal_(lin.weight, std=0.02)
            mats.append(mctq.PytorchQuantizationWrapper(lin, {"weight": lut_q(out_f)}))
    return torch.nn.ModuleList(mats)


def warm(model):
    """Run every weight quantizer once (its prepared parameter tables exist from then on, packed or not) and drop the result."""
    for mod in model.modules():
        if isinstance(mod, mctq.PytorchQuantizationWrapper):
            mod.get_quantized_weights()
    torch.cuda.synchronize()


def memory_rows(out):
    for name in ("resnet18", "mobilenet_v2"):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        m = tv_model(name)
        warm(m)
        before = torch.cuda.memory_allocated() - base
        pack_model_weights(m)
        torch.cuda.synchronize()
        after = torch.cuda.memory_allocated() - base
        x = torch.randn(32, 3, 224, 224, device="cuda")
        with torch.no_grad():
            m(x)
            torch.cuda.synchronize()
            resident = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            m(x)
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - resident
        out.append(dict(model=name, weights="8-bit per-channel symmetric", dtype="float32", before_MB=round(before / MB, 2),
                        after_MB=round(after / MB, 2), ratio=round(after / before, 4), forward_peak_above_resident_MB_batch32=round(peak / MB, 2)))
        print(out[-1], flush=True)
        del m, x
    for dtype in (torch.float32, torch.bfloat16):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        m = llama(dtype)
        warm(m)
        before = torch.cuda.memory_allocated() - base
        pack_model_weights(m)
        torch.cuda.synchronize()
        after = torch.cuda.memory_allocated() - base
        x = torch.randn(8, 4096, device="cuda")
        with torch.no_grad():
            m[0](x)
            torch.cuda.synchronize()
            resident = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            m[0](x)
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - resident
        out.append(dict(model="llama7b_96_matrices", weights="4-bit LUT K=16 per-channel", dtype=str(dtype).split(".")[-1],
                        before_MB=round(before / MB, 1), after_MB=round(after / MB, 1), ratio=round(after / before, 4),
                        forward_peak_above_resident_MB_one_wrapper=round(peak / MB, 1)))
        print(out[-1], flush=True)
        del x
        yield dtype, m
        del m


def weight_rows(out, dtype, packed, reps):
    """Per-wrapper unpack vs per-wrapper fake-quant on one 11008x4096 matrix; whole-model unpack vs WeightPlan."""
    n = 11008 * 4096
    w = torch.empty(11008, 4096, device="cuda", dtype=dtype).normal_(std=0.02)
    q = packed[0]._packed.entries[0].quantizer
    esz = torch.tensor([], dtype=dtype).element_size()
    fq_ms = events_ms(lambda: q(w), reps)
    st = packed[0]._packed
    up_ms = events_ms(lambda: st.rebuild(packed[0]), reps)
    out.append(dict(what="one 11008x4096 4-bit LUT matrix", dtype=str(dtype).split(".")[-1],
                    fake_quant_ms=round(fq_ms, 4), fake_quant_GBps=round(n * (esz + 4) / fq_ms / 1e6, 1),
                    unpack_ms=round(up_ms, 4), unpack_GBps=round(n * (0.5 + 4) / up_ms / 1e6, 1)))
    print(out[-1], flush=True)
    del w
    plan = mctq.plan_model_weights(packed)
    up_all = events_ms(plan.plan.run, max(5, reps // 5))
    unpack = plan.plan._unpack_plans[0][1]
    out.append(dict(what="all 96 matrices, one UnpackPlan", dtype=str(dtype).split(".")[-1], launches=unpack.n_launches,
                    unpack_ms=round(up_all, 3), unpack_GBps=round(96 * n * 4.5 / up_all / 1e6, 1)))
    print(out[-1], flush=True)
    del plan
    torch.cuda.empty_cache()


def fq_plan_row(out, dtype, reps):
    """WeightPlan's fake-quant launches over the float Llama matrices (the path packing replaces)."""
    m = llama(dtype)
    plan = mctq.plan_model_weights(m)
    n = 11008 * 4096
    esz = torch.tensor([], dtype=dtype).element_size()
    ms = events_ms(plan.plan.run, max(5, reps // 5))
    out.append(dict(what="all 96 matrices, WeightPlan fake-quant", dtype=str(dtype).split(".")[-1],
                    fake_quant_ms=round(ms, 3), fake_quant_GBps=round(96 * n * (esz + 4) / ms / 1e6, 1)))
    print(out[-1], flush=True)
    del plan, m
    torch.cuda.empty_cache()


def forward_rows(out, batches, reps):
    for name in ("mobilenet_v2", "resnet18"):
        fl = tv_model(name)
        pk = copy.deepcopy(fl)
        pack_model_weights(pk)
        pk_plan = copy.deepcopy(pk)
        plan = mctq.plan_model_weights(pk_plan).enable()
        for b in batches:
            x = torch.randn(b, 3, 224, 224, device="cuda")
            with torch.no_grad():
                want = fl(x)
                row = dict(model=name, batch=b)
                for arm, m in (("float", fl), ("packed", pk), ("packed+plan", pk_plan)):
                    row[arm + "_ms"] = round(events_ms(lambda: m(x), reps), 4)
                    row[arm + "_bit_equal"] = bool(torch.equal(m(x), want))
            out.append(row)
            print(row, flush=True)
        plan.disable()
        del fl, pk, pk_plan
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json")
    ap.add_argument("--batches", default="1,32,256")
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("packed_bench needs a CUDA device")
    res = dict(card=card(), torch=torch.__version__, memory=[], weights=[], forward=[])
    print(res["card"], flush=True)
    for dtype, packed in memory_rows(res["memory"]):
        weight_rows(res["weights"], dtype, packed, a.reps)
        del packed
        torch.cuda.empty_cache()
        fq_plan_row(res["weights"], dtype, a.reps)
    forward_rows(res["forward"], [int(b) for b in a.batches.split(",")], a.reps)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
