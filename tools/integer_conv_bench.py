#!/usr/bin/env python
"""Integer convolution mode (mctq_quantize_nhwc_i8 + mctq_packed_conv2d_i8) against the packed path and resident float weights,
per layer and per model, on one GPU.

    python tools/integer_conv_bench.py [--json out.json] [--txt out.txt] [--batches 1,32,256] [--reps 15]

Workload: the conv layers of MCT-style ResNet-18 and MobileNetV2 (tools/model_forward_bench.quantize_model: 8-bit symmetric
per-channel weights, a uniform 8-bit holder behind every ReLU / ReLU6) that pack_model_weights(integer_conv=True) switches,
at 224 x 224, batch 1 / 32 / 256, f32 and bf16.  Per distinct layer shape, each arm timed with CUDA events around one call,
with a 256 MB buffer overwritten before every call (the 126 MB L2 holds nothing of the layer), median over --reps, arms
alternated inside each repetition:
    packed    the wrapper's packed path: rebuild the weight (UnpackPlan) + F.conv2d (cuDNN; f32 runs TF32 when
              torch.backends.cudnn.allow_tf32, recorded below)
    float     F.conv2d on a resident rebuilt weight
    integer   the wrapper in integer mode end to end: NHWC quantizer + implicit GEMM (+ Sx when a weight zero point is not 0)
    gemm      mctq_packed_conv2d_i8 alone, on codes quantized once
Per row also: the GEMM's share of its binding bound, max((x code + weight code + y bytes) / 7.7 TB/s, 2 M Cout K / 4.5 POPS)
(data-sheet rates of one B200 at 1000 W: HBM3e bandwidth and dense int8 tensor-core rate; not measured figures), and whether
the integer and gemm outputs equal the exact integer reference (tests/test_integer_conv.conv_reference) bit for bit.
Whole models: forward of the packed model against the same model packed with integer_conv=True, integer_linear=True, eager
and replayed from a CUDA graph, with the number of switched convs and the largest output difference.  (The models are
randomly initialised: MobileNetV2's activations fall below its holders' first code step, so both of its outputs are 0.)
The card's name, power limit and clocks are read in the same run.
"""
import argparse
import copy
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mct_quantizers_b200 as mctq  # noqa: E402
from mct_quantizers_b200 import ops  # noqa: E402
from mct_quantizers_b200.pytorch import packed_weights as PW  # noqa: E402
from mct_quantizers_b200.pytorch import quantizers as Q  # noqa: E402
from model_forward_bench import quantize_model  # noqa: E402
from packed_linear_bench import HBM_TBPS, card  # noqa: E402
from test_integer_conv import _launch_args, conv_reference  # noqa: E402

INT8_POPS = 4.5


def models():
    import torchvision
    return {"resnet18": lambda: quantize_model(torchvision.models.resnet18(), mctq, Q),
            "mobilenet_v2": lambda: quantize_model(torchvision.models.mobilenet_v2(), mctq, Q)}


def timed(fns, reps, flush):
    """{name: median ms} of single calls, each after overwriting `flush`, the arms alternated per repetition."""
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            flush.add_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts[k].append(a.elapsed_time(b))
    return {k: statistics.median(v) for k, v in ts.items()}


def model_ms(fn, reps):
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
    return statistics.median(ts)


def graphed(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
        fn()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    return g.replay


def layer_inputs(model, names, x):
    """The input each named wrapper receives in one forward of `model`."""
    seen, hooks = {}, []
    for n in names:
        hooks.append(model.get_submodule(n).register_forward_pre_hook(lambda m, a, n=n: seen.setdefault(n, a[0])))
    model(x)
    for h in hooks:
        h.remove()
    return seen


def exact(h, w, x, y):
    """y equals the integer reference of wrapper w on input x (Q = holder h's quantizer) bit for bit."""
    e = w._packed.entries[0]
    s, z, qmin, qmax = _launch_args(h.activation_holder_quantizer)
    qx, _ = ops.quantize_nhwc_i8(x, s, z, qmin, qmax, False)
    shape = tuple(e.shape_out)
    it = e.plan_item()
    qw = ops.weight_code_values(e.codes, e.kind, e.is_signed, shape[0], shape[1] * shape[2] * shape[3]).reshape(shape)
    f = torch.tensor(s, dtype=torch.float32, device=x.device) * it[8]
    layer = w.layer
    ref = conv_reference(qx.permute(0, 3, 1, 2).to(torch.int64), z, qw.to(torch.int64), it[9], f, layer.bias, layer.stride,
                         layer.dilation, ops.conv_padding(layer), x.dtype)
    return bool(torch.equal(y.float(), ref.float()))


def bench(args):
    torch.backends.cudnn.benchmark = False
    flush = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")     # 256 MB
    rows, model_rows = [], []
    for mname, make in models().items():
        for dtype in (torch.float32, torch.bfloat16):
            torch.manual_seed(0)
            base = make().to(dtype).cuda().eval()
            packed = copy.deepcopy(base)
            PW.pack_model_weights(packed)
            integer = copy.deepcopy(base)
            reports = PW.pack_model_weights(integer, integer_conv=True, integer_linear=True)
            switched = [n for n, r in reports.items() if r["weight"].get("integer_conv")]
            holders = {n: integer.get_submodule(reports[n]["weight"]["input_holder"]) for n in switched}
            for batch in args.batches:
                x = torch.randn(batch, 3, 224, 224, device="cuda").to(dtype)
                with torch.no_grad():
                    ins = layer_inputs(integer, switched, x)
                    done = set()
                    for n in switched:
                        w, wp = integer.get_submodule(n), packed.get_submodule(n)
                        xi = ins[n]
                        L = w.layer
                        key = (tuple(xi.shape), L.out_channels, L.kernel_size, L.stride)
                        if key in done:
                            continue
                        done.add(key)
                        w_res = wp._packed.rebuild(wp)[0]
                        y_int = w(xi)
                        conv = w._packed._ilin[1]                          # the launch state the call above built
                        qx, sx = conv.quantize(xi)
                        cl = conv.weight_channels_last or ops._suggests_channels_last(xi.shape, xi.stride())
                        y_gemm = conv.gemm(qx, sx, L.bias, cl)
                        t = timed({"packed": lambda: wp(xi),
                                   "float": lambda: F.conv2d(xi, w_res, L.bias, L.stride, L.padding, L.dilation),
                                   "integer": lambda: w(xi),
                                   "gemm": lambda: conv.gemm(qx, sx, L.bias, cl)}, args.reps, flush)
                        N, Cin, H, W = xi.shape
                        Ho, Wo = conv.output_hw(H, W)
                        M, K, Cout = N * Ho * Wo, Cin * L.kernel_size[0] * L.kernel_size[1], L.out_channels
                        nbytes = N * H * W * Cin + Cout * K + M * Cout * xi.element_size()
                        bound_ms = max(nbytes / (HBM_TBPS * 1e12), 2 * M * Cout * K / (INT8_POPS * 1e15)) * 1e3
                        binding = "hbm" if nbytes / (HBM_TBPS * 1e12) >= 2 * M * Cout * K / (INT8_POPS * 1e15) else "int8"
                        rows.append(dict(model=mname, dtype=str(dtype).split(".")[-1], batch=batch, layer=n,
                                         shape=f"{Cin}x{H}x{W} -> {Cout}, k{L.kernel_size[0]}x{L.kernel_size[1]} "
                                               f"s{L.stride[0]}", M=M, K=K, ms=t, bound=binding,
                                         gemm_share=bound_ms / t["gemm"], exact_integer=exact(holders[n], w, xi, y_int),
                                         exact_gemm=exact(holders[n], w, xi, y_gemm)))
                        print(json.dumps(rows[-1]), flush=True)
                    del ins
                    # whole models, eager and graph replay
                    y_p, y_i = packed(x), integer(x)
                    mrow = dict(model=mname, dtype=str(dtype).split(".")[-1], batch=batch, switched_convs=len(switched),
                                eager_packed_ms=model_ms(lambda: packed(x), args.reps),
                                eager_integer_ms=model_ms(lambda: integer(x), args.reps),
                                max_abs_diff=float((y_i.float() - y_p.float()).abs().max()),
                                max_abs_packed=float(y_p.float().abs().max()))
                    rp, ri = graphed(lambda: packed(x)), graphed(lambda: integer(x))
                    mrow["graph_packed_ms"] = model_ms(rp, args.reps)
                    mrow["graph_integer_ms"] = model_ms(ri, args.reps)
                    model_rows.append(mrow)
                    print(json.dumps(mrow), flush=True)
            del base, packed, integer
            torch.cuda.empty_cache()
    return rows, model_rows


def text(meta, rows, model_rows):
    out = [f"# {meta['card']} | cudnn.allow_tf32={meta['allow_tf32']} | torch {meta['torch']}", "",
           "## per layer (ms, median of single calls after a 256 MB cache overwrite)",
           f"{'model':13} {'dt':8} {'B':>3} {'layer':24} {'shape':32} {'packed':>8} {'float':>8} {'integer':>8} {'gemm':>8} "
           f"{'int/pk':>7} {'share':>6} exact"]
    for r in rows:
        t = r["ms"]
        out.append(f"{r['model']:13} {r['dtype']:8} {r['batch']:>3} {r['layer']:24} {r['shape']:32} {t['packed']:8.4f} "
                   f"{t['float']:8.4f} {t['integer']:8.4f} {t['gemm']:8.4f} {t['integer'] / t['packed']:7.2f} "
                   f"{r['gemm_share']:5.0%}{r['bound'][0]} {r['exact_integer'] and r['exact_gemm']}")
    out += ["", "## whole models (ms)",
            f"{'model':13} {'dt':8} {'B':>3} {'convs':>5} {'eager pk':>9} {'eager int':>9} {'graph pk':>9} {'graph int':>9} "
            f"{'max |int - pk|':>14} {'max |pk|':>9}"]
    for m in model_rows:
        out.append(f"{m['model']:13} {m['dtype']:8} {m['batch']:>3} {m['switched_convs']:>5} {m['eager_packed_ms']:9.3f} "
                   f"{m['eager_integer_ms']:9.3f} {m['graph_packed_ms']:9.3f} {m['graph_integer_ms']:9.3f} "
                   f"{m['max_abs_diff']:14.2e} {m['max_abs_packed']:9.2e}")
    return "\n".join(out) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,32,256")
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--json")
    ap.add_argument("--txt")
    args = ap.parse_args()
    args.batches = [int(b) for b in args.batches.split(",")]
    if not torch.cuda.is_available():
        sys.exit("integer_conv_bench needs a GPU")
    meta = dict(card=card(), allow_tf32=torch.backends.cudnn.allow_tf32, torch=torch.__version__)
    print(json.dumps(meta), flush=True)
    rows, model_rows = bench(args)
    meta["card_after"] = card()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(meta=meta, layers=rows, models=model_rows), f, indent=1)
    txt = text(meta, rows, model_rows)
    if args.txt:
        with open(args.txt, "w") as f:
            f.write(txt)
    print(txt)


if __name__ == "__main__":
    main()
