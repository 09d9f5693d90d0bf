#!/usr/bin/env python
"""Integer convolution mode for depthwise Conv2d (mctq_packed_dwconv2d_i8) against the packed path, per layer and per model,
on one GPU.

    python tools/integer_depthwise_bench.py [--json out.json] [--txt out.txt] [--batches 1,32,256] [--reps 15]

Per layer: the distinct shapes of MobileNetV2's 17 depthwise 3x3 convs at 224 x 224 (C = 32..960, 112^2 down to 7^2,
stride 1 / 2, pad 1), each fed by a uniform 8-bit ReLU6 holder (tools/model_forward_bench.quantize_model), at every batch in
f32 and bf16 with int8 per-channel symmetric weights, and at the largest batch in f32 also with int4 symmetric and 4-bit
LUT weights.  Two arms, timed with CUDA events around one call, a 256 MB buffer overwritten before every call (the 126 MB
L2 holds nothing of the layer), median over --reps, arms alternated inside each repetition:
    packed    the wrapper's packed path: rebuild the weight (UnpackPlan) + F.conv2d (cuDNN; f32 runs TF32 when
              torch.backends.cudnn.allow_tf32, recorded below)
    kernel    the wrapper in integer depthwise mode: one mctq_packed_dwconv2d_i8 launch
Per row also the bytes the kernel must move (float x read + y write + weight codes), its share of the HBM bound at 7.7 TB/s
(the data-sheet bandwidth of one B200 at 1000 W, not a measured figure), and whether the kernel's output equals the formula
of include/mctq.h (tests/test_integer_depthwise.dw_reference) bit for bit.
Whole model: MobileNetV2 forward packed, with integer_conv=True, and with integer_conv=True, integer_depthwise=True, eager
at every batch and replayed from a CUDA graph up to batch 32, with the number of switched convs.  The card's name, power
limit and clocks are read in the same run.
"""
import argparse
import copy
import json
import os
import statistics
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mct_quantizers_b200 as mctq  # noqa: E402
from mct_quantizers_b200 import _native, ops  # noqa: E402
from mct_quantizers_b200.pytorch import packed_weights as PW  # noqa: E402
from mct_quantizers_b200.pytorch import quantizers as Q  # noqa: E402
from integer_conv_bench import graphed, model_ms, timed  # noqa: E402
from model_forward_bench import quantize_model  # noqa: E402
from packed_linear_bench import HBM_TBPS, card  # noqa: E402
from test_integer_conv import _launch_args  # noqa: E402
from test_integer_depthwise import dw_reference  # noqa: E402


def mobilenet():
    import torchvision
    return quantize_model(torchvision.models.mobilenet_v2(), mctq, Q)


def depthwise_shapes():
    """{(C, H, stride): [layer names]} of MobileNetV2's depthwise convs at 224 x 224."""
    import torchvision
    model, shapes, hooks = torchvision.models.mobilenet_v2(), {}, []
    for n, m in model.named_modules():
        if isinstance(m, torch.nn.Conv2d) and m.groups > 1:
            hooks.append(m.register_forward_pre_hook(
                lambda m, a, n=n: shapes.setdefault((a[0].shape[1], a[0].shape[2], m.stride[0]), []).append(n)))
    with torch.no_grad():
        model(torch.zeros(1, 3, 224, 224))
    for h in hooks:
        h.remove()
    return shapes


def weight_quantizer(fmt, conv):
    w = conv.weight.detach()
    thr = [float(t) for t in w.abs().reshape(w.shape[0], -1).amax(1).clamp_min(1e-6)]
    if fmt == "int8":
        return Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)
    if fmt == "int4":
        return Q.WeightsSymmetricInferableQuantizer(4, thr, True, 0)
    with warnings.catch_warnings():          # 4-bit LUT: 16 integer centroids on an 8-bit grid, power-of-two thresholds
        warnings.simplefilter("ignore")
        pot = [float(2.0 ** np.ceil(np.log2(t))) for t in thr]
        return Q.WeightsLUTPOTInferableQuantizer(4, [float(v) for v in range(-128, 128, 16)], pot, True, 0, 4, 8)


def exact(w, q, x, y):
    """y equals the formula for wrapper w (input quantizer q) on input x, bit for bit (reference in float64 on the GPU)."""
    e = w._packed.entries[0]
    s, z, qmin, qmax = _launch_args(q)
    codes, _ = ops.quantize_rows_i8(x.permute(0, 2, 3, 1), s, z, qmin, qmax, False)
    qx = codes.permute(0, 3, 1, 2).to(torch.int64)
    Cout, _, kh, kw = e.shape_out
    qw = ops.weight_code_values(e.codes, e.kind, e.is_signed, Cout, kh * kw).to(torch.int64)
    it = e.plan_item()
    sc, zw = it[8], it[9]
    if e.kind in _native.PACK_LUT_KINDS:
        qw = torch.as_tensor(e.quantizer._lut_values_np).to(torch.int64).to(x.device)[qw]
        sc = sc * 2.0 ** -(int(e.quantizer.lut_values_bitwidth) - 1)
        zw = torch.zeros(1, dtype=torch.int32, device=x.device)
    f = torch.tensor(np.float32(s), device=x.device) * sc
    L = w.layer
    ref = dw_reference(qx, z, qw.reshape(Cout, 1, kh, kw), zw, f, L.bias, L.stride, L.dilation, ops.conv_padding(L), x.dtype)
    return bool(torch.equal(y.float(), ref.float()))


def layer_rows(args, flush):
    rows = []
    holder_q = Q.ActivationUniformInferableQuantizer(8, [0.0], [6.0])
    holder = mctq.PytorchActivationQuantizationHolder(holder_q).cuda()
    cases = [(b, dt, "int8") for b in args.batches for dt in (torch.float32, torch.bfloat16)]
    cases += [(max(args.batches), torch.float32, fmt) for fmt in ("int4", "lut4")]
    for (C, H, s), names in depthwise_shapes().items():
        for batch, dtype, fmt in cases:
            torch.manual_seed(0)
            conv = torch.nn.Conv2d(C, C, 3, stride=s, padding=1, groups=C)
            base = mctq.PytorchQuantizationWrapper(conv, {"weight": weight_quantizer(fmt, conv)}).to(dtype).cuda()
            packed, integer = copy.deepcopy(base), copy.deepcopy(base)
            packed.pack_weights()
            rep = integer.pack_weights(integer_conv=True, integer_depthwise=True, integer_lut=fmt == "lut4",
                                       input_quantizer=holder_q)
            assert rep["weight"]["integer_conv"], rep
            with torch.no_grad():
                x = holder(torch.nn.functional.relu6(torch.randn(batch, C, H, H, device="cuda") * 3).to(dtype))
                y = integer(x)
                t = timed({"packed": lambda: packed(x), "kernel": lambda: integer(x)}, args.reps, flush)
                ok = exact(integer, holder_q, x, y)
            e = integer._packed.entries[0]
            nbytes = x.numel() * x.element_size() + y.numel() * y.element_size() + e.codes.numel()
            rows.append(dict(layers=names, dtype=str(dtype).split(".")[-1], weights=fmt, batch=batch,
                             shape=f"{C}x{H}x{H} s{s}", bytes=nbytes, ms=t,
                             hbm_share=nbytes / (HBM_TBPS * 1e12) * 1e3 / t["kernel"], exact=ok))
            print(json.dumps(rows[-1]), flush=True)
            del x, y, packed, integer, base
    return rows


def model_rows(args):
    rows = []
    for dtype in (torch.float32, torch.bfloat16):
        torch.manual_seed(0)
        base = mobilenet().to(dtype).cuda().eval()
        arms = {"packed": copy.deepcopy(base), "integer_conv": copy.deepcopy(base), "depthwise": copy.deepcopy(base)}
        switched = {"packed": 0}
        PW.pack_model_weights(arms["packed"])
        for k, flags in (("integer_conv", {}), ("depthwise", {"integer_depthwise": True})):
            rep = PW.pack_model_weights(arms[k], integer_conv=True, **flags)
            switched[k] = sum(bool(r["weight"]["integer_conv"]) for r in rep.values())
        for batch in args.batches:
            x = torch.randn(batch, 3, 224, 224, device="cuda").to(dtype)
            with torch.no_grad():
                row = dict(dtype=str(dtype).split(".")[-1], batch=batch, switched_convs=switched,
                           eager_ms={k: model_ms(lambda m=m: m(x), args.reps) for k, m in arms.items()})
                if batch <= 32:
                    row["graph_ms"] = {k: model_ms(graphed(lambda m=m: m(x)), args.reps) for k, m in arms.items()}
            rows.append(row)
            print(json.dumps(row), flush=True)
            del x
        del base, arms
        torch.cuda.empty_cache()
    return rows


def text(meta, rows, mrows):
    out = [f"# {meta['card']} | cudnn.allow_tf32={meta['allow_tf32']} | torch {meta['torch']}", "",
           "## per layer (ms, median of single calls after a 256 MB cache overwrite; share: of 7.7 TB/s for x + y + codes)",
           f"{'shape':16} {'dt':8} {'w':5} {'B':>3} {'MB':>8} {'packed':>8} {'kernel':>8} {'pk/kern':>7} {'share':>6} exact  layers"]
    for r in rows:
        t = r["ms"]
        out.append(f"{r['shape']:16} {r['dtype']:8} {r['weights']:5} {r['batch']:>3} {r['bytes'] / 1e6:8.1f} {t['packed']:8.4f} "
                   f"{t['kernel']:8.4f} {t['packed'] / t['kernel']:7.2f} {r['hbm_share']:6.0%} {str(r['exact']):5}  "
                   f"{','.join(n.replace('features.', 'f').replace('.conv', '') for n in r['layers'])}")
    out += ["", "## MobileNetV2 (ms per forward; switched convs: packed 0, integer_conv "
            f"{mrows[0]['switched_convs']['integer_conv']}, +depthwise {mrows[0]['switched_convs']['depthwise']})",
            f"{'dt':8} {'B':>3} {'eager pk':>9} {'eager ic':>9} {'eager dw':>9} {'graph pk':>9} {'graph ic':>9} {'graph dw':>9}"]
    for m in mrows:
        e, g = m["eager_ms"], m.get("graph_ms")
        gs = f"{g['packed']:9.3f} {g['integer_conv']:9.3f} {g['depthwise']:9.3f}" if g else f"{'-':>9} {'-':>9} {'-':>9}"
        out.append(f"{m['dtype']:8} {m['batch']:>3} {e['packed']:9.3f} {e['integer_conv']:9.3f} {e['depthwise']:9.3f} {gs}")
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
        sys.exit("integer_depthwise_bench needs a GPU")
    torch.backends.cudnn.benchmark = False
    meta = dict(card=card(), allow_tf32=torch.backends.cudnn.allow_tf32, torch=torch.__version__)
    print(json.dumps(meta), flush=True)
    flush = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")     # 256 MB
    rows = layer_rows(args, flush)
    mrows = model_rows(args)
    meta["card_after"] = card()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(meta=meta, layers=rows, models=mrows), f, indent=1)
    txt = text(meta, rows, mrows)
    if args.txt:
        with open(args.txt, "w") as f:
            f.write(txt)
    print(txt)


if __name__ == "__main__":
    main()
