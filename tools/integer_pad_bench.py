#!/usr/bin/env python
"""Padded integer modes (integer_pad=True, DESIGN §7f) against the packed path, per layer and per model, on one GPU.

    python tools/integer_pad_bench.py [--json out.json] [--txt out.txt] [--batches 1,32,256] [--reps 10]

Per layer: the groups-1 convs of MCT-style MobileNetV3-large and EfficientNet-B0 (tests/test_integer_pad.mct_style: every
Conv2d / Linear wrapped, a holder on the input and after every activation) that integer convolution mode refuses without
integer_pad (Cin off 16), distinct by shape, and the ResNet-18 / MobileNetV2 stems, at 224 x 224, every batch, f32 and bf16,
int8 per-channel symmetric weights.  Two arms, timed with CUDA events around one call, a 256 MB buffer overwritten before
every call (the 126 MB L2 holds nothing of the layer), median over --reps, arms alternated inside each repetition:
    packed    the wrapper's packed path: rebuild the weight (UnpackPlan) + F.conv2d (cuDNN)
    integer   the wrapper with integer_conv=True, integer_pad=True: the padded quantizer + mctq_packed_conv2d_i8_padded
Every integer output is compared bit for bit with the formula of include/mctq.h (tests/test_integer_conv.conv_reference).
Two ablations at the largest batch in f32, same timing: a Cin = 120 conv padded to 128 against the same conv with a native
Cin = 128; and the ResNet-18 stem through the narrow gather (Cp = 4) against the same stem padded to Cp = 16 through the wide
gather.  Whole model: eager forward of the two MCT-style models with integer_linear, integer_conv and integer_depthwise,
with and without integer_pad, with the number of switched layers.  The card's name, power limit and clocks are read in the
same run.
"""
import argparse
import copy
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mct_quantizers_b200 as mctq  # noqa: E402
from mct_quantizers_b200 import ops  # noqa: E402
from mct_quantizers_b200.pytorch import packed_weights as PW  # noqa: E402
from mct_quantizers_b200.pytorch import quantizers as Q  # noqa: E402
from integer_conv_bench import model_ms, timed  # noqa: E402
from packed_linear_bench import card  # noqa: E402
from test_integer_conv import _fake_pack_model, _launch_args, _scalar_codes, conv_reference  # noqa: E402
from test_integer_pad import mct_style  # noqa: E402

HOLDER_Q = Q.ActivationUniformInferableQuantizer(8, [-1.0], [6.0])


def new_layers():
    """[(model, layer names, Cin, Cout, k, stride, padding, H)] of the groups-1 convs integer_pad newly switches, plus the
    two stems, distinct by shape."""
    import torchvision
    shapes = {}
    for name in ("mobilenet_v3_large", "efficientnet_b0"):
        plain = getattr(torchvision.models, name)(weights=None).eval()
        seen, hooks = {}, []                          # input sizes, traced on the float model (mct_style's "1." prefix)
        for n, m in plain.named_modules():
            if isinstance(m, torch.nn.Conv2d):
                hooks.append(m.register_forward_pre_hook(lambda m, a, n=n: seen.__setitem__("1." + n, a[0].shape[2])))
        with torch.no_grad():
            plain(torch.zeros(1, 3, 224, 224))
        for h in hooks:
            h.remove()
        model = mct_style(plain)
        rep = PW.pack_model_weights(_fake_pack_model(copy.deepcopy(model)), integer_conv=True)
        for n, r in rep.items():
            L = model.get_submodule(n).layer
            if isinstance(L, torch.nn.Conv2d) and L.groups == 1 and "is not a multiple of 16" in r["weight"]["integer_conv_reason"]:
                key = (L.in_channels, L.out_channels, L.kernel_size[0], L.stride[0], L.padding[0], seen[n])
                shapes.setdefault(key, (name, []))[1].append(n)
    shapes.setdefault((3, 64, 7, 2, 3, 224), ("resnet18", []))[1].append("resnet18 conv1")
    shapes.setdefault((3, 32, 3, 2, 1, 224), ("mobilenet_v2", []))[1].append("mobilenet_v2 features.0.0")
    return [(m, names) + key for key, (m, names) in shapes.items()]


def wrappers(cin, cout, k, stride, padding, dtype):
    conv = torch.nn.Conv2d(cin, cout, k, stride=stride, padding=padding)
    thr = [float(t) for t in conv.weight.detach().abs().reshape(cout, -1).amax(1).clamp_min(1e-6)]
    base = mctq.PytorchQuantizationWrapper(conv, {"weight": Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0)})
    base = base.to(dtype).cuda()
    packed, integer = copy.deepcopy(base), copy.deepcopy(base)
    packed.pack_weights()
    rep = integer.pack_weights(integer_conv=True, integer_pad=True, input_quantizer=HOLDER_Q)
    assert rep["weight"]["integer_conv"], rep
    return packed, integer


def exact(w, x, y):
    """y equals the formula for wrapper w on input x, bit for bit."""
    e = w._packed.entries[0]
    s, z, qmin, qmax = _launch_args(HOLDER_Q)
    qx = _scalar_codes(x, s, z, qmin, qmax).to(torch.int64)
    Cout, Cin, kh, kw = e.shape_out
    qw = ops.weight_code_values(e.codes, e.kind, e.is_signed, Cout, Cin * kh * kw).to(torch.int64).reshape(Cout, Cin, kh, kw)
    it = e.plan_item()
    f = torch.tensor(np.float32(s), device=x.device) * it[8]
    L = w.layer
    ref = conv_reference(qx, z, qw, it[9], f, L.bias, L.stride, L.dilation, ops.conv_padding(L), x.dtype)
    return bool(torch.equal(y.float(), ref.float()))


def holder_input(batch, cin, h, dtype):
    holder = mctq.PytorchActivationQuantizationHolder(HOLDER_Q).cuda()
    return holder(torch.nn.functional.relu6(torch.randn(batch, cin, h, h, device="cuda") * 3).to(dtype))


def layer_rows(args, flush):
    rows = []
    for model, names, cin, cout, k, stride, padding, h in new_layers():
        for batch in args.batches:
            for dtype in (torch.float32, torch.bfloat16):
                torch.manual_seed(0)
                packed, integer = wrappers(cin, cout, k, stride, padding, dtype)
                with torch.no_grad():
                    x = holder_input(batch, cin, h, dtype)
                    y = integer(x)
                    t = timed({"packed": lambda: packed(x), "integer": lambda: integer(x)}, args.reps, flush)
                    ok = exact(integer, x, y)
                rows.append(dict(model=model, layers=names, dtype=str(dtype).split(".")[-1], batch=batch,
                                 shape=f"{cin}->{cout} k{k} s{stride} {h}^2", cp=integer._packed._ilin[1].cp, ms=t,
                                 exact=ok))
                print(json.dumps(rows[-1]), flush=True)
                del x, y, packed, integer
    return rows


def ablation_rows(args, flush):
    rows, batch = [], max(args.batches)
    with torch.no_grad():
        # padding cost: Cin 120 padded to 128 against a native Cin = 128 (1x1 to 480 at 28 x 28, MobileNetV3-large's shape)
        arms, outs = {}, {}
        for cin in (120, 128):
            torch.manual_seed(0)
            _, integer = wrappers(cin, 480, 1, 1, 0, torch.float32)
            x = holder_input(batch, cin, 28, torch.float32)
            arms[f"cin{cin}"] = (lambda w=integer, x=x: w(x))
            outs[cin] = exact(integer, x, integer(x))
        rows.append(dict(case="Cin 120 padded to 128 vs native 128, 1x1 -> 480, 28^2, f32", batch=batch,
                         ms=timed(arms, args.reps, flush), exact=all(outs.values())))
        print(json.dumps(rows[-1]), flush=True)
        # the stem: narrow gather (Cp = 4) against the wide gather with Cp = 16
        torch.manual_seed(0)
        _, integer = wrappers(3, 64, 7, 2, 3, torch.float32)
        x = holder_input(batch, 3, 224, torch.float32)
        y = integer(x)
        narrow = integer._packed._ilin[1]
        e = integer._packed.entries[0]
        qw = ops.padded_code_rows(e.codes, e.kind, e.is_signed, 64, 3, 7, 7, False, 16, 49 * 16)
        wide = ops.IntegerConv2d.from_parts(ops.pack_code_rows(qw, e.kind, e.is_signed, e.codes), e.kind, e.is_signed,
                                            torch.float32, 64, 3, (7, 7), (2, 2), (1, 1), (3, 3, 3, 3), narrow.factor,
                                            narrow._w._keep[2], qw.sum(1, dtype=torch.int32), narrow.x_zp, cp=16)
        s, z, qmin, qmax = _launch_args(HOLDER_Q)

        def run_wide():
            qx, P = ops.quantize_nhwc_i8_padded(x, 16, s, z, qmin, qmax, False)
            return wide.gemm(qx, None, integer.layer.bias)
        same = bool(torch.equal(run_wide(), y))
        rows.append(dict(case="ResNet-18 stem 3->64 k7 s2 224^2 f32: narrow Cp=4 vs wide Cp=16", batch=batch,
                         ms=timed({"narrow_cp4": lambda: integer(x), "wide_cp16": run_wide}, args.reps, flush),
                         exact=exact(integer, x, y) and same))
        print(json.dumps(rows[-1]), flush=True)
    return rows


def model_rows(args):
    import torchvision
    rows = []
    for name in ("mobilenet_v3_large", "efficientnet_b0"):
        torch.manual_seed(0)
        base = mct_style(getattr(torchvision.models, name)(weights=None).eval()).cuda()
        arms, switched = {}, {}
        flags = dict(integer_linear=True, integer_conv=True, integer_depthwise=True)
        for k, pad in (("packed", None), ("integer", False), ("integer_pad", True)):
            arms[k] = copy.deepcopy(base)
            rep = PW.pack_model_weights(arms[k], **(dict(flags, integer_pad=pad) if pad is not None else {}))
            switched[k] = sum(bool(r["weight"].get("integer_conv") or r["weight"].get("integer")) for r in rep.values())
        for batch in args.batches:
            x = torch.randn(batch, 3, 224, 224, device="cuda")
            with torch.no_grad():
                row = dict(model=name, dtype="float32", batch=batch, switched_layers=switched,
                           eager_ms={k: model_ms(lambda m=m: m(x), args.reps) for k, m in arms.items()})
            rows.append(row)
            print(json.dumps(row), flush=True)
            del x
        del base, arms
        torch.cuda.empty_cache()
    return rows


def text(meta, rows, arows, mrows):
    out = [f"# {meta['card']} | cudnn.allow_tf32={meta['allow_tf32']} | torch {meta['torch']}", "",
           "## per layer (ms, median of single calls after a 256 MB cache overwrite)",
           f"{'model':18} {'shape':24} {'Cp':>4} {'dt':8} {'B':>3} {'packed':>8} {'integer':>8} {'pk/int':>7} exact  layers"]
    for r in rows:
        t = r["ms"]
        out.append(f"{r['model']:18} {r['shape']:24} {r['cp']:>4} {r['dtype']:8} {r['batch']:>3} {t['packed']:8.4f} "
                   f"{t['integer']:8.4f} {t['packed'] / t['integer']:7.2f} {str(r['exact']):5}  {','.join(r['layers'])}")
    out += ["", "## ablations (ms, same timing)"]
    for r in arows:
        out.append(f"{r['case']} | B={r['batch']} | " + " ".join(f"{k}={v:.4f}" for k, v in r["ms"].items()) +
                   f" | exact={r['exact']}")
    out += ["", "## whole model, eager f32 (ms per forward; switched layers in brackets)",
            f"{'model':18} {'B':>3} {'packed':>9} {'integer':>9} {'+pad':>9}"]
    for m in mrows:
        e, s = m["eager_ms"], m["switched_layers"]
        out.append(f"{m['model']:18} {m['batch']:>3} {e['packed']:9.3f} {e['integer']:9.3f} {e['integer_pad']:9.3f}   "
                   f"[{s['integer']} / {s['integer_pad']}]")
    return "\n".join(out) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,32,256")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--json")
    ap.add_argument("--txt")
    args = ap.parse_args()
    args.batches = [int(b) for b in args.batches.split(",")]
    if not torch.cuda.is_available():
        sys.exit("integer_pad_bench needs a GPU")
    torch.backends.cudnn.benchmark = False
    meta = dict(card=card(), allow_tf32=torch.backends.cudnn.allow_tf32, torch=torch.__version__)
    print(json.dumps(meta), flush=True)
    flush = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")     # 256 MB
    rows = layer_rows(args, flush)
    arows = ablation_rows(args, flush)
    mrows = model_rows(args)
    meta["card_after"] = card()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(meta=meta, layers=rows, ablations=arows, models=mrows), f, indent=1)
    txt = text(meta, rows, arows, mrows)
    if args.txt:
        with open(args.txt, "w") as f:
            f.write(txt)
    print(txt)


if __name__ == "__main__":
    main()
