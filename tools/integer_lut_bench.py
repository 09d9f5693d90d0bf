"""Integer modes for LUT weights against the existing paths, on one GPU.

Linear: the Llama-7B MLP matrices (gate / up 11008x4096, down 4096x11008) as 4-bit LUT f32 weights (packed_bench.lut_q:
16 integer centroids on an 8-bit grid, per-channel thresholds), M = 1 .. 4096 input rows, and one 8-bit-index LUT
shape (64 centroids).  Arms, per (shape, M):
  int_lut_e2e    IntegerLinear with the LUT table: row quantizer + GEMM (mctq_packed_linear_i8_lut)
  int_lut_gemm   the GEMM alone, on precomputed codes
  int4_gemm      the int4 affine integer GEMM at the same shape (mctq_packed_linear_i8)
  f32_best       the best existing f32 LUT path: fused (M <= 8), batched (M <= 256), else rebuild + F.linear
Every integer output is checked bit for bit against the exact formula (f64 code sums, exact at these sizes).
Conv: ResNet-18 with 4-bit LUT POT weights on every Conv2d / Linear and an 8-bit holder behind every ReLU, eager f32
forward at batch 1 and 256 (224x224), packed path against integer_conv + integer_linear + integer_lut; the integer model's
output must be the same bits in every timed call.
A 256 MB buffer is overwritten before every timed call, so no call reads its weights from L2.  The card's name and power
limit are read in the same run.  Writes profiles/r08_integer_lut_bench.{json,txt} (or --out PREFIX).

    python tools/integer_lut_bench.py [--reps 20] [--out profiles/r08_integer_lut_bench]
"""
import argparse
import copy
import importlib.util
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mct_quantizers_b200 as mctq  # noqa: E402
from mct_quantizers_b200 import _native, ops  # noqa: E402
from mct_quantizers_b200.pytorch import packed_weights as PW  # noqa: E402
from mct_quantizers_b200.pytorch import quantizers as Q  # noqa: E402

_spec = importlib.util.spec_from_file_location("packed_bench", os.path.join(ROOT, "tools", "packed_bench.py"))
pb = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(pb)

MS = [1, 8, 16, 32, 64, 128, 256, 512, 1024, 4096]
SHAPES = [(11008, 4096, 16), (4096, 11008, 16), (11008, 4096, 64)]       # (out, in, LUT entries)


class Flush:
    def __init__(self):
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def __call__(self):
        self.buf.fill_(1)


def timed(fn, flush, reps):
    """Median device time (ms) of fn, the cache overwritten before each call; returns (ms, outputs of every timed call)."""
    for _ in range(2):
        fn()
    outs, ts = [], []
    for _ in range(reps):
        flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        y = fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
        outs.append(y)
    ts.sort()
    return ts[len(ts) // 2], outs


def lut_quantizer(N, K):
    if K == 16:
        return pb.lut_q(N)
    lut = [float(v) for v in np.linspace(-128, 127, K).round()]
    return Q.WeightsLUTSymmetricInferableQuantizer(6, lut, [0.02 + 0.0001 * (c % 97) for c in range(N)], True, 0, 2, 8)


def exact(qx, qw, zx, f):
    c = qx.double() @ qw.double().T - zx * qw.double().sum(1)[None, :]
    return c.to(torch.int64).to(torch.float32) * f[None, :]


def linear_rows(reps, flush):
    rows = []
    xq_ = Q.ActivationSymmetricInferableQuantizer(8, [4.0], True)
    from mct_quantizers_b200.pytorch.fused_activation_holder import affine_scalar_params
    s, z, _, _ = affine_scalar_params(xq_)
    x_scale, x_zp, qmin, qmax = xq_._validated_launch_args(s, z)[1]
    for N, K, L in SHAPES:
        torch.manual_seed(0)
        lin = torch.nn.Linear(K, N, bias=False, device="cuda")
        torch.nn.init.normal_(lin.weight, std=0.02)
        w = mctq.PytorchQuantizationWrapper(lin, {"weight": lut_quantizer(N, L)})
        w.pack_weights(fused_linear=True, batched_linear=True)
        e = w._packed.entries[0]
        item = e.plan_item()
        wq = e.quantizer
        sw = item[8] * 2.0 ** -(int(wq.lut_values_bitwidth) - 1)
        ilut = ops.IntegerLinear(e.codes, e.kind, False, torch.float32, N, K, sw, None, x_scale, x_zp, qmin, qmax,
                                 wq._lut_values_np)
        qw = torch.from_numpy(ilut.lut.astype(np.int64)).cuda()[ops.weight_code_values(e.codes, e.kind, False, N, K).long()]
        g = torch.Generator(device="cuda").manual_seed(1)
        i4codes = torch.randint(0, 256, (N * K // 2,), dtype=torch.uint8, device="cuda", generator=g)
        i4 = ops.IntegerLinear(i4codes, _native.PACK_AFFINE_I4, True, torch.float32, N, K, sw, torch.zeros_like(sw, dtype=torch.int32),
                               x_scale, x_zp, qmin, qmax)
        plan = ops.UnpackPlan([item], fresh=True)
        for M in MS:
            x = torch.randn(M, K, device="cuda") * 2
            qx, _ = ilut.quantize(x)
            ref = exact(qx, qw, x_zp, ilut.factor)
            t_e2e, o1 = timed(lambda: ilut(x), flush, reps)
            t_gemm, o2 = timed(lambda: ilut.gemm(qx), flush, reps)
            t_i4, _ = timed(lambda: i4.gemm(qx), flush, reps)
            if M <= 256:                                 # the wrapper's fused (M <= 8) or batched kernel
                best, fn = "fused" if M <= 8 else "batched", lambda: w(x)
            else:
                best, fn = "rebuild+F.linear", lambda: torch.nn.functional.linear(x, plan.run()[0])
            with torch.no_grad():
                t_f32, _ = timed(lambda: fn(), flush, reps)
            ok = all(torch.equal(o.view(torch.int32), ref.view(torch.int32)) for o in o1 + o2)
            rows.append(dict(shape=f"{N}x{K}", lut_entries=L, kind=PW._KIND_NAMES[e.kind], M=M, int_lut_e2e_ms=t_e2e,
                             int_lut_gemm_ms=t_gemm, int4_gemm_ms=t_i4, f32_best_ms=t_f32, f32_best=best,
                             gemm_over_int4=t_gemm / t_i4, e2e_speedup_vs_f32=t_f32 / t_e2e, bit_exact=ok))
            print(json.dumps(rows[-1]), flush=True)
            assert ok, rows[-1]
    return rows


def lut_resnet18():
    import torchvision
    torch.manual_seed(0)
    model = torchvision.models.resnet18(weights=None).eval()

    def convert(parent):
        for name, child in list(parent.named_children()):
            if isinstance(child, (torch.nn.Conv2d, torch.nn.Linear)):
                w = child.weight.detach()
                thr = [2.0 ** float(np.ceil(np.log2(max(float(t), 1e-6)))) for t in w.abs().reshape(w.shape[0], -1).amax(1)]
                lut = [float(v) for v in range(-128, 128, 16)]
                q = Q.WeightsLUTPOTInferableQuantizer(4, lut, thr, True, 0, w.dim(), 8)
                setattr(parent, name, mctq.PytorchQuantizationWrapper(child, {"weight": q}))
            elif isinstance(child, torch.nn.ReLU):
                holder = mctq.PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [0.0], [4.0]))
                setattr(parent, name, torch.nn.Sequential(torch.nn.ReLU(), holder))
            else:
                convert(child)
    convert(model)
    return model.cuda()


def resnet_rows(reps, flush):
    rows = []
    base = lut_resnet18()
    packed = copy.deepcopy(base)
    PW.pack_model_weights(packed)
    integer = copy.deepcopy(base)
    rep = PW.pack_model_weights(integer, integer_linear=True, integer_conv=True, integer_lut=True)
    switched = sum(1 for r in rep.values() if r["weight"].get("integer_conv") or r["weight"].get("integer"))
    for B in (1, 256):
        x = torch.randn(B, 3, 224, 224, device="cuda")
        with torch.no_grad():
            t_p, _ = timed(lambda: packed(x), flush, reps)
            t_i, outs = timed(lambda: integer(x), flush, reps)
        same = all(torch.equal(o, outs[0]) for o in outs)
        rows.append(dict(model="resnet18_lut4_pot", batch=B, switched_layers=switched, packed_ms=t_p, integer_ms=t_i,
                         speedup=t_p / t_i, repeat_bit_identical=same))
        print(json.dumps(rows[-1]), flush=True)
        assert same
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_integer_lut_bench"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    card = pb.card()
    print(card, flush=True)
    flush = Flush()
    lin = linear_rows(a.reps, flush)
    res = resnet_rows(a.reps, flush)
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out + ".json", "w") as fh:
        json.dump(dict(card=card, cache="256 MB overwritten before every timed call", reps=a.reps, linear=lin, resnet18=res),
                  fh, indent=1)
    with open(a.out + ".txt", "w") as fh:
        fh.write(f"# {card}\n# median of {a.reps} calls, ms, cache overwritten before each call; f32 LUT weights\n")
        fh.write(f"{'shape':>11} {'L':>3} {'M':>5} {'lut_e2e':>8} {'lut_gemm':>8} {'int4_gemm':>9} {'gemm/i4':>7} "
                 f"{'f32_best':>8} {'(path)':>16} {'f32/e2e':>7}\n")
        for r in lin:
            fh.write(f"{r['shape']:>11} {r['lut_entries']:>3} {r['M']:>5} {r['int_lut_e2e_ms']:8.4f} {r['int_lut_gemm_ms']:8.4f} "
                     f"{r['int4_gemm_ms']:9.4f} {r['gemm_over_int4']:7.2f} {r['f32_best_ms']:8.4f} {r['f32_best']:>16} "
                     f"{r['e2e_speedup_vs_f32']:7.2f}\n")
        for r in res:
            fh.write(f"resnet18 LUT4 POT batch {r['batch']}: packed {r['packed_ms']:.3f} ms, integer {r['integer_ms']:.3f} ms "
                     f"({r['switched_layers']} layers switched), speedup {r['speedup']:.2f}\n")
    print("wrote", a.out + ".{json,txt}")


if __name__ == "__main__":
    main()
