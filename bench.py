#!/usr/bin/env python
"""bench.py -- fake-quant throughput of the B200 path on BASELINE.json's configs[1]:
"MobileNetV2 full-model PytorchQuantizationWrapper 8-bit per-channel weights + uniform activations, batch 256".

A step = one pass of the hot path over the whole model: the 53 conv/linear weight tensors through
WeightsSymmetricInferableQuantizer (8 bit, per-channel axis 0; one multi-tensor launch) and the 53 conv/linear
output activations at batch 256 through PytorchActivationQuantizationHolder(ActivationUniformInferableQuantizer
8 bit) -- 1.71 G f32 elements, 13.7 GB of algorithmic HBM traffic per step per GPU.

    python bench.py --gpus N --steps K --warmup W                 (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W (the reference's CPU torch path, rank 0 only)
    python bench.py ... --dump-outputs DIR                         (also write the last timed step's outputs to DIR/*.npy)

Prints ONE JSON line (rank 0).  metric = algorithmic GB/s (8 B per f32 element), whole job.
Multi-GPU: activations shard by batch (every rank owns 256 images: weak scaling), weights shard by layer; there is
no collective on the data path -- NCCL only gathers checksums after the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# torchvision.models.mobilenet_v2: conv / linear weight shapes and per-image output shapes (53 each)
MBV2_WEIGHTS = [(32, 3, 3, 3), (32, 1, 3, 3), (16, 32, 1, 1), (96, 16, 1, 1), (96, 1, 3, 3), (24, 96, 1, 1), (144, 24, 1, 1),
                (144, 1, 3, 3), (24, 144, 1, 1), (144, 24, 1, 1), (144, 1, 3, 3), (32, 144, 1, 1), (192, 32, 1, 1),
                (192, 1, 3, 3), (32, 192, 1, 1), (192, 32, 1, 1), (192, 1, 3, 3), (32, 192, 1, 1), (192, 32, 1, 1),
                (192, 1, 3, 3), (64, 192, 1, 1), (384, 64, 1, 1), (384, 1, 3, 3), (64, 384, 1, 1), (384, 64, 1, 1),
                (384, 1, 3, 3), (64, 384, 1, 1), (384, 64, 1, 1), (384, 1, 3, 3), (64, 384, 1, 1), (384, 64, 1, 1),
                (384, 1, 3, 3), (96, 384, 1, 1), (576, 96, 1, 1), (576, 1, 3, 3), (96, 576, 1, 1), (576, 96, 1, 1),
                (576, 1, 3, 3), (96, 576, 1, 1), (576, 96, 1, 1), (576, 1, 3, 3), (160, 576, 1, 1), (960, 160, 1, 1),
                (960, 1, 3, 3), (160, 960, 1, 1), (960, 160, 1, 1), (960, 1, 3, 3), (160, 960, 1, 1), (960, 160, 1, 1),
                (960, 1, 3, 3), (320, 960, 1, 1), (1280, 320, 1, 1), (1000, 1280)]
MBV2_ACTS = [(32, 112, 112), (32, 112, 112), (16, 112, 112), (96, 112, 112), (96, 56, 56), (24, 56, 56), (144, 56, 56),
             (144, 56, 56), (24, 56, 56), (144, 56, 56), (144, 28, 28), (32, 28, 28), (192, 28, 28), (192, 28, 28),
             (32, 28, 28), (192, 28, 28), (192, 28, 28), (32, 28, 28), (192, 28, 28), (192, 14, 14), (64, 14, 14),
             (384, 14, 14), (384, 14, 14), (64, 14, 14), (384, 14, 14), (384, 14, 14), (64, 14, 14), (384, 14, 14),
             (384, 14, 14), (64, 14, 14), (384, 14, 14), (384, 14, 14), (96, 14, 14), (576, 14, 14), (576, 14, 14),
             (96, 14, 14), (576, 14, 14), (576, 14, 14), (96, 14, 14), (576, 14, 14), (576, 7, 7), (160, 7, 7), (960, 7, 7),
             (960, 7, 7), (160, 7, 7), (960, 7, 7), (960, 7, 7), (160, 7, 7), (960, 7, 7), (960, 7, 7), (320, 7, 7),
             (1280, 7, 7), (1000,)]
BYTES_PER_ELEM = 8           # f32 in + f32 out (SURVEY 8d)
METRIC = "fake-quant algorithmic HBM GB/s (MobileNetV2 weights + activations, batch 256 per GPU)"
WORKLOAD = "MobileNetV2 full model: 53 per-channel 8-bit WeightsSymmetric tensors + 53 ActivationUniform 8-bit sites, batch 256, f32"


def numel(shape):
    n = 1
    for s in shape:
        n *= s
    return n


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="images per GPU")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--profiler-range", action="store_true", help="bracket the timed region with cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-batch", type=int, default=64, help="images per step of the cpu_baseline sample inside the B200 arm's line "
                    "(--impl reference itself runs the full --batch)")
    ap.add_argument("--no-per-config", action="store_true", help="skip the C1 / C3 / C4 / C5 rows (per_config)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned as "
                    "DIR/<name>.npy (float32): every quantized weight tensor and a fixed sample of every activation site")
    return ap.parse_args()


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU through NVML while a timed region runs."""

    def __init__(self, index, period=0.02):
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None       # samples: (perf_counter, MHz, reason names)
        self.window = None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
        while not self._stop.is_set():
            try:
                mhz = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, [k for k, bit in names.items() if mask & bit]))
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        """Samples taken inside `window` = (t0, t1) of perf_counter (the timed region); the thread itself is started
        before the warm-up because the first NVML queries take tens of milliseconds and stall kernel launches."""
        lo, hi = self.window if self.window else (float("-inf"), float("inf"))
        inside = [(m, r) for t, m, r in self.samples if lo <= t <= hi]
        if not inside and self.samples:          # region shorter than one period: the sample closest to it
            t, m, r = min(self.samples, key=lambda smp: min(abs(smp[0] - lo), abs(smp[0] - hi)))
            inside = [(m, r)]
        mhz = sorted(m for m, _ in inside)
        reasons = sorted({k for _, r in inside for k in r})
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(mhz)}


# ------------------------------------------------------------------------------------------------- workload
def make_quantizers(Q, weights):
    """8-bit per-channel symmetric weight quantizers (threshold_c = max|w_c|) and one 8-bit uniform activation
    quantizer per site."""
    wq = []
    for w in weights:
        thr = w.detach().abs().flatten(1).amax(1).double().cpu().tolist()
        thr = [t if t > 0 else 1.0 for t in thr]
        wq.append(Q.WeightsSymmetricInferableQuantizer(8, thr, True, 0))
    return wq


REF_DIR = os.path.join(ROOT, "baseline", "_ref")      # pip install --no-deps --target baseline/_ref <reference> (git-ignored, travels with gpurun)


def load_reference():
    """The UNMODIFIED reference package (sony/mct_quantizers 1.6.0) from baseline/_ref, or None when it is not installed."""
    if not os.path.isdir(os.path.join(REF_DIR, "mct_quantizers")):
        return None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        import mct_quantizers
        if not os.path.abspath(mct_quantizers.__file__).startswith(REF_DIR):
            return None
        return mct_quantizers
    except Exception:
        return None


def build_reference_model(torch, batch, seed=1234):
    """BASELINE configs[1] on CPU tensors, built with the reference's own classes when baseline/_ref is importable
    (kind "reference"), else with oracle/torch_cpu_port.py, the reference's ATen call sites restated (kind "port").
    Returns (step, nelem, kind).  Activation ranges are the [min, max] of each tensor, as BASELINE.md C2 says."""
    import logging
    import warnings
    warnings.filterwarnings("ignore")
    g = torch.Generator().manual_seed(seed)
    weights = []
    for shp in MBV2_WEIGHTS:
        fan_out = shp[0] * numel(shp[2:])
        weights.append(torch.empty(shp).normal_(0, (2.0 / fan_out) ** 0.5, generator=g))
    acts = [torch.empty((batch,) + shp).normal_(0, 1, generator=g) for shp in MBV2_ACTS]
    nelem = sum(w.numel() for w in weights) + sum(x.numel() for x in acts)
    ref = load_reference()
    if ref is not None:
        logging.getLogger("MCT Quantizers").setLevel(logging.ERROR)
        from mct_quantizers import PytorchActivationQuantizationHolder, PytorchQuantizationWrapper, pytorch_quantizers as RQ
        wrappers = []
        for w in weights:
            thr = [t if t > 0 else 1.0 for t in w.abs().flatten(1).amax(1).double().tolist()]
            layer = torch.nn.Conv2d(1, 1, 1) if w.dim() == 4 else torch.nn.Linear(1, 1)
            layer.weight = torch.nn.Parameter(w)
            wrappers.append(PytorchQuantizationWrapper(layer, {'weight': RQ.WeightsSymmetricInferableQuantizer(8, thr, True, 0)}))
        holders = [PytorchActivationQuantizationHolder(RQ.ActivationUniformInferableQuantizer(8, [float(x.min())], [float(x.max())]))
                   for x in acts]

        def step():
            out = None
            for wr in wrappers:
                out = wr.get_quantized_weights()            # quantize_wrapper.py:262-270 -> quantizer(w) per weight
            for h, x in zip(holders, acts):
                out = h(x)                                  # activation_quantization_holder.py:43-53
            return out
        return step, nelem, "reference"
    from oracle import torch_cpu_port as port
    wparams = [port.weights_symmetric_qparams([t if t > 0 else 1.0 for t in w.abs().flatten(1).amax(1).double().tolist()], 8)[:2]
               for w in weights]
    aparams = [port.activation_uniform_qparams([float(x.min())], [float(x.max())], 8)[2:4] for x in acts]

    def step():
        out = None
        for w, (s_, z_) in zip(weights, wparams):
            out = port.affine_per_channel(w, s_, z_, 0, -128, 127)
        for x, (scale, zp) in zip(acts, aparams):
            out = port.affine_scalar_qparams(x, scale, zp, 0, 255)
        return out
    return step, nelem, "port"


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path -- the unmodified package from baseline/_ref
    through its public API (PytorchQuantizationWrapper.get_quantized_weights, PytorchActivationQuantizationHolder.__call__)
    on CPU tensors, all host threads, same workload as the B200 arm (53 + 53 tensors at --batch images).  The GPUs are
    hidden from this process: the reference creates its parameters on `cuda` whenever one is visible, and this arm times
    its CPU path."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    batch = args.batch
    try:
        import psutil
        while batch > 8 and numel((batch,) + (6679112,)) * 4 * 1.6 > psutil.virtual_memory().available:
            batch //= 2                                   # host RAM guard; the sample says what ran
    except Exception:
        pass
    step, nelem, kind = build_reference_model(torch, batch)
    with torch.no_grad():
        for _ in range(max(args.warmup, 1)):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        dt = (time.perf_counter() - t0) / args.steps
    gbs = nelem * BYTES_PER_ELEM / dt / 1e9
    sample = f"all 53 weight tensors + 53 activation sites at batch {batch} ({nelem} f32 elements per step)"
    what = ("unmodified sony/mct_quantizers 1.6.0 from baseline/_ref, public API" if kind == "reference"
            else "oracle/torch_cpu_port.py (baseline/_ref missing): the ATen ops the reference calls")
    line = {"impl": "reference", "metric": METRIC, "value": round(gbs, 3), "unit": "GB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": batch, "elements_per_step_per_gpu": nelem, "sample": sample,
                       "ranges": "ActivationUniform [min, max] of each tensor", "implementation": what,
                       "host": "CPU torch %s, %d threads" % (torch.__version__, cores)},
            "cpu_baseline": {"value": round(gbs, 3), "unit": "GB/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": round(gbs, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "elements_per_s": round(nelem / dt, 1)}
    print(json.dumps(line), flush=True)


def cpu_baseline_leg(args):
    """cpu_baseline of the B200 arm: the reference arm itself (a fresh process with the GPUs hidden), on a bounded sample."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--batch", str(args.ref_batch), "--steps", "5", "--warmup", "1"]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    for ln in reversed(out.stdout.strip().splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)["cpu_baseline"]
    raise RuntimeError("cpu_baseline leg failed: " + out.stderr[-400:])


def verify_against_oracle(torch, wplan, weights, wq, holders, acts, last, aplan):
    """After the timed region: windows of what the timed path produces (the last step's output, three more sites incl. the
    largest, two weight tensors of the multi-tensor launch) against the CPU oracle, bit for bit.  oracle/ is the checker
    only; a mismatch fails the run."""
    import numpy as np
    import oracle
    checked = 0

    def check_window(y, x, q, lo, hi, what):
        nonlocal checked
        xs = x.reshape(-1)[lo:hi].cpu().numpy()
        ys = y.reshape(-1)[lo:hi].cpu().numpy()
        want = oracle.fq_affine(xs, oracle.F32, np.array([q.scale], np.float64).astype(np.float32),
                                np.array([q.zero_point], np.int32), 1, 1, 0, 255)
        if not np.array_equal(ys.view(np.uint32), want.reshape(-1).view(np.uint32)):
            raise RuntimeError("bench output differs from the oracle: " + what)
        checked += hi - lo

    sites = sorted(range(len(acts)), key=lambda i: acts[i].numel())
    picked = [(len(acts) - 1, last)] + [(i, None) for i in (sites[-1], sites[len(sites) // 2], sites[0]) if i != len(acts) - 1]
    for i, y in picked:
        x, q = acts[i], holders[i].activation_holder_quantizer
        y = aplan.outputs_of(i) if y is None else y         # what the timed launch wrote for this site
        n = x.numel()
        w = min(n, 1 << 16)
        for lo in sorted({0, (n // 2) // 4096 * 4096, n - w}):
            check_window(y, x, q, lo, min(lo + w, n), f"activation site {i} [{lo}:{lo + w}]")
    if wplan is not None:
        outs = wplan.run()
        for k in sorted({0, len(weights) // 2, len(weights) - 1}):
            w, q = weights[k], wq[k]
            want = oracle.fq_affine(w.detach().cpu().numpy(), oracle.F32, q.scales.cpu().numpy().astype(np.float32),
                                    q.zero_points.cpu().numpy().astype(np.int32), w.shape[0], w[0].numel(), -128, 127)
            if not np.array_equal(outs[k].cpu().numpy().reshape(-1).view(np.uint32), want.reshape(-1).view(np.uint32)):
                raise RuntimeError(f"bench weight tensor {k} differs from the oracle")
            checked += w.numel()
    return {"ok": True, "elements_compared": int(checked), "against": "oracle/mctq_oracle.c (CPU restatement), bit-exact",
            "what": "3 windows of <= 65536 elements of 4 activation sites (incl. the last timed output and the largest site) + 3 weight tensors"}


DUMP_SAMPLE = 1 << 17      # elements written per activation site: 53 sites -> at most 27.8 MB, + 13.9 MB of weights


def dump_outputs(out_dir, layer_ids, weights_out, acts_out):
    """Writes the outputs of one step so that two builds can be compared array for array: weight_<layer>.npy, every
    quantized weight tensor whole; act_<site>.npy, the site's output whole if it has at most DUMP_SAMPLE elements, else
    DUMP_SAMPLE of its flat elements at indices drawn without replacement by numpy's default_rng(<site>), increasing."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for k, y in zip(layer_ids, weights_out):
        np.save(os.path.join(out_dir, f"weight_{k:02d}.npy"), y.to(torch.float32).cpu().numpy())
    for i, y in enumerate(acts_out):
        if y.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(i).choice(y.numel(), DUMP_SAMPLE, replace=False))
            y = y.reshape(-1)[torch.from_numpy(idx).to(y.device)]
        np.save(os.path.join(out_dir, f"act_{i:02d}.npy"), y.to(torch.float32).cpu().numpy())


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank, local_rank, world = dist_env()
    if world != args.gpus and world == 1 and args.gpus > 1:
        # not under torchrun: relaunch ourselves with one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path to fall back to)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import logging
    import mct_quantizers_b200 as mctq
    from mct_quantizers_b200 import _native, sharding
    logging.getLogger("MCT Quantizers B200").setLevel(logging.ERROR)     # 53 identical "range adjusted" notices
    from mct_quantizers_b200.pytorch import quantizers as Q
    from mct_quantizers_b200.pytorch.model_quantization import WeightPlan
    lib = _native.load()

    # ---- synthetic model state, generated on the device (seeded per rank)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    gw = torch.Generator(device=dev).manual_seed(1234)            # weights are the same model on every rank
    all_weights = []
    for shp in MBV2_WEIGHTS:
        fan_out = shp[0] * numel(shp[2:])
        all_weights.append(torch.empty(shp, device=dev).normal_(0, (2.0 / fan_out) ** 0.5, generator=gw))
    my_layers = sharding.shard_layers([w.numel() for w in all_weights], world)[rank]
    weights = [all_weights[i] for i in my_layers]
    wq = make_quantizers(Q, weights)
    wrappers = []
    for w, q in zip(weights, wq):
        layer = torch.nn.Conv2d(1, 1, 1) if w.dim() == 4 else torch.nn.Linear(1, 1)
        layer.weight = torch.nn.Parameter(w)
        wrappers.append(mctq.PytorchQuantizationWrapper(layer, {'weight': q}))
    triples = [tv for wr in wrappers for tv in wr.get_weights_vars()]
    wplan = WeightPlan(triples) if triples else None

    acts = [torch.empty((args.batch,) + shp, device=dev).normal_(0, 1, generator=g) for shp in MBV2_ACTS]
    ranges = [(float(x.min()), float(x.max())) for x in acts]        # BASELINE C2: [min, max] of the tensor
    holders = [mctq.PytorchActivationQuantizationHolder(Q.ActivationUniformInferableQuantizer(8, [lo], [hi])).to(dev)
               for lo, hi in ranges]
    n_w = sum(w.numel() for w in weights)
    n_a = sum(x.numel() for x in acts)
    n_sites = len(acts)
    bytes_step = (n_w + n_a) * BYTES_PER_ELEM

    # every activation site's input exists up front in this workload, so the sites run as ONE launch (ActivationPlan ->
    # mctq_fq_affine_scalar_multi), like the weights (WeightPlan -> mctq_fq_affine_multi): 2 launches per step.  The same
    # step as 53 holder calls (one launch each) is timed after it and reported as `per_call`.
    aplan = mctq.ActivationPlan(list(zip(holders, acts)))
    assert not aplan.other and len(aplan._plans) == 1

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    step_outputs = {"weights": [], "acts": []}        # what the latest step() returned (plan-owned buffers, no copies)

    def step():
        if wplan is not None:
            step_outputs["weights"] = wplan.run()
        step_outputs["acts"] = aplan.run()
        return step_outputs["acts"][-1]

    def step_per_call():
        if wplan is not None:
            wplan.run()
        out = None
        for h, x in zip(holders, acts):
            out = h(x)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(torch.cuda.current_device() if os.environ.get("CUDA_VISIBLE_DEVICES") is None else local_rank)
    sampler.__enter__()
    n_warm = 0
    last = None
    for _ in range(max(args.warmup, 3)):
        last = step()          # same object lifetimes as the timed loop: `last` keeps one output alive across a step, and a
        n_warm += 1            # first-time cudaMalloc by the caching allocator inside the timed region costs 3-126 ms
    # keep warming (untimed) the way the timed region runs -- back-to-back steps, no host sync in between -- for ~0.5 s:
    # clocks settle under the power cap and every allocator / driver first-time cost is paid here
    torch.cuda.synchronize()
    t_settle = time.perf_counter()
    prev_ev = None
    while time.perf_counter() - t_settle < 0.5:
        for _ in range(10):
            last = step()
            n_warm += 1
        ev_s = ev()
        ev_s.record()
        if prev_ev is not None:
            prev_ev.synchronize()            # bound the launch queue without draining it: wait for the batch BEFORE this one
        prev_ev = ev_s
    barrier()
    # duration of the weights launch alone (one multi-tensor kernel, ~1 % of a step), measured here so that no event has
    # to be recorded in the middle of a timed step
    w_ms = 0.0
    if wplan is not None:
        wa, wb = ev(), ev()
        reps_w = 6
        wplan.run()
        big = max(range(len(acts)), key=lambda i: acts[i].numel())
        keep = [holders[big](acts[big]) for _ in range(8)]          # ~2.8 ms of queued GPU work: the host runs ahead, so the
        wa.record()                                                  # events bracket back-to-back kernels, not host time
        for _ in range(reps_w):
            wplan.run()
        wb.record()
        wb.synchronize()
        w_ms = wa.elapsed_time(wb) / reps_w
        del keep
    launches0 = lib.mctq_launch_count()
    e0, e1 = ev(), ev()
    step_ev = [ev() for _ in range(args.steps + 1)]
    # torch creates the underlying cudaEvent lazily at the first record(): create them all before the timed region
    for e in [e0, e1] + step_ev:
        e.record()
    import gc
    gc.collect()
    gc.disable()                         # no interpreter-heap collection inside the timed loop
    barrier()
    if args.profiler_range:              # ncu --profile-from-start off captures exactly the timed region
        torch.cuda.profiler.start()
    t_region0 = time.perf_counter()
    e0.record()
    step_ev[0].record()
    cpu_t = [time.perf_counter()]
    for k in range(args.steps):
        last = step()
        step_ev[k + 1].record()
        cpu_t.append(time.perf_counter())
    e1.record()
    barrier()
    gc.enable()
    sampler.window = (t_region0, time.perf_counter())
    if args.profiler_range:
        torch.cuda.profiler.stop()
    sampler.__exit__()
    launches = lib.mctq_launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    per_step = [step_ev[k].elapsed_time(step_ev[k + 1]) for k in range(args.steps)]
    act_ms = ms_total - w_ms * args.steps        # the 53 activation launches of every step
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    tot_bytes = torch.tensor([float(bytes_step)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot_bytes, op=dist.ReduceOp.SUM)
    ms_step = t.item() / args.steps
    value = tot_bytes.item() / (ms_step * 1e-3) / 1e9
    clocks = sampler.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, my_layers, step_outputs["weights"], step_outputs["acts"])

    # ---- the same step as per-holder calls (53 + 1 launches), same timing rules
    torch.cuda.synchronize()
    for _ in range(3):
        last_pc = step_per_call()
    barrier()
    pc0, pc1 = ev(), ev()
    pc0.record()
    pc_l0 = lib.mctq_launch_count()
    for _ in range(args.steps):
        last_pc = step_per_call()
    pc1.record()
    barrier()
    pc_launches = lib.mctq_launch_count() - pc_l0
    tpc = torch.tensor([pc0.elapsed_time(pc1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tpc, op=dist.ReduceOp.MAX)
    pc_ms = tpc.item() / args.steps
    if sharding.checksum64(last_pc) != sharding.checksum64(last):
        raise RuntimeError("one-launch ActivationPlan result differs from the per-holder result")
    per_call = {"value": round(tot_bytes.item() / (pc_ms * 1e-3) / 1e9, 2), "unit": "GB/s", "ms_per_step": round(pc_ms, 4),
                "gpu_launches": int(pc_launches), "pct_of_8TBs": round(100 * tot_bytes.item() / (pc_ms * 1e-3) / 1e9 / world / 8000.0, 2),
                "what": "the same step as 53 PytorchActivationQuantizationHolder calls (one launch each, programmatic dependent launch) "
                        "+ the weights launch"}
    # ... and inside `with private_stream():` (opt-in early order: these inputs exist before the step starts)
    with mctq.private_stream():
        for _ in range(3):
            last_pc = step_per_call()
        barrier()
        pp0, pp1 = ev(), ev()
        pp0.record()
        for _ in range(args.steps):
            last_pc = step_per_call()
        pp1.record()
        barrier()
    tpp = torch.tensor([pp0.elapsed_time(pp1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tpp, op=dist.ReduceOp.MAX)
    per_call["private_stream_value"] = round(tot_bytes.item() / (tpp.item() / args.steps * 1e-3) / 1e9, 2)
    if sharding.checksum64(last_pc) != sharding.checksum64(last):
        raise RuntimeError("private_stream() result differs")
    del last_pc

    # ---- verification outside the timed region: checksums gathered with NCCL (no data-path collective)
    chk = torch.tensor([sharding.checksum64(last)], device=dev, dtype=torch.int64)
    if world > 1:
        gathered = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(gathered, chk)
        checks = [int(c.item()) for c in gathered]
    else:
        checks = [int(chk.item())]

    # ---- parity outside the timed region: windows of the timed path's outputs against the CPU oracle (the checker)
    oracle_check = verify_against_oracle(torch, wplan, weights, wq, holders, acts, last, aplan) if rank == 0 else None

    # ---- e2e: same step through the public API with HOST (pinned) tensors: H2D + kernel + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        import psutil
        need = n_a * 4 * 2.2 * (world if world > 1 else 1)
        e2e_batch = args.batch
        while need > psutil.virtual_memory().available * 0.5 and e2e_batch > 8:
            e2e_batch //= 2
            need /= 2
        host_acts = []
        for x in acts:
            hx = torch.empty((e2e_batch,) + tuple(x.shape[1:]), dtype=x.dtype, pin_memory=True)
            hx.copy_(x[:e2e_batch])
            host_acts.append(hx)
        host_w = [w.detach().cpu().pin_memory() for w in weights]
        n_e2e = sum(h.numel() for h in host_acts) + sum(h.numel() for h in host_w)

        def e2e_calls():
            res = None
            for hw_, q in zip(host_w, wq):
                res = q(hw_)
            for h, hx in zip(holders, host_acts):
                res = h(hx)
            return res

        def e2e_step():
            # the model's 106 quantizer / holder calls inside one host_pipeline() block: each call only enqueues its
            # H2D / kernel / D2H chunks, every result is complete in host memory when the block exits
            with mctq.host_pipeline():
                res = e2e_calls()
            return res

        def time_e2e(fn):
            fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                r = fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / args.e2e_steps, r

        dt_sync, res_sync = time_e2e(e2e_calls)          # every call returns a finished host tensor (pipeline drains per call)
        dt, res = time_e2e(e2e_step)
        if sharding.checksum64(res) != sharding.checksum64(res_sync):
            raise RuntimeError("host_pipeline() result differs from the per-call result")
        td = torch.tensor([dt], device=dev, dtype=torch.float64)
        nb = torch.tensor([float(n_e2e * BYTES_PER_ELEM)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
            dist.all_reduce(nb, op=dist.ReduceOp.SUM)
        e2e = {"value": round(nb.item() / td.item() / 1e9, 3), "unit": "GB/s", "h2d_bytes_per_step": int(nb.item()) // 2,
               "d2h_bytes_per_step": int(nb.item()) // 2, "steps": args.e2e_steps, "ms_per_step": round(td.item() * 1e3, 3),
               "batch_per_gpu": e2e_batch,
               "per_call_sync_value": round(n_e2e * BYTES_PER_ELEM / dt_sync / 1e9, 3),
               "path": "with host_pipeline(): quantizer(cpu_pinned_tensor) x 106 -> mctq_fq_affine_host: chunked H2D / kernel / "
                       "D2H on 3 streams, one wait at block exit (per_call_sync_value: the same calls outside the block, this rank)"}
        # the host link's own ceiling, measured the same way on every rank at once: pinned H2D and D2H copies running together
        # (what the e2e value can reach at most, in algorithmic bytes: one byte up + one byte down per 2 algorithmic bytes)
        probe_n = min(128 << 20, host_acts[3].numel())
        p_in, p_out = host_acts[3].reshape(-1)[:probe_n], torch.empty(probe_n, dtype=torch.float32, pin_memory=True)
        d_a, d_b = torch.empty(probe_n, device=dev), torch.empty(probe_n, device=dev)
        sa, sb = torch.cuda.Stream(), torch.cuda.Stream()

        def link_both():
            with torch.cuda.stream(sa):
                d_a.copy_(p_in, non_blocking=True)
            with torch.cuda.stream(sb):
                p_out.copy_(d_b, non_blocking=True)
        link_both()
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            link_both()
        torch.cuda.synchronize()
        tl = torch.tensor([(time.perf_counter() - t0) / 3], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        link_gbs = 2 * p_in.numel() * 4 * world / tl.item() / 1e9
        e2e["host_link_ceiling"] = round(link_gbs, 1)
        e2e["frac_of_host_link"] = round(e2e["value"] / link_gbs, 3)
        e2e["host_link_how"] = "pinned H2D + D2H copies of 512 MB running together on every rank, aggregate GB/s (max over ranks)"
        del p_out, d_a, d_b
        # the host-buffer path must give the device path's bits (same inputs: host_acts are copies of acts)
        if sharding.checksum64(res) != sharding.checksum64(last[:e2e_batch]):
            raise RuntimeError("e2e (host-buffer) result differs from the device-resident result")
        del host_acts, host_w

    # ---- the other BASELINE configs (C1 / C3 / C4 / C5), strong scaling at N > 1: tools/scale_bench.py, all ranks take part
    per_config = None
    if not args.no_per_config:
        del acts, holders, last, aplan
        torch.cuda.empty_cache()
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import scale_bench
        rows, _ = scale_bench.run_configs(dev, rank, world, reps=5, max_gb=16.0, log=sys.stderr)
        per_config = [{"config": r["config"], "scaling": r.get("scaling"), "kernel": r.get("kernel"), "ms": r["ms"], "GBs": r["GBs"],
                       "GBs_per_gpu": r["GBs_per_gpu"], "pct_of_8TBs": r["pct_of_8TBs_per_gpu"],
                       "frac_of_copy_peak": r["frac_of_copy_peak_per_gpu"]} for r in rows if "GBs" in r]

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        achieved = n_a * BYTES_PER_ELEM / (act_ms / args.steps * 1e-3) / 1e9
        # dram bytes per launch of the dominant kernel: from the committed ncu capture of this same command
        # (profiles/r01_bench_traffic.json, made by tools/ncu_summary.py traffic); only valid for the default batch
        traffic, traffic_src, kname = None, None, None
        try:
            if args.batch == 256:
                import glob
                cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_bench_traffic.json")))
                with open(cands[-1]) as f:                       # the newest round's capture
                    for k, v in json.load(f).items():
                        if k.startswith("fq_affine_sites_kernel"):
                            traffic = int(v["dram_bytes_per_launch"])
                            kname = k
                            traffic_src = ("profiles/%s (ncu dram__bytes_read.sum + dram__bytes_write.sum of the one launch "
                                           "of a step)" % os.path.basename(cands[-1]))
        except Exception:
            pass
        line = {"metric": METRIC, "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "warmup_steps_run": n_warm, "ms_per_step": round(ms_step, 4),
                "step_ms": {"min": round(min(per_step), 4), "median": round(sorted(per_step)[len(per_step) // 2], 4),
                            "max": round(max(per_step), 4), "first": [round(v, 4) for v in per_step[:3]],
                            "cpu_launch_ms_first": [round((b - a) * 1e3, 3) for a, b in zip(cpu_t[:6], cpu_t[1:7])],
                            "cpu_launch_ms_max": round(max(b - a for a, b in zip(cpu_t, cpu_t[1:])) * 1e3, 3)}, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "batch_per_gpu": args.batch, "elements_per_step_per_gpu": n_w + n_a,
                           "bytes_per_element": BYTES_PER_ELEM, "l2": "inputs larger than L2 (6.8 GB read + 6.8 GB written per step)",
                           "ranges": "ActivationUniform [min, max] of each tensor",
                           "sharding": "activations by batch, weights by layer; no collective on the data path"},
                "elements_per_s": round(value * 1e9 / BYTES_PER_ELEM, 1),
                "pct_of_8TBs": round(100 * value / world / 8000.0, 2),
                "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                             "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                             "kernel": "fq_affine_sites_kernel (all 53 ActivationUniform sites in one grid: per-tensor body of fq_affine_kernel<T, CH_PT>, "
                                       "8 KB tiles, site table in kernel parameters)",
                             "launches_per_step": 1,
                             "avg_launch_us": round(act_ms / args.steps * 1e3, 2),
                             "how": "CUDA events around every timed step minus the weights launch (%.1f us, timed separately)" % (w_ms * 1e3),
                             "algorithmic_bytes_per_launch": int(n_a * BYTES_PER_ELEM), "sites_per_launch": n_sites},
                "clocks": clocks, "gpu_launches": int(launches), "per_call": per_call, "checksums": checks}
        if e2e is not None:
            line["e2e"] = e2e
        line["oracle_check"] = oracle_check
        if per_config is not None:
            line["per_config"] = per_config
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_leg(args)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
