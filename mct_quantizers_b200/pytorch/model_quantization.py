"""Whole-model weight quantization in one launch (SURVEY 8f rank 1).

The reference re-quantizes each wrapped weight with its own kernel(s) on every forward
(mct_quantizers/pytorch/quantize_wrapper.py:228-240): 53 launches (+ 106 host syncs) for MobileNetV2.  Here all
affine weight quantizers of a model are gathered into one descriptor table and run as ONE kernel
(mctq_fq_affine_multi), all LUT weight quantizers as a second one (mctq_fq_lut_prepared_multi) and all packed weights
(packed_weights.py) as a third (mctq_unpack_multi); user-defined quantizers and tensors outside the prepared paths keep
their own call."""
from typing import Dict, List

import torch

from mct_quantizers_b200.ops import MultiTensorPlan, LutMultiPlan, ScalarSitesPlan, UnpackPlan
from mct_quantizers_b200.pytorch.packed_weights import PackedWeight


def _is_affine_weight_quantizer(q) -> bool:
    from mct_quantizers_b200.pytorch.quantizers import WeightsSymmetricInferableQuantizer, WeightsUniformInferableQuantizer
    return isinstance(q, (WeightsSymmetricInferableQuantizer, WeightsUniformInferableQuantizer)) and not q._use_custom_impl


def _lut_item(q, w):
    """LutMultiPlan item of a LUT weight quantizer (WeightsLUTSymmetric / WeightsLUTPOT), or None."""
    from mct_quantizers_b200.pytorch.quantizers import WeightsLUTSymmetricInferableQuantizer
    from mct_quantizers_b200.pytorch.quantizer_utils import lut_search_table
    if not isinstance(q, WeightsLUTSymmetricInferableQuantizer) or q._use_custom_impl or not w.is_cuda:
        return None
    if q.per_channel and q.input_rank is not None and q.input_rank != w.dim():
        return None                                   # the per-layer call raises the reference's error
    if q.__dict__.get('_search_table') is None:
        q._search_table = lut_search_table(q._lut_values_np, q.lut_values_bitwidth, True)
    thr, = q._on(w.device, q._threshold_torch)
    thr = thr.reshape(-1)
    item = (w.detach(), q._search_table, int(q._lut_values_torch.numel()), thr, bool(q.per_channel),
            int(q.channel_axis) if q.per_channel else 0, float(q.eps))
    return item if LutMultiPlan.accepts(item) else None


def plan_for(weight_vars) -> "WeightPlan":
    return WeightPlan(weight_vars)


_PARAM_NAMES = ('scales', 'zero_points', '_threshold_torch')


def _plan_watch(qs):
    """(quantizer, attribute) pairs whose identity and (parameter tensors that track one) in-place version a plan must watch."""
    attrs, versioned = [], []
    for q in qs:
        d = getattr(q, '__dict__', {})
        for name in _PARAM_NAMES:
            t = d.get(name)
            if isinstance(t, torch.Tensor):
                attrs.append((d, name))
                if not t.is_inference():
                    versioned.append(t)
    return attrs, versioned


def _live_signature(ws, attrs, versioned, qs):
    """What a plan captured of its (weight, quantizer) pairs: storage, placement and layout of every weight; identity and
    in-place version of the quantizers' parameter tensors; the reuse flags.  A plan whose signature no longer matches the
    live objects (model.to(), .half(), load_state_dict into new storage, a re-assigned parameter, edited thresholds) is
    rebuilt.  Flat comprehensions over pre-resolved objects: < 1 us per tensor."""
    return ([(w.data_ptr(), w.dtype, w.shape, w.stride()) for w in ws],
            [id(d.get(name)) for d, name in attrs],
            [t._version for t in versioned],
            [getattr(q, 'enable_reuse', False) for q in qs])


class WeightPlan:
    """Launch plan over (name, weight, quantizer) triples: one multi-tensor launch per quantizer family and device.
    Output buffers are kept and refreshed by run().

    The plan captures raw pointers, so run() first compares every triple's live signature (storage pointer, device, dtype,
    shape, strides, parameter tensors) with what was captured and REBUILDS when anything moved -- after `model.to()`,
    `.half()` or a re-assigned parameter the stale storage is never quantized.  Tensors a multi-tensor launch cannot take
    (non-dense views, CPU tensors, user-defined quantizers, uniform quantizers whose zero point leaves the range: the
    per-layer call raises the reference's error) go through their quantizer's own `__call__`, which also owns the
    reuse contract (`enable_reuse` / `resue_outputs`).

    Packed weights (a PackedWeight in the weight slot) are the third family: all of a device are rebuilt by one UnpackPlan
    into plan-owned outputs, so a plan holds every rebuilt weight at once -- one launch instead of one per wrapper, at the
    cost of the memory saving that packing gives a per-wrapper forward."""

    def __init__(self, weight_vars):
        self.vars = [(name, w, q) for name, w, q in weight_vars]
        self.names = [name for name, _, _ in self.vars]
        self.n = len(self.vars)
        self._build()

    def _build(self):
        self.fused_idx, self.lut_idx, self.packed_idx, self.other = [], [], [], []
        self._plans, self._lut_plans, self._unpack_plans = [], [], []     # [(indices, plan)] per device
        by_dev, lut_by_dev, packed_by_dev = {}, {}, {}
        for k, (name, w, q) in enumerate(self.vars):
            if isinstance(w, PackedWeight):
                idx, items = packed_by_dev.setdefault(w.device, ([], []))
                idx.append(k)
                items.append(w.plan_item())
                self.packed_idx.append(k)
                continue
            ok_dtype = w.is_cuda and w.dtype in (torch.float32, torch.bfloat16, torch.float16) and w.numel() > 0
            reuse = bool(q.__dict__.get('enable_reuse', False))
            item = None
            if ok_dtype and not reuse and _is_affine_weight_quantizer(q) and not q.__dict__.get('_zero_point_out_of_range', False):
                scales, zps = q._on(w.device, q.scales, q.zero_points)
                item = (w.detach(), scales.flatten(), zps.flatten(), q.channel_axis if q.per_channel else None,
                        q.min_quantized_domain, q.max_quantized_domain)
                if MultiTensorPlan.accepts(item):
                    w.requires_grad = False
                    by_dev.setdefault(w.device, ([], []))
                    by_dev[w.device][0].append(k)
                    by_dev[w.device][1].append(item)
                    self.fused_idx.append(k)
                    continue
            lut_item = _lut_item(q, w) if ok_dtype and not reuse else None
            if lut_item is not None:
                w.requires_grad = False
                lut_by_dev.setdefault(w.device, ([], []))
                lut_by_dev[w.device][0].append(k)
                lut_by_dev[w.device][1].append(lut_item)
                self.lut_idx.append(k)
            else:
                self.other.append((k, w, q))
        for dev, (idx, items) in by_dev.items():
            self._plans.append((idx, MultiTensorPlan(items)))
        for dev, (idx, items) in lut_by_dev.items():
            self._lut_plans.append((idx, LutMultiPlan(items)))
        for dev, (idx, items) in packed_by_dev.items():
            self._unpack_plans.append((idx, UnpackPlan(items)))
        self._ws = [w for _, w, _ in self.vars]
        self._qs = [q for _, _, q in self.vars]
        self._attrs, self._versioned = _plan_watch(self._qs)
        self._sigs = _live_signature(self._ws, self._attrs, self._versioned, self._qs)

    # first plan of each family (single-device models: the only one)
    @property
    def plan(self):
        return self._plans[0][1] if self._plans else None

    @property
    def lut_plan(self):
        return self._lut_plans[0][1] if self._lut_plans else None

    def stale(self) -> bool:
        return _live_signature(self._ws, self._attrs, self._versioned, self._qs) != self._sigs

    def run(self, validate: bool = True) -> List[torch.Tensor]:
        """`validate=False` skips the staleness check (for callers that own the weights and know nothing moved)."""
        if validate and self.stale():
            self._build()
        out = [None] * self.n
        for idx, plan in self._plans:
            for k, y in zip(idx, plan.run()):
                out[k] = y
        for idx, plan in self._lut_plans:
            for k, y in zip(idx, plan.run()):
                out[k] = y
        for idx, plan in self._unpack_plans:
            for k, y in zip(idx, plan.run()):
                out[k] = y
        for k, w, q in self.other:
            out[k] = q(w)
        return out


class ActivationPlan:
    """Launch plan over (holder or activation quantizer, tensor) pairs whose inputs ALREADY EXIST: every per-tensor affine
    site (ActivationSymmetric / POT / Uniform) of a device runs in ONE launch (`ScalarSitesPlan`), any other quantizer
    (LUT, user-defined), CPU tensor or non-dense view through its own call.  Use it where a model's activations are
    available together -- calibration / analysis passes over recorded activations, batched post-processing, benchmarks;
    inside a forward pass each holder still sees its input only after the producing layer ran, so holders keep their
    per-call path there (or are fused into their producer, fused_activation_holder.py).

        plan = ActivationPlan([(holder_k, x_k) for k in sites])
        ys = plan.run()            # output buffers are owned by the plan and refreshed by every run()

    run() revalidates what the plan captured (storage pointer, dtype, shape, strides of every input; scale / zero point /
    range of every quantizer) and rebuilds on any difference.  Results are bit-identical to `holder(x)`."""

    def __init__(self, pairs):
        self.pairs = [(getattr(h, 'activation_holder_quantizer', h), x) for h, x in pairs]
        self.n = len(self.pairs)
        self._build()

    @staticmethod
    def _params(q):
        from mct_quantizers_b200.pytorch.fused_activation_holder import affine_scalar_params
        if q.__dict__.get('_use_custom_impl', False) and torch.jit.is_tracing():
            return None
        return affine_scalar_params(q)

    def _sig(self):
        return [(x.data_ptr(), x.dtype, x.shape, x.stride(), self._params(q)) for q, x in self.pairs]

    def _build(self):
        self._plans, self.other = [], []
        by_dev = {}
        for k, (q, x) in enumerate(self.pairs):
            prm = self._params(q)
            if prm is not None and ScalarSitesPlan.accepts(x):
                idx, items = by_dev.setdefault(x.device, ([], []))
                idx.append(k)
                items.append((x.detach(), prm[0], prm[1], prm[2], prm[3]))
            else:
                self.other.append((k, q, x))
        for dev, (idx, items) in by_dev.items():
            self._plans.append((idx, ScalarSitesPlan(items)))
        self._sigs = self._sig()

    def run(self) -> List[torch.Tensor]:
        if self._sig() != self._sigs:
            self._build()
        out = [None] * self.n
        for idx, plan in self._plans:
            for k, y in zip(idx, plan.run()):
                out[k] = y
        for k, q, x in self.other:
            out[k] = q(x)
        return out

    def outputs_of(self, k: int) -> torch.Tensor:
        """The plan-owned output buffer of pair `k` as the last run() left it (None for pairs outside the fused launch)."""
        for idx, plan in self._plans:
            if k in idx:
                return plan.outputs[idx.index(k)]
        return None


def quantize_activations(pairs) -> List[torch.Tensor]:
    """[holder_k(x_k)] for (holder or quantizer, tensor) pairs, per-tensor affine sites in one launch per device."""
    return ActivationPlan(pairs).run()


def _wrapper_weight_vars(mod):
    """(name, weight, quantizer) of a wrapper's float weights, then (name, PackedWeight, quantizer) of its packed ones."""
    packed = mod.__dict__.get('_packed')
    return list(mod.get_weights_vars()) + (packed.weight_vars(mod) if packed is not None else [])


def quantize_weight_vars(weight_vars) -> Dict[str, torch.Tensor]:
    plan = WeightPlan(weight_vars)
    return dict(zip(plan.names, plan.run()))


def quantize_model_weights(model: torch.nn.Module) -> Dict[str, Dict[str, torch.Tensor]]:
    """{wrapper module name: {weight name: quantized weight}} for every PytorchQuantizationWrapper in `model`,
    all affine quantizers of the whole model in one kernel launch."""
    from mct_quantizers_b200.pytorch.quantize_wrapper import PytorchQuantizationWrapper
    triples, owners = [], []
    for mod_name, mod in model.named_modules():
        if isinstance(mod, PytorchQuantizationWrapper):
            for name, w, q in _wrapper_weight_vars(mod):
                triples.append((name, w, q))
                owners.append(mod_name)
    result: Dict[str, Dict[str, torch.Tensor]] = {}
    if not triples:
        return result
    plan = WeightPlan(triples)
    for owner, name, y in zip(owners, plan.names, plan.run()):
        result.setdefault(owner, {})[name] = y
    return result


class ModelWeightPlan:
    """Whole-model weight quantization hoisted out of the per-layer forward (SURVEY 8f rank 1).

    The reference re-quantizes every wrapped weight inside every `PytorchQuantizationWrapper.forward`
    (mct_quantizers/pytorch/quantize_wrapper.py:228-240).  A plan gathers the weights of ALL wrappers of a model,
    quantizes them with one multi-tensor launch (`refresh()`), installs the results in the wrapped layers and tells the
    wrappers to skip their own quantization while the plan is active:

        plan = plan_model_weights(model)      # builds the descriptor table once, output buffers are reused
        with plan:                            # refresh(): ONE kernel for every affine weight quantizer of the model
            y = model(x)                      # wrappers run their layers on the installed weights, no per-layer launches

    or, for inference with constant weights, `plan.enable()` once (and `plan.refresh()` again only if the float weights
    change).  Results are identical to the per-layer path (same kernels' arithmetic, checked by tests).  Packed weights
    (packed_weights.py) are rebuilt by one unpack launch per device and stay installed while the plan is enabled: the
    plan holds every rebuilt weight of the model at once.  Wrappers in fused linear mode are not part of the plan."""

    def __init__(self, model: torch.nn.Module):
        from mct_quantizers_b200.pytorch.quantize_wrapper import PytorchQuantizationWrapper
        # wrappers in fused linear mode (packed_weights.py) are left out: rebuilding their weights is what the mode avoids
        self.wrappers = [mod for mod in model.modules()
                         if isinstance(mod, PytorchQuantizationWrapper) and mod.is_weights_quantization
                         and not getattr(mod.__dict__.get('_packed'), 'fused', False)]
        self.plan = None
        self._collect()
        self.active = False

    def _collect(self):
        """(Re)build the plan from the wrappers' CURRENT weight variables."""
        triples, self._owner = [], []
        for mod in self.wrappers:
            for name, w, q in _wrapper_weight_vars(mod):
                triples.append((name, w, q))
                self._owner.append(mod)
        self._ids = [(id(w), id(q)) for _, w, q in triples]
        self.plan = WeightPlan(triples) if triples else None

    def refresh(self):
        """Quantize every weight (one launch per quantizer family and device) and install the results.  The wrappers'
        weight variables are looked at again on every refresh: re-assigned parameters or quantizers rebuild the plan, moved
        / converted storage (`model.to()`, `.half()`) is caught by WeightPlan's signature check."""
        if self.plan is None:
            return
        live = [(id(w), id(q)) for mod in self.wrappers for _, w, q in _wrapper_weight_vars(mod)]
        if live != self._ids:
            self._collect()
        per_wrapper = {}
        for owner, name, y in zip(self._owner, self.plan.names, self.plan.run()):
            per_wrapper.setdefault(id(owner), (owner, {}))[1][name] = y
        for owner, weights in per_wrapper.values():
            owner.set_quantize_weights(weights)

    def enable(self):
        self.refresh()
        for w in self.wrappers:
            w._prequantized = True
        self.active = True
        return self

    def disable(self):
        for w in self.wrappers:
            w._prequantized = False
        self.active = False

    def __enter__(self):
        return self.enable()

    def __exit__(self, *exc):
        self.disable()


def plan_model_weights(model: torch.nn.Module) -> ModelWeightPlan:
    return ModelWeightPlan(model)
