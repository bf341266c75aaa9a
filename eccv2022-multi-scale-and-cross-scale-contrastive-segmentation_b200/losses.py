"""Drop-in replacements of the reference loss classes, same names, constructor keys and call.

  DenseContrastiveLossV2      <- losses/DenseContrastiveLossV2.py:11-206
  DenseContrastiveLossV2_ms   <- losses/DenseContrastiveLossV2_ms.py:12-161

They are dispatched by class name from the reference's ``LossWrapper`` (LossWrapper.py:33,68-71),
which calls ``module(labels, deep_features)``; ``install_into_reference()`` registers them there.
All computation happens in libmscs.so (see _ops.py); these classes only resolve the config keys
exactly as the reference constructors do and expose the attributes its logger reads
(``ms_losses``, ``cs_losses``, ``cross_scale_contrast``, ``log_this_step``).
"""
import sys

import torch
import torch.nn as nn

from . import _ops
from ._ops import GRAPH_CALL_BASE, CompactLabels, LossSpec, MsCsContrastiveFn
from .datasets import class_facts


def _spec_from_config(config, scales, weights, ms=False):
    """Key rules of V2.py:12-31 and _ms.py:13-31 (defaults included)."""
    n_all, _n_real, _ignore = class_facts(config["dataset"], config["experiment"])
    n_all = int(config.get("num_all_classes", n_all))        # explicit override (not a reference key)
    temperature = config["temperature"] if "temperature" in config else 0.5              # V2.py:19
    # _ms.py:28: config['temperature'] unless the key cross_scale_temperature exists -> 0.1 (hard-coded)
    # -- and a KeyError when neither key is present, like the reference
    if ms:
        cs_temperature = config["temperature"] if "cross_scale_temperature" not in config else 0.1
    else:
        cs_temperature = temperature
    return LossSpec(
        num_classes=n_all, temperature=float(temperature), cs_temperature=float(cs_temperature),
        min_views=int(config.get("min_views_per_class", 5)),                             # V2.py:21
        max_views=int(config.get("max_views_per_class", 2500)),                          # V2.py:27
        max_total=int(config.get("max_features_total", 10000)),                          # V2.py:28
        weights=[float(w) for w in weights],
        cross_scale=bool(config.get("cross_scale_contrast", False)),                     # V2.py:23, _ms.py:27
        detach_deepest=bool(config.get("detach_deepest", False)),                        # _ms.py:29
        w_high_low=float(config.get("w_high_low", 1.0)), w_high_mid=float(config.get("w_high_mid", 1.0)),
        sampler=_sampler_key(config), seed=int(config.get("sampler_seed", 0)))


def _sampler_key(config):
    """``sampler`` is NOT a reference key: "reference" (default) consumes the torch CPU generator exactly like the
    reference's ``torch.randperm`` calls (V2.py:121); "philox" draws the permutations from a counter-based stream keyed
    by (``sampler_seed``, call index of the module) and leaves the torch generator alone."""
    s = str(config.get("sampler", "reference"))
    if s not in ("reference", "philox"):
        raise ValueError(f"sampler must be 'reference' or 'philox', got {s!r}")
    return s


def _philox_key(module, holder, dev):
    """Call index of the counter-based stream.  Eager calls use the host counter ``_sampler_calls`` (0, 1, ...).  A call
    captured into a CUDA graph uses the module's int64 device counter instead (``graph_call_index``, created at the
    first call on a device with the value 2**62): every replay reads it and increments it on the device, so replays
    draw from the call indices 2**62, 2**62 + 1, ..., which eager calls never reach, and leave the host counter alone."""
    if module._spec.sampler != "philox":
        return
    if dev.type == "cuda" and torch.cuda.is_current_stream_capturing():
        holder["philox"] = (module._spec.seed, module._graph_counter)       # (None: refused by _ops.graph_mode)
        return
    if dev.type == "cuda" and (module._graph_counter is None or module._graph_counter.device != dev):
        module._graph_counter = torch.full((), GRAPH_CALL_BASE, dtype=torch.int64, device=dev)
    holder["philox"] = (module._spec.seed, module._sampler_calls)
    module._sampler_calls += 1


class _GraphReadout:
    """What the loss classes share for CUDA graphs (INTEGRATION.md, "CUDA graphs"): the device call counter and the
    readout of a captured call's results after a replay."""
    _graph_counter = None

    @property
    def graph_call_index(self):
        """0-d int64 CUDA tensor: the Philox call index the next replay of a captured call draws from (None before the
        first call).  Assigning copies the value in place, so graphs already captured see it (checkpoint restore)."""
        return self._graph_counter

    @graph_call_index.setter
    def graph_call_index(self, value):
        if self._graph_counter is None:
            raise RuntimeError("graph_call_index exists after the module's first call on a GPU")
        self._graph_counter.copy_(torch.as_tensor(value, dtype=torch.int64))

    def fetch_samples(self, state=None):
        """ScaleSample list of the last call (``state``: of that call's state instead, e.g. a captured one).  For a
        captured call, read from the device plan records of its latest replay (one synchronisation); it raises the
        reference's exception when that replay's sampling failed."""
        st = self.last_state if state is None else state
        if not getattr(st, "graph", False):
            return st.samples
        _scalars, plan = _ops.fetch_graph_plan(st)
        _ops._raise_plan_errors(plan, st.sp.S, st.sp.spec)
        return _ops.graph_samples(st, plan)


class DenseContrastiveLossV2(_GraphReadout, nn.Module):
    """Single-scale dense supervised contrastive loss.  ``forward(label, features)`` (argument
    order as in the reference, V2.py:44); returns the loss, or -- when ``cross_scale_contrast`` --
    the reference's 4-tuple ``(loss, sampled_features (T,C,V), sampled_labels (T,), False)``."""

    def __init__(self, config):
        super().__init__()
        self.experiment = config["experiment"]
        self.dataset = config["dataset"]
        self.num_all_classes, self.num_real_classes, self.ignore_class = class_facts(self.dataset, self.experiment)
        self._spec = _spec_from_config(config, 1, [1.0])
        self.num_all_classes = self._spec.num_classes
        self.temperature = self._spec.temperature
        self.min_views_per_class = self._spec.min_views
        self.max_views_per_class = self._spec.max_views
        self.max_features_total = self._spec.max_total
        self.label_scaling_mode = config.get("label_scaling_mode", "nn")                 # V2.py:22
        self.cross_scale_contrast = self._spec.cross_scale
        self.log_this_step = False
        self._scale = None
        self.last_samples = None
        self._sampler_calls = 0

    def forward(self, label: torch.Tensor, features: torch.Tensor):
        if isinstance(label, CompactLabels):           # labels of the fused label pass (coloss.py): same results
            label = label.lab16
        holder = {}
        _philox_key(self, holder, features.device)
        self._spec.num_classes = self.num_all_classes          # the reference lets callers override it (V2.py:238)
        total, _terms = MsCsContrastiveFn.apply(label, self._spec, True, holder, features)
        self.last_samples, self.last_state = holder["samples"], holder["state"]
        self._scale = int(label.shape[-1] // features.shape[-1])                         # V2.py:46,203
        if holder["samples"] is None:          # captured into a CUDA graph: see fetch_logged / fetch_samples
            self.nan_flag = holder["state"].scalars[-1]
            return total
        smp = holder["samples"][0]
        if smp.log_flag:
            self.log_this_step = True                                                    # V2.py:75,83
        self.nan_flag = holder["state"].scalars[-1]      # 0-d device tensor: 1.0 if the loss is inf/NaN (no sync)
        if self.cross_scale_contrast:
            n, c = features.shape[:2]
            flat = features.reshape(n, c, -1)
            img = smp.pair_ref[:, 0].long()
            sampled = flat[img[:, None], :, smp.idx_ref.long()].permute(0, 2, 1)          # (T, C, V)
            return total, sampled, smp.pair_ref[:, 1].float(), False
        return total

    def fetch_logged(self, state=None):
        """Scalars of the last call (or of `state`) for the logger with a single device->host copy (see the _ms
        class)."""
        return _fetch_logged(self, self.last_state if state is None else state, 1, [])


class DenseContrastiveLossV2_ms(_GraphReadout, nn.Module):
    """Multi-scale + cross-scale loss.  ``forward(label, features: list)`` (_ms.py:44).

    ``comm`` (not a reference argument) switches on the POOLED cross-batch mode: the loss is then the
    reference loss of the concatenated batch of all ranks (one process per GPU, each passing its local
    images); anchor rows are sharded over the ranks, the normalised key set is exchanged over NVLink peer memory.
    Pass ``mscs_b200.TorchDistComm(process_group)``.  With ``sampler='reference'`` every rank's CPU generator must be in
    the same state; with ``sampler='philox'`` the generators need not agree, but every rank's module must have been
    called the same number of times (the call index keys the stream)."""

    def __init__(self, config, comm=None):
        super().__init__()
        self.comm = comm
        self.experiment = config["experiment"]
        self.dataset = config["dataset"]
        self.num_all_classes, self.num_real_classes, self.ignore_class = class_facts(self.dataset, self.experiment)
        self.scales = config["scales"] if "scales" in config else 2                      # _ms.py:21
        self.weights = config["weights"] if "weights" in config else [1.0] * self.scales # _ms.py:22
        assert self.scales == len(self.weights), \
            f"given dc loss number of scales [{self.scales}] not equal len of weights {self.weights}"
        self._spec = _spec_from_config(config, self.scales, self.weights, ms=True)
        self.num_all_classes = self._spec.num_classes
        self.cross_scale_contrast = self._spec.cross_scale
        self.cross_scale_temperature = self._spec.cs_temperature
        self.detach_cs_deepest = self._spec.detach_deepest
        self.w_high_low, self.w_high_mid = self._spec.w_high_low, self._spec.w_high_mid
        self.ms_losses, self.cs_losses = [], []
        self.log_this_step = False
        self.last_samples = None
        self._sampler_calls = 0

    def forward(self, label: torch.Tensor, features: list, **kwargs):
        if isinstance(label, CompactLabels):           # labels of the fused label pass (coloss.py): same results
            label = label.lab16
        self.cs_losses, self.ms_losses = [], []
        feats = list(features[:self.scales])
        if len(feats) < self.scales:
            raise IndexError("list index out of range")     # features[s] in the reference (_ms.py:53)
        if self.cross_scale_contrast:
            assert len(feats) > 1                            # _ms.py:63
        holder = {"comm": self.comm}
        _philox_key(self, holder, feats[0].device)
        total, terms = MsCsContrastiveFn.apply(label, self._spec, False, holder, *feats)
        state = holder["state"]
        self.last_samples, self.last_state = holder["samples"], state
        self.ms_losses = [terms[s] for s in range(state.num_ms)]
        self.cs_losses = [terms[i] for i in state.cs_logged]
        self.nan_flag = state.scalars[-1]                # 0-d device tensor: 1.0 if the loss is inf/NaN (no sync)
        if holder["samples"] is not None and any(s.log_flag for s in holder["samples"]):
            self.log_this_step = True
        return total

    def fetch_logged(self, state=None):
        """Scalars of the last call for the logger -- total, ms_losses, cs_losses (unweighted, as the reference logs
        them) and the inf/NaN flag -- with a single device->host copy (SURVEY.md §8f item 3).  ``state``: the state of
        another call, e.g. the ``last_state`` a CUDA graph capture left (its latest replay's values)."""
        st = self.last_state if state is None else state
        return _fetch_logged(self, st, st.num_ms, st.cs_logged)


def _fetch_logged(module, state, num_ms, cs_logged):
    """Everything the reference's logger reads per step, in ONE device->host copy (the reference does one
    ``.item()`` per scalar plus ``has_inf_or_nan`` = 4+ syncs per step, LoggingManager.py:179-196).  A captured call
    reads its latest replay's plan records in the same copy: the logging flag, and the sampling errors, which raise
    here as the eager forward would have raised them."""
    if getattr(state, "graph", False):
        v, plan = _ops.fetch_graph_plan(state)
        _ops._raise_plan_errors(plan, state.sp.S, state.sp.spec)
        if any(plan[s].log_flag for s in range(state.sp.S)):
            module.log_this_step = True                                                  # V2.py:75,83
    else:
        v = state.scalars.detach().cpu().tolist()
    nt = len(v) - 2
    return {"total": v[nt], "ms_losses": v[:num_ms], "cs_losses": [v[i] for i in cs_logged],
            "has_inf_or_nan": v[nt + 1] != 0.0, "log_this_step": bool(module.log_this_step)}


def install_into_reference():
    """Register the classes where the reference's LossWrapper looks them up by name
    (``globals()[loss_class](config)``, LossWrapper.py:33).  Call after ``import losses``."""
    mods = [sys.modules.get("losses"), sys.modules.get("losses.LossWrapper")]
    if not any(mods):
        raise RuntimeError("the reference package `losses` is not imported")
    for m in mods:
        if m is not None:
            m.DenseContrastiveLossV2 = DenseContrastiveLossV2
            m.DenseContrastiveLossV2_ms = DenseContrastiveLossV2_ms
