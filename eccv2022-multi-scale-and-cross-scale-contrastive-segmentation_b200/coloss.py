"""Co-losses on ONE read of the label map (SURVEY.md section 8f, item 2).

The reference's ``LossWrapper`` (losses/LossWrapper.py:22-37,81-82) evaluates a class-weighted
``nn.CrossEntropyLoss(ignore_index=ignore_class, weight=class_weights)`` on the full-resolution logits next to
``DenseContrastiveLossV2_ms``; ``TwoScaleLoss`` (losses/TwoScaleLoss.py:62-73) applies the same loss to two logit maps.
Each of them reads the int64 label map on its own.  Here one sweep (csrc/ce.cu:k_label_pass) yields compact int16
labels + the full-resolution class histogram, and both losses work from those:

  * ``CrossEntropyLabelPass``  == ``nn.CrossEntropyLoss(ignore_index, weight)`` (mean reduction): two fused HBM-bound
    kernels (forward: one read of the logits; backward: one read + one write, final scale included because the
    normaliser comes from the histogram), against ATen's log_softmax / nll_loss forward + two backward kernels;
  * the contrastive classes accept the ``CompactLabels`` in place of the int64 tensor (K1 reads a quarter of the bytes).

``FusedCoLosses`` is the LossWrapper-shaped combination of the two for the keys ``CrossEntropyLoss`` and
``DenseContrastiveLossV2_ms`` (same config dict, same ``loss_vals`` entries).  Not reference class names: the reference
dispatches those by name and nothing here shadows them.
"""
import torch
import torch.nn as nn

from . import _lib, _ops
from ._ops import CompactLabels
from .datasets import class_facts
from .losses import DenseContrastiveLossV2_ms

# class weights the reference hard-codes for Cityscapes (losses/LossWrapper.py:26-29)
CITYSCAPES_CLASS_WEIGHTS = [0.8373, 0.918, 0.866, 1.0345, 1.0166, 0.9969, 0.9754, 1.0489, 0.8786, 1.0023, 0.9539, 0.9843,
                            1.1116, 0.9037, 1.0865, 1.0955, 1.0865, 1.1529, 1.0507]


def label_pass(labels, num_all_classes):
    """One sweep over the int64 labels (n, H, W) -> CompactLabels (int16 map, class histogram int32[A])."""
    _ops._require_device(labels)
    if labels.dtype != torch.int64:
        labels = labels.long()
    labels = labels.contiguous()
    lab16 = torch.empty(labels.shape, dtype=torch.int16, device=labels.device)
    hist = torch.empty(num_all_classes, dtype=torch.int32, device=labels.device)
    with torch.cuda.device(labels.device):
        _lib.check(_lib.load().mscs_label_pass(labels.data_ptr(), labels.numel(), num_all_classes, lab16.data_ptr(),
                                               hist.data_ptr(), _ops._stream()), "mscs_label_pass")
    return CompactLabels(lab16, hist, num_all_classes)


class _FusedCEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, compact, weight, ignore_index):
        lib = _lib.load()
        _ops._require_device(logits)
        # fp32, bf16 and fp16 logits are read as they are (dlogits come back in the same dtype); others as an fp32 copy
        x = logits.detach()
        if x.dtype not in _ops._DTYPE_CODE:
            x = x.float()
        x = x.contiguous()
        if x.dtype != torch.float32 and x.data_ptr() % 8:      # a view at an odd offset: the kernels load 8 bytes
            x = x.clone()
        n, K, H, W = x.shape
        if compact.shape != (n, H, W):
            raise ValueError(f"labels {compact.shape} do not match the logits {tuple(x.shape)}")
        w = None if weight is None else weight.detach().to(device=x.device, dtype=torch.float32).contiguous()
        scratch = torch.empty(2, dtype=torch.float64, device=x.device)
        out = torch.empty(2, dtype=torch.float32, device=x.device)           # [loss, normaliser]
        loss = torch.empty((), dtype=torch.float32, device=x.device)          # own storage: LossWrapper multiplies in place
        with torch.cuda.device(x.device):
            _lib.check(lib.mscs_ce_forward(x.data_ptr(), compact.lab16.data_ptr(), n, K, H * W,
                                           None if w is None else w.data_ptr(), int(ignore_index), compact.hist.data_ptr(),
                                           compact.num_classes, scratch.data_ptr(), out.data_ptr(), _ops._stream(),
                                           _ops._DTYPE_CODE[x.dtype]), "mscs_ce_forward")
            loss.copy_(out[0])
        ctx.x, ctx.compact, ctx.w, ctx.ignore, ctx.out, ctx.dtype = x, compact, w, int(ignore_index), out, logits.dtype
        return loss

    @staticmethod
    def backward(ctx, grad):
        lib = _lib.load()
        x = ctx.x
        n, K, H, W = x.shape
        g = grad.detach().to(device=x.device, dtype=torch.float32).reshape(1).contiguous()
        dx = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(lib.mscs_ce_backward(x.data_ptr(), ctx.compact.lab16.data_ptr(), n, K, H * W,
                                            None if ctx.w is None else ctx.w.data_ptr(), ctx.ignore, g.data_ptr(),
                                            ctx.out[1:].data_ptr(), dx.data_ptr(), _ops._stream(),
                                            _ops._DTYPE_CODE[x.dtype]), "mscs_ce_backward")
        return (dx if dx.dtype == ctx.dtype else dx.to(ctx.dtype)), None, None, None


class CrossEntropyLabelPass(nn.Module):
    """``forward(prediction, labels)`` == ``nn.CrossEntropyLoss(ignore_index=ignore_index, weight=weight)`` (fp32, mean
    over the non-ignored pixels weighted by class).  ``labels``: int64 (n, H, W) or the ``CompactLabels`` of a label
    pass that has already been made for this step (``label_pass``)."""

    def __init__(self, num_all_classes, ignore_index=-100, weight=None):
        super().__init__()
        self.num_all_classes, self.ignore_index = int(num_all_classes), int(ignore_index)
        self.register_buffer("weight", None if weight is None else torch.as_tensor(weight, dtype=torch.float32))

    def forward(self, prediction, labels):
        compact = labels if isinstance(labels, CompactLabels) else label_pass(labels, self.num_all_classes)
        return _FusedCEFn.apply(prediction, compact, self.weight, self.ignore_index)


class FusedCoLosses(nn.Module):
    """LossWrapper-shaped combination (losses/LossWrapper.py:40-103) of ``CrossEntropyLoss`` and
    ``DenseContrastiveLossV2_ms`` on ONE label read: ``forward(prediction, labels, deep_features=...)`` returns the
    weighted total and fills ``loss_vals`` with the same keys the reference's wrapper logs."""

    def __init__(self, config):
        super().__init__()
        self.loss_weightings = dict(config["losses"])
        unknown = set(self.loss_weightings) - {"CrossEntropyLoss", "DenseContrastiveLossV2_ms"}
        if unknown:
            raise ValueError(f"FusedCoLosses handles CrossEntropyLoss and DenseContrastiveLossV2_ms, not {sorted(unknown)}")
        self.dataset, self.experiment = config["dataset"], config["experiment"]
        n_all, _n_real, ignore = class_facts(self.dataset, self.experiment)
        self.num_all_classes, self.ignore_class = n_all, ignore
        weights = CITYSCAPES_CLASS_WEIGHTS if self.dataset == "CITYSCAPES" else None        # LossWrapper.py:24-29
        self.ce = CrossEntropyLabelPass(n_all, ignore, weights) if "CrossEntropyLoss" in self.loss_weightings else None
        self.dc = DenseContrastiveLossV2_ms(config) if "DenseContrastiveLossV2_ms" in self.loss_weightings else None
        self.loss_vals = {k: 0 for k in self.loss_weightings}
        self.total_loss = None

    def forward(self, prediction, labels, deep_features=None):
        compact = label_pass(labels, self.num_all_classes)          # the one read of the int64 label map
        total = None
        for key, w in self.loss_weightings.items():
            if key == "CrossEntropyLoss":
                loss = self.ce(prediction, compact)
            else:
                assert deep_features is not None, f"for loss_class {key}, deep_features must be given"
                loss = self.dc(compact, deep_features)
            loss *= w                                                # LossWrapper.py:90
            self.loss_vals[key] = loss.detach()
            if key == "DenseContrastiveLossV2_ms":                   # LossWrapper.py:94-101
                for s, v in enumerate(self.dc.ms_losses):
                    self.loss_vals[f"{key}_ms{s}"] = v
                if self.dc.cross_scale_contrast:
                    for s, v in enumerate(self.dc.cs_losses):
                        self.loss_vals[f"{key}_cs{s}"] = v
            total = loss if total is None else total + loss
        self.total_loss = total
        return total
