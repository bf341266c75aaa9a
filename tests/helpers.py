"""Shared helpers of the test-suite (oracle-side config, golden loading, comparisons)."""
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# num_all_classes per (dataset, experiment) -- SURVEY.md §8a
CLASSES = {("CITYSCAPES", 1): 20, ("ADE20K", 1): 151, ("CADIS", 1): 8, ("CADIS", 2): 18, ("CADIS", 3): 26}


def load_npz(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def oracle_cfg_for(meta):
    from oracle.config import oracle_cfg
    lc = meta["loss_cfg"]
    cfg = oracle_cfg(lc, CLASSES[(lc["dataset"], lc["experiment"])])
    if meta["single_scale"]:
        cfg["cross_scale"] = False
        cfg["weights"] = [1.0]
    return cfg


def small_case_inputs(name):
    """labels (int64) and feature list (fp32) of a fully stored golden case."""
    z = load_npz(name)
    feats = []
    s = 0
    while f"feat{s}" in z:
        feats.append(torch.from_numpy(z[f"feat{s}"]))
        s += 1
    return torch.from_numpy(z["labels"].astype(np.int64)), feats, z


def cosine(a, b):
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    return float(a @ b / np.sqrt((a @ a) * (b @ b)))


class LossWrapperBoundary:
    """The calling convention of the reference's ``losses/LossWrapper.py`` for the contrastive classes, restated: the
    class is built by NAME from the ``losses`` namespace (``globals()[loss_class](config)``, :33), called as
    ``module(labels, deep_features)`` (:68-71), the returned tensor is multiplied IN PLACE by the loss weight (:90) and
    logged detached (:91), the per-scale ``ms_losses`` / ``cs_losses`` of the _ms class are logged under
    ``<name>_ms<i>`` / ``<name>_cs<i>`` (:94-101) and the weighted losses are summed into ``total_loss`` (:102)."""

    def __init__(self, config, namespace):
        self.loss_weightings = dict(config["losses"])
        self.loss_classes = {k: getattr(namespace, k)(config) for k in self.loss_weightings}
        self.loss_vals = {k: 0 for k in self.loss_weightings}
        self.total_loss = None

    def __call__(self, prediction, labels, deep_features=None):
        total = None
        for key, w in self.loss_weightings.items():
            module = self.loss_classes[key]
            loss = module(labels, deep_features)
            loss *= w
            self.loss_vals[key] = loss.detach()
            if key == "DenseContrastiveLossV2_ms":
                for i, v in enumerate(module.ms_losses):
                    self.loss_vals[f"{key}_ms{i}"] = v
                if module.cross_scale_contrast:
                    for i, v in enumerate(module.cs_losses):
                        self.loss_vals[f"{key}_cs{i}"] = v
            total = loss if total is None else total + loss
        self.total_loss = total
        return total


def make_module(meta, device=None):
    import mscs_b200
    cls = mscs_b200.DenseContrastiveLossV2 if meta["single_scale"] else mscs_b200.DenseContrastiveLossV2_ms
    return cls(dict(meta["loss_cfg"]))


RANDOM_DATASETS = [("CITYSCAPES", 1), ("CADIS", 2), ("CADIS", 1), ("ADE20K", 1)]


def random_case(rs):
    """One randomly drawn configuration + inputs (``rs``: numpy RandomState).  Shared by the CPU test that pins the
    oracle against the live reference and by the GPU parity test, so both walk the same cases: 1..4 scales, strides
    that repeat (Q11), datasets with / without an ignore id (Q2), caps that do / do not bind (Q3, Q4), the cross-scale
    temperature rule (Q5), detach_deepest (Q6), ragged label widths (nearest rule, V2.py:194-206), maps too small to
    keep any (image, class) pair at the deepest scale (Q8).  Returns None for a draw that is not a valid input."""
    from mscs_b200 import synth
    ds, exp = RANDOM_DATASETS[rs.randint(len(RANDOM_DATASETS))]
    A = CLASSES[(ds, exp)]
    S = int(rs.randint(1, 5))
    single = S == 1
    n = int(rs.randint(1, 4))
    cell = int(rs.choice([4, 8]))
    strides = sorted(int(rs.choice([2, 4])) * (2 ** s if rs.rand() < 0.8 else max(1, 2 ** (s - 1))) for s in range(S))
    unit = int(np.lcm(cell, strides[-1]))
    if rs.rand() < 0.2:       # so small that the deepest scale keeps no pair: reference, oracle and kernels must all refuse
        H, W = unit, int(rs.randint(1, 3)) * unit
    else:
        H, W = int(rs.randint(3, 7)) * unit, int(rs.randint(4, 9)) * unit
    ragged = rs.rand() < 0.3
    k = int(rs.randint(2, min(5, A - 1) + 1))
    # class id A-1 is the dropped column: the ignore id, or the last REAL class of a dataset without a 255 key (Q2)
    labels = synth.synth_labels(n, H, W, A - 1, k, cell, 0.1, int(rs.randint(1 << 30)))
    C = int(rs.choice([8, 24, 48]))
    g = torch.Generator().manual_seed(int(rs.randint(1 << 30)))
    feats = [torch.randn(n, C, H // s, W // s, generator=g) for s in strides]
    valid = True
    if ragged:            # a few extra label columns: the integer stride (V2.py:46) stays, the nearest rule is no longer a stride
        pad = int(rs.randint(1, strides[0]))
        labels = torch.nn.functional.pad(labels, (0, pad, 0, 0), value=int(labels[0, 0, 0]))
        valid = all(labels.shape[-1] // f.shape[-1] == s for f, s in zip(feats, strides))
    cfg = dict(dataset=ds, experiment=exp, temperature=float(rs.choice([0.07, 0.1, 0.5])),
               min_views_per_class=int(rs.randint(2, 6)), max_views_per_class=int(rs.choice([1, 7, 30, 2500])),
               max_features_total=int(rs.choice([60, 300, 10000])))
    if not single:
        cfg.update(scales=S, weights=[float(x) for x in rs.rand(S).round(2) + 0.1],
                   cross_scale_contrast=bool(rs.rand() < 0.75), detach_deepest=bool(rs.rand() < 0.3),
                   w_high_low=float(rs.choice([1.0, 0.5])), w_high_mid=float(rs.choice([1.0, 0.25])))
        if rs.rand() < 0.3:
            cfg["cross_scale_temperature"] = 0.3      # presence of the key -> 0.1 (Q5)
    seed = int(rs.randint(1 << 30))
    if not valid:
        return None
    return dict(cfg=cfg, single=single, labels=labels, feats=feats, seed=seed, S=S, strides=strides)
