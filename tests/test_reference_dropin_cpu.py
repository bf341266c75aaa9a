"""CPU, needs a checkout of the original project (MSCS_REFERENCE=<checkout>, skipped without one): the UNMODIFIED
reference LossWrapper builds
and dispatches this repository's classes once they are registered under the reference's names
(LossWrapper.py:33 `globals()[loss_class](config)`, :68-71 `module(labels, deep_features)`).
Runs in a subprocess: the import shims (stub `utils` / `losses` packages) must not leak into other tests."""
import os
import subprocess
import sys

import pytest

from helpers import ROOT

REF = os.environ.get("MSCS_REFERENCE", "")

SCRIPT = r'''
import importlib, os, sys, types
import torch
REF, ROOT = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
utils = types.ModuleType("utils"); utils.__path__ = [os.path.join(REF, "utils")]; sys.modules["utils"] = utils
defaults = importlib.import_module("utils.defaults")              # the real dataset tables (pure Python)
utils.DATASETS_INFO = defaults.DATASETS_INFO
losses = types.ModuleType("losses"); losses.__path__ = [os.path.join(REF, "losses")]; sys.modules["losses"] = losses
wrapper_mod = importlib.import_module("losses.LossWrapper")       # the reference file, unmodified

import mscs_b200
mscs_b200.install_into_reference()

loss_cfg = {"losses": {"DenseContrastiveLossV2_ms": 0.1, "DenseContrastiveLossV2": 0.5},
            "device": "cpu", "dataset": "CITYSCAPES", "experiment": 1, "temperature": 0.1,
            "scales": 4, "weights": [1.0, 0.7, 0.4, 0.1], "cross_scale_contrast": True,
            "w_high_low": 1.0, "w_high_mid": 0.5, "max_views_per_class": 2500, "unknown_key": 1}
lw = wrapper_mod.LossWrapper(loss_cfg)
ms, ss = lw.loss_classes["DenseContrastiveLossV2_ms"], lw.loss_classes["DenseContrastiveLossV2"]
assert type(ms) is mscs_b200.DenseContrastiveLossV2_ms and type(ss) is mscs_b200.DenseContrastiveLossV2
assert lw.ignore_class == 19 == ms.ignore_class and ms.num_all_classes == 20
# the built-in class table (used when the reference's `utils` is not importable) agrees with the reference's own
# tables for every dataset / experiment both know
from mscs_b200.datasets import _TABLE
checked = 0
for (ds, exp), (n_all, has255) in _TABLE.items():
    table = defaults.DATASETS_INFO[ds].CLASS_INFO
    id_to_name = table[exp][1]
    assert n_all == len(id_to_name) and has255 == (255 in id_to_name), (ds, exp, n_all, has255, len(id_to_name))
    checked += 1
assert checked == len(_TABLE) >= 10
assert ms.scales == 4 and ms.weights == [1.0, 0.7, 0.4, 0.1] and ms.cross_scale_contrast is True
assert ms.cross_scale_temperature == 0.1 and ms.w_high_mid == 0.5 and ms.ms_losses == [] and ms.cs_losses == []
assert ss.temperature == 0.1 and ss.max_views_per_class == 2500 and ss.log_this_step is False
# dispatch: LossWrapper.forward reaches our module with (labels, deep_features); on this CPU-only machine the
# module refuses loudly (no fallback) instead of computing something else
labels = torch.zeros((1, 64, 64), dtype=torch.long)
feats = [torch.randn(1, 8, 64 >> (2 + s), 64 >> (2 + s)) for s in range(4)]
try:
    lw(None, labels, loss_list=["DenseContrastiveLossV2_ms"], deep_features=feats)
except RuntimeError as e:
    assert "mscs_b200" in str(e), e
else:
    raise AssertionError("the CUDA-only loss ran on CPU tensors")
print("DROPIN-OK")
'''


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "losses")),
                    reason="needs a checkout of the original project (MSCS_REFERENCE)")
def test_reference_losswrapper_builds_and_dispatches_our_classes(tmp_path):
    script = tmp_path / "dropin.py"
    script.write_text(SCRIPT)
    r = subprocess.run([sys.executable, str(script), REF, ROOT], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "DROPIN-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
