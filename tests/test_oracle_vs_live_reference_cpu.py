"""CPU, needs a checkout of the original project (MSCS_REFERENCE=<checkout>, skipped without one): the oracle
restatements against the EXECUTABLE reference on randomly drawn configurations -- number of scales 1..4, strides that repeat (Q11), datasets
with and without an ignore id (Q2), caps that do / do not bind (Q3, Q4), the cross-scale temperature rule (Q5),
detach_deepest (Q6), label maps whose size is not a multiple of the stride (nearest rule of V2.py:194-206).
The committed fixtures pin fixed cases; this pins the rules between them.  Runs in a subprocess because the import
shims (stub `utils` / `losses` packages, `Tensor.cuda` -> identity) must not leak into other tests."""
import os
import subprocess
import sys

import pytest

from helpers import ROOT

REF = os.environ.get("MSCS_REFERENCE", "")

SCRIPT = r'''
import os, sys
import numpy as np
import torch
ROOT = sys.argv[1]
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers                                # random_case(): the generator shared with the GPU parity test
import make_golden as mg                      # import_reference(), ref_indices(): the shims of SURVEY.md 8c
from mscs_b200 import synth
from oracle import loss_fp64, torch_port
from oracle.config import oracle_cfg
from oracle.mt19937 import MT19937

DCV2, DCV2ms, INFO = mg.import_reference()
torch.set_num_threads(4)
rs = np.random.RandomState(20221017)
n_cases = int(sys.argv[2])
done = refused = 0
for case in range(n_cases):
    rc = helpers.random_case(rs)
    if rc is None:
        continue
    cfg, single, labels, feats, seed, S = rc["cfg"], rc["single"], rc["labels"], rc["feats"], rc["seed"], rc["S"]
    A = len(INFO[cfg["dataset"]].CLASS_INFO[cfg["experiment"]][1])
    assert A == helpers.CLASSES[(cfg["dataset"], cfg["experiment"])]
    ocfg = helpers.oracle_cfg_for(dict(loss_cfg=cfg, single_scale=single))
    fg = [f.clone().requires_grad_(True) for f in feats]
    torch.manual_seed(seed)
    state0 = torch.get_rng_state()
    try:
        if single:
            mod = DCV2(dict(cfg)); loss = mod(labels, fg[0]); inner = [mod]
            ms_l, cs_l = [float(loss)], []
        else:
            mod = DCV2ms(dict(cfg)); loss = mod(labels, fg)
            ms_l, cs_l = [float(x) for x in mod.ms_losses], [float(x) for x in mod.cs_losses]
            inner = [getattr(mod, f"DCV2_scale{s}") for s in range(S)]
    except (RuntimeError, IndexError, ValueError):
        # no kept pair / count-1 pair (Q8): the oracle must refuse the same input
        gen = MT19937.from_torch_state(state0.numpy().tobytes())
        try:
            loss_fp64.ms_cs_loss(labels.numpy(), [f.numpy() for f in feats], ocfg, gen, need_grad=False)
        except Exception:
            refused += 1
            continue
        raise AssertionError(f"case {case}: the reference raised, the oracle did not ({cfg})")
    if not np.isfinite(float(loss)):
        continue
    loss.backward()
    state1 = torch.get_rng_state()
    st, idxs, pairs = state0, [], []
    for s, f in enumerate(feats):
        i_, p_ = mg.ref_indices(inner[s], labels, f.shape, st)
        st = torch.get_rng_state()
        idxs.append(i_); pairs.append(p_)
    assert torch.equal(st, state1)
    gen = MT19937.from_torch_state(state0.numpy().tobytes())
    res = loss_fp64.ms_cs_loss(labels.numpy(), [f.numpy() for f in feats], ocfg, gen, need_grad=True)
    for s in range(S):
        assert np.array_equal(res["samples"][s]["idx"], idxs[s]), (case, s, cfg)
        assert np.array_equal(res["samples"][s]["pairs"], pairs[s]), (case, s, cfg)
    after = MT19937.from_torch_state(state1.numpy().tobytes())
    assert gen.pos == after.pos and np.array_equal(gen.mt, after.mt), (case, cfg)
    assert abs(res["total"] - float(loss)) <= 5e-6 * abs(float(loss)) + 1e-6, (case, res["total"], float(loss), cfg)
    assert len(res["ms"]) == len(ms_l) and len(res["cs"]) == len(cs_l), (case, res["cs"], cs_l, cfg)
    for a, b in zip(res["ms"] + res["cs"], ms_l + cs_l):
        assert abs(a - b) <= 5e-6 * abs(b) + 1e-6, (case, a, b, cfg)     # a one-class scale has loss ~0 (fp32 noise)
    for s in range(S):
        g64 = res["grads"][s].ravel()
        g32 = (fg[s].grad.numpy() if fg[s].grad is not None else np.zeros_like(feats[s].numpy())).ravel().astype(np.float64)
        if max(np.abs(g64).max(), np.abs(g32).max()) < 1e-7:      # a one-class scale: gradient 0 up to fp32 noise
            continue
        cos = float(g64 @ g32 / np.sqrt((g64 @ g64) * (g32 @ g32)))
        assert cos > 0.99999, (case, s, cos, cfg)
    torch.set_rng_state(state0)
    fp = [f.clone().requires_grad_(True) for f in feats]
    tot_p, _, _, idx_p = torch_port.ms_cs_loss(labels, fp, ocfg)
    assert abs(float(tot_p) - float(loss)) <= 2e-6 * abs(float(loss)) + 1e-6, (case, float(tot_p), float(loss))
    for s in range(S):
        assert np.array_equal(idx_p[s].numpy(), idxs[s])
    done += 1
print(f"LIVE-OK {done} of {n_cases} cases compared, {refused} refused by both")
assert done >= n_cases // 2 and done + refused >= n_cases - 4, (done, refused)
'''


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "losses")),
                    reason="needs a checkout of the original project (MSCS_REFERENCE)")
def test_oracle_matches_live_reference_on_random_configs(tmp_path):
    script = tmp_path / "live.py"
    script.write_text(SCRIPT)
    r = subprocess.run([sys.executable, str(script), ROOT, "40"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "LIVE-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
