"""GPU tests through the reference's boundary: this repository's classes registered under the reference's names in a
``losses`` namespace (``mscs_b200.install_into_reference``), built by name and driven the way the reference's
``losses/LossWrapper.py`` drives them (``helpers.LossWrapperBoundary``): ``module(labels, deep_features)``, the result
multiplied IN PLACE by the loss weight, detached for the logger, ``ms_losses`` / ``cs_losses`` copied into
``loss_vals`` and added to ``total_loss``; the test then calls ``total_loss.backward()`` like ``forward_step`` does.
Checked against the recorded outputs of the reference (tests/golden, tests/golden/make_golden.py) on the same inputs
and generator state: the small fully stored cases and every BASELINE configuration whose recording holds gradient rows
(cfg-4-large: recorded from the fp64 oracle, which the other cases pin against the reference).

Tolerances (north_star): loss <= 1e-3 relative, gradient cosine >= 0.999, max-abs printed.
"""
import sys
import types

import numpy as np
import pytest
import torch

from helpers import LossWrapperBoundary, cosine, load_npz, small_case_inputs

pytestmark = pytest.mark.gpu

MS, SS = "DenseContrastiveLossV2_ms", "DenseContrastiveLossV2"


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


class _installed:
    """A ``losses`` namespace with our classes registered under the reference's names (install_into_reference), removed
    again afterwards."""

    def __enter__(self):
        import mscs_b200
        assert "losses" not in sys.modules, "a module named 'losses' is already imported"
        self.ns = sys.modules["losses"] = types.ModuleType("losses")
        mscs_b200.install_into_reference()
        return self.ns

    def __exit__(self, *exc):
        del sys.modules["losses"]


def _wrapper_cfg(loss_cfg, key, weight, dev):
    cfg = dict(loss_cfg)
    cfg.update(losses={key: weight}, device=dev)
    return cfg


def _run_wrapper(ns, cfg, key, labels, feats, rng_state, dev):
    """LossWrapper(cfg) -> forward(None, labels, deep_features=...) -> total_loss.backward(), as forward_step does."""
    lw = LossWrapperBoundary(cfg, ns)
    fg = [f.detach().clone().to(dev).requires_grad_(True) for f in feats]
    torch.set_rng_state(rng_state)
    total = lw(None, labels.to(dev), deep_features=fg[0] if key == SS else fg)
    total.backward()
    torch.cuda.synchronize()
    return lw, total, fg


@pytest.mark.parametrize("name", ["tiny_ms", "tiny_ms_detach", "tiny_ss", "odd_ss"])
def test_unmodified_losswrapper_small_vs_recorded_reference(name, golden, dev):
    """The reference's LossWrapper calling convention, RESTATED by helpers.LossWrapperBoundary (the unmodified file
    itself runs only in tests/test_reference_dropin_cpu.py, given a checkout), on the fully recorded small cases."""
    import mscs_b200
    meta = golden[name]
    labels, feats, z = small_case_inputs(name)
    key, w = (SS if meta["single_scale"] else MS), 0.1
    with _installed() as ns:
        cfg = _wrapper_cfg(meta["loss_cfg"], key, w, dev)
        lw, total, fg = _run_wrapper(ns, cfg, key, labels, feats, torch.from_numpy(z["rng_state0"]), dev)
        assert type(lw.loss_classes[key]) is getattr(mscs_b200, key)
    assert total.dim() == 0 and total.dtype == torch.float32
    assert abs(float(total) - w * meta["total"]) < 1e-3 * abs(w * meta["total"])
    assert abs(float(lw.loss_vals[key]) - w * meta["total"]) < 1e-3 * abs(w * meta["total"])
    assert not lw.loss_vals[key].requires_grad
    if key == MS:
        # logged per-scale values are the UNWEIGHTED term losses (LossWrapper.py:96-101)
        for i, v in enumerate(meta["ms"]):
            assert abs(float(lw.loss_vals[f"{MS}_ms{i}"]) - v) < 1e-3 * abs(v)
        for i, v in enumerate(meta["cs"]):
            assert abs(float(lw.loss_vals[f"{MS}_cs{i}"]) - v) < 1e-3 * abs(v)
        assert f"{MS}_ms{len(meta['ms'])}" not in lw.loss_vals and f"{MS}_cs{len(meta['cs'])}" not in lw.loss_vals
        # the in-place multiply of the wrapper must not leak into the logged scalars of the module
        logged = lw.loss_classes[key].fetch_logged()
        assert abs(logged["total"] - meta["total"]) < 1e-3 * abs(meta["total"])
    for s, f in enumerate(fg):
        got, want = f.grad.cpu().numpy(), w * z[f"grad{s}"]
        cs, err = cosine(got, want), np.abs(got - want).max()
        print(f"{name} via LossWrapper, scale {s}: grad cosine {cs:.7f} max-abs {err:.3e} (max {np.abs(want).max():.3e})")
        assert cs >= 0.999
    assert torch.equal(torch.get_rng_state(), torch.from_numpy(z["rng_state1"]))


def test_unmodified_losswrapper_cfg2_vs_recorded_reference(golden, dev):
    """As above (the wrapper is the restatement helpers.LossWrapperBoundary) at cfg-2, against the recorded losses,
    gradient norms and generator state."""
    from mscs_b200 import synth
    meta, z = golden["cfg2"], load_npz("cfg2")
    labels, feats = synth.make_inputs("cfg2")
    w = 0.1
    with _installed() as ns:
        lw, total, fg = _run_wrapper(ns, _wrapper_cfg(meta["loss_cfg"], MS, w, dev), MS, labels, feats,
                                     torch.from_numpy(z["rng_state0"]), dev)
    assert abs(float(total) - w * meta["total"]) < 1e-3 * abs(w * meta["total"])
    for i, v in enumerate(meta["ms"]):
        assert abs(float(lw.loss_vals[f"{MS}_ms{i}"]) - v) < 1e-3 * abs(v)
    for i, v in enumerate(meta["cs"]):
        assert abs(float(lw.loss_vals[f"{MS}_cs{i}"]) - v) < 1e-3 * abs(v)
    for s, f in enumerate(fg):
        tot = float(f.grad.double().norm())
        assert abs(tot - w * meta["grad_l2"][s]) < 1e-2 * w * meta["grad_l2"][s]
    assert torch.equal(torch.get_rng_state(), torch.from_numpy(z["rng_state1"]))


BENCH = ["cfg1", "cfg2", "cfg3", "cfg4", "cfg4_large"]


@pytest.mark.parametrize("name", BENCH)
def test_losswrapper_bench_configs_vs_recorded_reference(name, golden, dev):
    """Our classes behind the wrapper, same inputs and generator state as the recorded run: total loss, every logged
    scalar, the generator state after the call, and the dense gradients (exactly the recorded sampled pixels carry a
    gradient; recorded gradient rows, norms of every sampled row and the global norm)."""
    from mscs_b200 import synth
    meta, z = golden[name], load_npz(name)
    labels, feats = synth.make_inputs(name)
    key, w = (SS if meta["single_scale"] else MS), 0.1
    with _installed() as ns:
        lw, total, fg = _run_wrapper(ns, _wrapper_cfg(meta["loss_cfg"], key, w, dev), key, labels, feats,
                                     torch.from_numpy(z["rng_state0"]), dev)
    state1 = z["rng_state1"] if "rng_state1" in z else load_npz(name + "_sampling")["rng_state1"]
    assert torch.equal(torch.get_rng_state(), torch.from_numpy(state1)), "generator state after the call differs"
    want = {key: w * meta["total"]}
    if key == MS:
        want.update({f"{MS}_ms{i}": v for i, v in enumerate(meta["ms"])})
        want.update({f"{MS}_cs{i}": v for i, v in enumerate(meta["cs"])})
    assert set(lw.loss_vals) == set(want), (sorted(lw.loss_vals), sorted(want))
    for k, v in want.items():
        rel = abs(float(lw.loss_vals[k]) - v) / abs(v)
        print(f"{name} {k}: ours {float(lw.loss_vals[k]):.7f} reference {v:.7f} rel {rel:.2e}")
        assert rel < 1e-3, (k, float(lw.loss_vals[k]), v)
    assert abs(float(total) - w * meta["total"]) < 1e-3 * abs(w * meta["total"])
    for s, f in enumerate(fg):
        n, C, h, w_ = f.shape
        g = f.grad.reshape(n, C, h * w_)
        idx, pairs = z[f"idx{s}"].astype(np.int64), z[f"pairs{s}"].astype(np.int64)
        T, V = idx.shape
        ball = torch.from_numpy(np.repeat(pairs[:, 0], V)).to(dev)
        pall = torch.from_numpy(idx.ravel()).to(dev)
        sampled = torch.zeros((n, h * w_), dtype=torch.bool, device=dev)
        sampled[ball, pall] = True
        assert torch.equal((g != 0).any(dim=1), sampled), "different pixels carry a gradient"
        rows_all = g[ball, :, pall]
        ids = z[f"grad_row_ids{s}"].astype(np.int64)
        rows, want_rows = rows_all[torch.from_numpy(ids).to(dev)].double().cpu().numpy(), w * z[f"grad_rows{s}"]
        cs, err, mx = cosine(rows, want_rows), np.abs(rows - want_rows).max(), np.abs(want_rows).max()
        l2_cos = cosine(rows_all.norm(dim=1).cpu().numpy(), z[f"grad_row_l2_{s}"])
        tot = float(f.grad.double().norm())
        print(f"{name} scale {s}: grad rows cosine {cs:.8f} max-abs {err:.3e} (reference max {mx:.3e}); row-norm "
              f"cosine {l2_cos:.8f}; |grad| {tot:.6e} vs {w * meta['grad_l2'][s]:.6e}")
        assert cs >= 0.999 and l2_cos >= 0.999
        assert err < 0.05 * mx
        assert abs(tot - w * meta["grad_l2"][s]) < 1e-2 * w * meta["grad_l2"][s]
