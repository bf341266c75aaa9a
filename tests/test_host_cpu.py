"""CPU: host-side logic, config rules, and that the C-ABI library loads and exports every
symbol include/mscs.h declares (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import mscs_b200
from mscs_b200 import _lib, _ops
from mscs_b200.datasets import class_facts
from helpers import ROOT


def test_library_exports_header_symbols():
    lib = mscs_b200.load()
    header = open(os.path.join(ROOT, "include", "mscs.h")).read()
    declared = set(re.findall(r"\b(mscs_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in mscs.h but not exported"
    assert set(_lib.EXPORTS) == declared
    assert b"sm_100a" in lib.mscs_version()


def test_struct_layouts_match_header():
    # sizes the C side uses (checked against the header by reading the field lists)
    assert ctypes.sizeof(_lib.ScalePlan) == 48
    assert ctypes.sizeof(_lib.SampleCfg) == 4 * 4 + 2 * 8 * 4 + 6 * 4
    assert ctypes.sizeof(_lib.Term) == 6 * 8 + 4 * 4 + 2 * 4 + 2 * 4 + 4 * 4 + 5 * 8 + 2 * 8      # + n1_dev, n2_dev


def test_struct_layouts_match_compiler(tmp_path):
    """Every struct of include/mscs.h as a C compiler lays it out (gcc, plain C: the header must stay C-clean) against
    the ctypes mirror the host side passes through the ABI: size and the offset of every field."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    pairs = {"mscs_sample_cfg": _lib.SampleCfg, "mscs_scale_plan": _lib.ScalePlan, "mscs_gather_item": _lib.GatherItem,
             "mscs_scatter_item": _lib.ScatterItem, "mscs_rows_item": _lib.RowsItem, "mscs_term": _lib.Term,
             "mscs_sim_job": _lib.SimJob, "mscs_forward_chain_args": _lib.ForwardChainArgs}
    header = open(os.path.join(ROOT, "include", "mscs.h")).read()
    assert set(re.findall(r"^}\s*(mscs_[a-z_]+);", header, re.M)) == set(pairs), "a header struct has no ctypes mirror"
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "mscs.h"', "int main(void) {"]
    for cname, cls in pairs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, *_ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True,
                                                       text=True).stdout.splitlines())
    for cname, cls in pairs.items():
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for fname, *_ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, f"{cname}.{fname}"


def test_mt_advance_host_matches_torch():
    lib = mscs_b200.load()
    for seed, k in [(0, 9), (1, 623), (2, 624), (3, 625), (4, 100000)]:
        torch.manual_seed(seed)
        mt, pos = _ops.torch_mt_state()
        _ops.torch_mt_advance(mt.copy(), pos, k)
        mine = torch.get_rng_state().clone()
        torch.manual_seed(seed)
        torch.randperm(k + 1)          # consumes exactly k draws
        assert torch.equal(mine, torch.get_rng_state()), (seed, k)
    assert lib.mscs_last_error() is not None


def test_class_facts_table():
    assert class_facts("CITYSCAPES", 1) == (20, 19, 19)
    assert class_facts("ADE20K", 1) == (151, 150, 150)
    assert class_facts("CADIS", 1) == (8, 8, -1)
    with pytest.raises(KeyError):
        class_facts("NOPE", 0)


def test_config_rules():
    base = dict(dataset="CITYSCAPES", experiment=1)
    m = mscs_b200.DenseContrastiveLossV2(base)
    assert m.temperature == 0.5 and m.min_views_per_class == 5 and m.max_views_per_class == 2500
    assert m.max_features_total == 10000 and m.cross_scale_contrast is False and m.log_this_step is False
    ms = mscs_b200.DenseContrastiveLossV2_ms(dict(base, temperature=0.2))
    assert ms.scales == 2 and ms.weights == [1.0, 1.0] and ms.cross_scale_temperature == pytest.approx(0.2)
    # Q5: presence of the key switches to the hard-coded 0.1
    ms = mscs_b200.DenseContrastiveLossV2_ms(dict(base, temperature=0.2, cross_scale_temperature=0.07))
    assert ms.cross_scale_temperature == pytest.approx(0.1)
    with pytest.raises(KeyError):
        mscs_b200.DenseContrastiveLossV2_ms(base)       # neither temperature key (_ms.py:28)
    with pytest.raises(AssertionError):
        mscs_b200.DenseContrastiveLossV2_ms(dict(base, temperature=0.1, scales=3, weights=[1.0, 1.0]))


def test_no_cpu_fallback():
    m = mscs_b200.DenseContrastiveLossV2(dict(dataset="CITYSCAPES", experiment=1, temperature=0.1))
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 8, 8, dtype=torch.long), torch.zeros(1, 4, 2, 2))


def test_workspace_queries_and_arg_validation():
    lib = mscs_b200.load()
    cfg = _lib.SampleCfg()
    cfg.n, cfg.H, cfg.W, cfg.num_scales = 2, 64, 128, 1
    cfg.fh[0], cfg.fw[0] = 16, 32
    cfg.num_classes, cfg.min_views, cfg.max_views, cfg.max_total = 20, 5, 100, 10000
    assert lib.mscs_sample_workspace_bytes(ctypes.byref(cfg)) > 0
    assert lib.mscs_sample_max_draws(ctypes.byref(cfg)) == 2 * 16 * 32
    cfg.fw[0] = 256                      # wider than the label map
    assert lib.mscs_sample_workspace_bytes(ctypes.byref(cfg)) == 0
    assert b"wider" in lib.mscs_last_error()


def test_step_plan_slab_layout():
    """The single allocation of a forward call (_StepPlan.slab_off): parts are 256-byte aligned, do not overlap, and
    are large enough for the upper bounds they are sized by."""
    import ctypes
    import torch
    from mscs_b200 import _lib, _ops
    spec = _ops.LossSpec(num_classes=20, temperature=0.1, cs_temperature=0.1, max_views=2500, max_total=10000,
                         weights=[1.0, 0.7, 0.4, 0.1], cross_scale=True)
    shapes = [(12, 256, 128, 256), (12, 256, 64, 128), (12, 256, 32, 64), (12, 256, 16, 32)]
    sp = _ops._StepPlan(torch.device("cpu"), (12, 512, 1024), shapes, spec, False)
    sizes = {"ws": sp.ws_bytes, "plan": 4 * ctypes.sizeof(_lib.ScalePlan), "work": sp.work_bytes, "stats": 4 * sp.stats_n,
             "misc": 4 * sp.misc_n, "fslab": 4 * sp.fslab_n, "islab": 4 * sp.islab_n, "slot": 4 * sum(sp.slot_sizes),
             "bslab": 2 * sp.bslab_n}
    spans = sorted((sp.slab_off[k], sp.slab_off[k] + v, k) for k, v in sizes.items())
    for (b0, e0, k0), (b1, e1, k1) in zip(spans, spans[1:]):
        assert e0 <= b1, (k0, k1)
    assert all(b % 256 == 0 for b, _, _ in spans) and spans[-1][1] <= sp.slab_bytes
    assert sp.v_cap == 2500 and sp.Ncap == [10000, 10000, 10000, 12 * 16 * 32]      # N <= min(max_features_total, pixels)
    assert len(sp.terms) == 6 and sp.cs_logged == [4, 5]              # 4 ms terms + cs(0,3) + cs(0,2)   (_ms.py:62-80)
    assert sp.slot_sizes == [12 * 128 * 256, 12 * 64 * 128, 12 * 32 * 64, 12 * 16 * 32]
    # a plane that is not a multiple of 8 pixels has no slot map (general scatter path)
    sp2 = _ops._StepPlan(torch.device("cpu"), (2, 60, 100), [(2, 32, 15, 25)], spec, True)
    assert sp2.slot_sizes == [0]
    assert _ops.LAUNCHES_PER_STEP(4, False) == 15


def test_launch_count_claim_matches_committed_launch_list():
    """`gpu_launches` of the bench line is LAUNCHES_PER_STEP x steps: the per-step figure must equal the number of
    libmscs.so kernels between two `k_label_hist` launches of the committed ncu launch list (same command)."""
    import csv
    for name in ("r02_launches_cfg2.csv",):
        rows = [r for r in csv.reader(open(os.path.join(ROOT, "profiles", name))) if r and r[0].isdigit()]
        names = [r[4] for r in rows]
        first = [i for i, n in enumerate(names) if "k_label_hist" in n]
        assert len(first) >= 2, name
        step = names[first[0]:first[1]]
        ours = [n for n in step if re.search(r"\bk_[a-z_0-9]+", n) and "at::" not in n]
        assert len(ours) == _ops.LAUNCHES_PER_STEP(4, False), (name, ours)
        assert any("k_sim_fwd" in n for n in ours) and any("k_sim_bwd" in n for n in ours)


def test_plan_errors_map_to_the_reference_exceptions():
    """Q8: no kept pair -> RuntimeError (torch.min of an empty tensor, V2.py:110); a kept class with one pixel ->
    IndexError (0-d squeeze, V2.py:119-121); error codes come from the device plan records."""
    spec = _ops.LossSpec(num_classes=20, temperature=0.1, cs_temperature=0.1, min_views=5)
    plan = (_lib.ScalePlan * 2)()
    _ops._raise_plan_errors(plan, 2, spec)            # both clean
    plan[1].error = 1
    with pytest.raises(RuntimeError, match="scale 1.*min_views_per_class=5"):
        _ops._raise_plan_errors(plan, 2, spec)
    plan[0].error = 2                                   # the first failing scale wins, like the reference's scale loop
    with pytest.raises(IndexError, match="scale 0"):
        _ops._raise_plan_errors(plan, 2, spec)


def test_fast_path_gate():
    """Device-driven order: a single process.  The selection table (12 B per view) always fits the 200 KB of shared
    memory, because V is capped at 16384 views (192 KB)."""
    mk = lambda **kw: _ops.LossSpec(num_classes=20, temperature=0.1, cs_temperature=0.1, **kw)
    assert _ops.fast_path_ok(mk(), 1)                                   # reference defaults: V <= 2500
    assert not _ops.fast_path_ok(mk(), 2)                               # pooled mode takes the host-driven order
    assert _ops.fast_path_ok(mk(max_views=1, max_total=10000), 1)       # max_views == 1 means "no per-class cap" (Q3)
    assert _ops.fast_path_ok(mk(max_views=1, max_total=65536), 1)       # V is capped at 16384 views: 192 KB, just inside
    assert _ops.fast_path_ok(mk(max_views=1000, max_total=32768), 1)    # cfg-4 large
