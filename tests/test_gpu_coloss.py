"""GPU: the co-losses on one label read (SURVEY.md 8f item 2, mscs_b200/coloss.py, csrc/ce.cu) against ATen, and the
LossWrapper-shaped combination CrossEntropyLoss + DenseContrastiveLossV2_ms against ATen plus the fp64 oracle.

Tolerances: the label pass and K1 on compact labels are bit-exact; the fused cross entropy is fp32 against fp32 ATen
(loss <= 1e-5 relative, gradient max-abs <= 1e-5 of the gradient's max); the combined total follows north_star
(1e-3 relative; gradient cosine >= 0.999)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def test_label_pass_bit_exact(dev):
    import mscs_b200
    g = torch.Generator().manual_seed(0)
    for shape, A in (((3, 97, 131), 20), ((2, 512, 1024), 151), ((1, 8, 9), 8)):
        lab = torch.randint(-2, A + 3, shape, generator=g)
        lab[0, 0, 0] = 255
        c = mscs_b200.label_pass(lab.to(dev), A)
        want = torch.where((lab >= 0) & (lab < A), lab, torch.full_like(lab, -1)).to(torch.int16)
        assert torch.equal(c.lab16.cpu(), want)
        assert torch.equal(c.hist.cpu().long(), torch.bincount(lab[(lab >= 0) & (lab < A)].flatten(), minlength=A))


@pytest.mark.parametrize("case", ["cityscapes", "ade20k", "all_ignored_quads"])
def test_fused_cross_entropy_vs_aten(case, dev):
    import mscs_b200
    from mscs_b200.coloss import CITYSCAPES_CLASS_WEIGHTS
    g = torch.Generator().manual_seed(1)
    if case == "ade20k":
        n, K, H, W, A, ignore, wts = 2, 150, 64, 96, 151, 150, None
    else:
        n, K, H, W, A, ignore, wts = 3, 19, 128, 256, 20, 19, CITYSCAPES_CLASS_WEIGHTS
    x = (3.0 * torch.randn(n, K, H, W, generator=g)).to(dev)
    lab = torch.randint(0, A, (n, H, W), generator=g)
    if case == "all_ignored_quads":
        lab[:, ::2] = ignore
    lab = lab.to(dev)
    wt = None if wts is None else torch.tensor(wts, device=dev)
    ref = torch.nn.CrossEntropyLoss(ignore_index=ignore, weight=wt)
    xr = x.clone().requires_grad_(True)
    lr = ref(xr, lab) * 0.7
    lr.backward()
    mod = mscs_b200.CrossEntropyLabelPass(A, ignore, wts).to(dev)
    xo = x.clone().requires_grad_(True)
    lo = mod(xo, lab)
    lo *= 0.7                                   # LossWrapper.py:90: in place on the returned tensor
    lo.backward()
    rel = abs(float(lo) - float(lr)) / abs(float(lr))
    err = float((xo.grad - xr.grad).abs().max()) / float(xr.grad.abs().max())
    print(f"{case}: loss {float(lo):.7f} ATen {float(lr):.7f} rel {rel:.1e}; gradient max-abs error / max {err:.1e}")
    assert rel < 1e-5 and err < 1e-5
    assert torch.equal(xo.grad == 0, xr.grad == 0) or float(xo.grad[(xo.grad == 0) != (xr.grad == 0)].abs().max()) < 1e-12


def test_k1_on_compact_labels_is_bit_exact(dev):
    import mscs_b200
    from mscs_b200 import synth
    cfg = synth.CONFIGS["cfg2"]
    labels, _ = synth.make_inputs("cfg2", with_features=False)
    feats = [torch.randn(12, 256, 512 // s, 1024 // s, device=dev) for s in cfg["strides"]]
    mod = mscs_b200.DenseContrastiveLossV2_ms(dict(cfg["loss"]))
    torch.manual_seed(0)
    with torch.no_grad():
        l64 = mod(labels.to(dev), feats)
    idx64 = [s.idx_ref.clone() for s in mod.last_samples]
    state64 = torch.get_rng_state()
    torch.manual_seed(0)
    with torch.no_grad():
        l16 = mod(mscs_b200.label_pass(labels.to(dev), 20), feats)
    assert torch.equal(torch.get_rng_state(), state64)
    assert all(torch.equal(a, s.idx_ref) for a, s in zip(idx64, mod.last_samples))
    assert float(l64) == float(l16)


# What the reference's LossWrapper builds for CrossEntropyLoss (LossWrapper.py:22-31), kept here independently of the
# code under test: (number of label ids incl. the ignore id, ignore_index, class weights).  The Cityscapes weights are
# the published HRNet Cityscapes cross-entropy weights the reference hard-codes; every other dataset is unweighted.
CE_SETUP = {
    "CITYSCAPES": (20, 19, [0.8373, 0.918, 0.866, 1.0345, 1.0166, 0.9969, 0.9754, 1.0489, 0.8786, 1.0023, 0.9539,
                            0.9843, 1.1116, 0.9037, 1.0865, 1.0955, 1.0865, 1.1529, 1.0507]),
    "ADE20K": (151, 150, None),
}


def test_fused_colosses_vs_aten_and_fp64_oracle(dev):
    """CrossEntropyLoss + DenseContrastiveLossV2_ms as the reference's LossWrapper combines them -- its
    ``nn.CrossEntropyLoss(ignore_index, weight)`` (ATen, this GPU, set up from CE_SETUP: class-weighted for Cityscapes)
    and the fp64 oracle of the contrastive loss, each weighted, same ``loss_vals`` keys -- against FusedCoLosses on the
    same inputs and generator state."""
    _colosses_vs_aten_and_fp64_oracle("CITYSCAPES", dev)


def test_fused_colosses_unweighted_dataset_vs_aten_and_fp64_oracle(dev):
    """The same for a dataset the reference's LossWrapper does not weight (ADE20K: plain cross entropy, ignore 150)."""
    _colosses_vs_aten_and_fp64_oracle("ADE20K", dev)


def _colosses_vs_aten_and_fp64_oracle(dataset, dev):
    import mscs_b200
    from mscs_b200 import synth
    from oracle import loss_fp64
    from oracle.config import oracle_cfg
    from oracle.mt19937 import MT19937
    A, ignore, class_weights = CE_SETUP[dataset]
    cfg = dict(dataset=dataset, experiment=1, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
               cross_scale_contrast=True, w_high_low=0.5, w_high_mid=0.25, min_views_per_class=5,
               max_views_per_class=40, max_features_total=1200,
               losses={"CrossEntropyLoss": 1.0, "DenseContrastiveLossV2_ms": 0.1}, device=dev)
    n, H, W = 3, 128, 256
    labels = synth.synth_labels(n, H, W, ignore, 7, 16, 0.05, 51).to(dev)
    g = torch.Generator().manual_seed(52)
    pred = (2.0 * torch.randn(n, A - 1, H, W, generator=g)).to(dev)
    feats = [torch.randn(n, 64, H // s, W // s, generator=g).to(dev) for s in (4, 8, 16)]
    torch.manual_seed(7)
    rng = torch.get_rng_state()

    w_ce, w_dc = cfg["losses"]["CrossEntropyLoss"], cfg["losses"]["DenseContrastiveLossV2_ms"]
    p = pred.clone().requires_grad_(True)
    wt = None if class_weights is None else torch.tensor(class_weights, device=dev)
    ce = torch.nn.CrossEntropyLoss(ignore_index=ignore, weight=wt)(p, labels)
    (w_ce * ce).backward()
    gen = MT19937.from_torch_state(rng.numpy().tobytes())
    dc = loss_fp64.ms_cs_loss(labels.cpu().numpy(), [f.cpu().numpy() for f in feats], oracle_cfg(cfg, A), gen)
    t_r = w_ce * float(ce) + w_dc * dc["total"]
    vals_r = {"CrossEntropyLoss": w_ce * float(ce), "DenseContrastiveLossV2_ms": w_dc * dc["total"]}
    vals_r.update({f"DenseContrastiveLossV2_ms_ms{i}": v for i, v in enumerate(dc["ms"])})
    vals_r.update({f"DenseContrastiveLossV2_ms_cs{i}": v for i, v in enumerate(dc["cs"])})
    gp_r = p.grad
    gf_r = [torch.from_numpy(w_dc * g) for g in dc["grads"]]

    wrapper = mscs_b200.FusedCoLosses(cfg)
    p = pred.clone().requires_grad_(True)
    f = [x.clone().requires_grad_(True) for x in feats]
    torch.set_rng_state(rng)
    total = wrapper(p, labels, deep_features=f)
    total.backward()
    torch.cuda.synchronize()
    t_o, vals_o = float(total), {k: float(v) for k, v in wrapper.loss_vals.items()}
    gp_o, gf_o = p.grad, [x.grad.cpu() for x in f]
    print(f"{dataset} co-losses: total {t_o:.6f} ATen cross entropy + fp64 oracle {t_r:.6f}")
    assert abs(t_o - t_r) < 1e-3 * abs(t_r)
    assert set(vals_o) == set(vals_r)
    for k in vals_r:
        assert abs(vals_o[k] - vals_r[k]) <= 1e-3 * abs(vals_r[k]) + 1e-6, (k, vals_o[k], vals_r[k])
    a, b = gp_o.double().flatten(), gp_r.double().flatten()
    assert float((a @ b) / (a.norm() * b.norm())) > 0.999999
    for go, gr in zip(gf_o, gf_r):
        a, b = go.double().flatten(), gr.double().flatten()
        assert float((a @ b) / (a.norm() * b.norm())) >= 0.999


def test_fused_cross_entropy_throughput_cityscapes_shape(dev):
    """HBM figures of the two CE kernels at the Cityscapes training shape (12 x 19 x 512 x 1024 fp32 logits = 478 MB),
    next to ATen's cross entropy on the same tensors (printed; CUDA events, 10 iterations after 3)."""
    import mscs_b200
    from mscs_b200.coloss import CITYSCAPES_CLASS_WEIGHTS
    n, K, H, W = 12, 19, 512, 1024
    x = torch.randn(n, K, H, W, device=dev)
    lab = torch.randint(0, 20, (n, H, W), device=dev)
    wt = torch.tensor(CITYSCAPES_CLASS_WEIGHTS, device=dev)
    ref = torch.nn.CrossEntropyLoss(ignore_index=19, weight=wt)
    mod = mscs_b200.CrossEntropyLabelPass(20, 19, CITYSCAPES_CLASS_WEIGHTS).to(dev)

    def timed(fn):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(10):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 10

    def step(m):
        xr = x.requires_grad_(True)
        xr.grad = None
        m(xr, lab).backward()
    t_ref, t_own = timed(lambda: step(ref)), timed(lambda: step(mod))
    gb = x.numel() * 4 / 1e9
    print(f"cross entropy fwd+bwd at 12x19x512x1024: fused {t_own:.3f} ms (label pass included; algorithmic traffic "
          f"{3 * gb:.2f} GB -> {3 * gb / t_own * 1e3:.0f} GB/s), ATen {t_ref:.3f} ms")
    assert t_own < t_ref
