"""bf16 / fp16 feature maps and logits read and written natively by the kernels (no fp32 copy of an input, gradients in
the input's dtype), against the fp32 path run on the exact fp32 widening of the same inputs.

What the half path makes deterministic is compared exactly: sampling, the gathered operand rows / unit rows / inverse
norms (a half element widens exactly, the arithmetic after the load is the fp32 kernel's), the dense gradient written
from the dx rows, and the cross-entropy dlogits.  The loss and end-to-end gradients go through the similarity kernels,
whose atomics accumulate in an order that changes from run to run: those are compared with tolerances (loss 2e-6
relative; gradients 3e-4 of their maximum plus one ulp of the half type).

The tests at the end (not marked gpu) check the argument validation of the element-type codes without a device."""
import ctypes as C

import pytest
import torch

HALF = [torch.bfloat16, torch.float16]
LAYOUTS = ["nchw", "channels_last"]
MS_CFG = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
              cross_scale_contrast=True, min_views_per_class=5, max_views_per_class=40, max_features_total=600)
SS_CFG = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, min_views_per_class=5, max_views_per_class=100,
              max_features_total=1000)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import mscs_b200
    assert mscs_b200.load().mscs_device_ok() == 1, "libmscs.so needs a compute-capability 10.x device"
    return torch.device("cuda:0")


def _case(name):
    """(module class, config, labels, fp32 maps) on the CPU."""
    import mscs_b200
    from mscs_b200 import synth
    if name == "cfg2":
        labels, feats = synth.make_inputs("cfg2")
        return mscs_b200.DenseContrastiveLossV2_ms, dict(synth.CONFIGS["cfg2"]["loss"]), labels, feats
    labels = synth.synth_labels(2, 128, 256, 19, 6, 16, 0.05, 1)
    if name == "ss":
        return mscs_b200.DenseContrastiveLossV2, dict(SS_CFG), labels, synth.synth_features(2, 64, 128, 256, [4], 2)
    cfg = dict(MS_CFG, detach_deepest=(name == "ms_detach"))
    return mscs_b200.DenseContrastiveLossV2_ms, cfg, labels, synth.synth_features(2, 128, 128, 256, [4, 8, 16], 2)


def _layout(x, layout):
    return x.contiguous(memory_format=torch.channels_last) if layout == "channels_last" else x.contiguous()


def _workspace(st):
    """Clones of what the gather left in the step's workspace, per scale: bf16 operand rows (N, C_pad), fp32 unit rows
    (N, C), inverse norms (N)."""
    sp, e = st.sp, st.entry
    so = sp.slab_off
    bsl = e.slab[so["bslab"]:so["bslab"] + 2 * sp.bslab_n].view(torch.bfloat16)
    fsl = e.slab[so["fslab"]:so["fslab"] + 4 * sp.fslab_n].view(torch.float32)
    out = []
    for s, smp in enumerate(st.samples):
        N, Cc = smp.N, sp.C
        out.append((bsl[sp.boff[s]:sp.boff[s] + N * sp.C_pad].view(N, sp.C_pad).clone(),
                    fsl[sp.foff[s][0]:sp.foff[s][0] + N * Cc].view(N, Cc).clone(),
                    fsl[sp.foff[s][1]:sp.foff[s][1] + N].clone()))
    return out


def _dx_rows(st):
    """The dx rows the one-pass dense writer consumed (k_dx_rows turns the gradient rows into them in place)."""
    sp, e = st.sp, st.entry
    so = sp.slab_off
    dF = e.slab[so["dF"]:so["dF"] + 4 * sp.dF_n].view(torch.float32)
    return [dF[sp.dF_off[s]:sp.dF_off[s] + smp.N * sp.C_pad].view(smp.N, sp.C_pad)[:, :sp.C].clone()
            for s, smp in enumerate(st.samples)]


def _run(cls, cfg, labels, maps, seed, grad_mask=None, dx_rows=False):
    """One forward + backward with torch.manual_seed(seed) in front; everything the comparisons need, cloned."""
    mod = cls(dict(cfg))
    grad_mask = grad_mask or [True] * len(maps)
    leaves = [m.detach().requires_grad_(g) for m, g in zip(maps, grad_mask)]
    torch.manual_seed(seed)
    loss = mod(labels, leaves[0] if cls.__name__ == "DenseContrastiveLossV2" else leaves)
    rng = torch.get_rng_state()
    st = mod.last_state
    rec = dict(total=float(loss.detach()), terms=st.term_loss.detach().double().cpu(), rng=rng,
               smp=[(s.idx_ref.cpu(), s.pair_ref.cpu(), s.pix.cpu()) for s in mod.last_samples], ws=_workspace(st),
               pix=[s.pix.long().cpu() for s in mod.last_samples])
    want = [x for x, g in zip(leaves, grad_mask) if g]
    grads = iter(torch.autograd.grad(loss, want))
    rec["grads"] = [next(grads) if g else None for g in grad_mask]
    if dx_rows:
        rec["dx"] = _dx_rows(st)
    return rec


def _close_grad(g, ref32, dtype):
    """g (half) against the fp32 path's gradient: 3e-4 of its maximum (run-to-run variation of the atomics) plus one
    ulp of the half type per element."""
    ref = ref32.to(dtype).float()
    mant = 7 if dtype == torch.bfloat16 else 10
    tol = 3e-4 * ref32.abs().max().item() + ref.abs() * 2.0 ** -mant + (2.0 ** -24 if dtype == torch.float16 else 0.0)
    assert bool(((g.float() - ref).abs() <= tol).all()), float((g.float() - ref).abs().max())


def _nonzero_pixels(g):
    return (g != 0).any(dim=1)


def _compare(nat, ref, maps):
    for (a, b) in zip(nat["smp"], ref["smp"]):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    assert torch.equal(nat["rng"], ref["rng"])
    for (b1, f1, i1), (b2, f2, i2) in zip(nat["ws"], ref["ws"]):
        assert torch.equal(b1, b2) and torch.equal(f1, f2) and torch.equal(i1, i2)
    assert abs(nat["total"] - ref["total"]) <= 2e-6 * abs(ref["total"])
    assert torch.allclose(nat["terms"], ref["terms"], rtol=2e-6, atol=0)
    for m, g, g32 in zip(maps, nat["grads"], ref["grads"]):
        if g is None:
            continue
        assert g.dtype == m.dtype and g.shape == m.shape and g.stride() == m.stride()
        assert torch.equal(_nonzero_pixels(g), _nonzero_pixels(g32.to(g.dtype)))
        _close_grad(g, g32, g.dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("name", ["ms", "ms_detach", "ss", "cfg2"])
def test_half_maps_match_fp32_on_widened_maps(name, dtype, layout, dev):
    cls, cfg, labels, feats = _case(name)
    labels = labels.to(dev)
    maps = [_layout(f.to(dev).to(dtype), layout) for f in feats]
    nchw = layout == "nchw"
    nat = _run(cls, cfg, labels, maps, 11, dx_rows=nchw)
    ref = _run(cls, cfg, labels, [m.float() for m in maps], 11)
    _compare(nat, ref, maps)
    if nchw:      # the dense writer: zeros, and each sampled pixel's dx row rounded to the dtype -- exactly
        for m, g, dx, pix in zip(maps, nat["grads"], nat["dx"], nat["pix"]):
            n, Cc, h, w = m.shape
            want = torch.zeros(n * h * w, Cc, dtype=dtype, device=dev)
            want[pix.to(dev)] = dx.to(dtype)
            assert torch.equal(g, want.view(n, h * w, Cc).permute(0, 2, 1).reshape(n, Cc, h, w))


@pytest.mark.gpu
def test_half_maps_peak_memory_cfg2(dev):
    """bf16 NCHW at cfg-2: one forward + backward allocates less than one fp32 copy of the maps (534.8 MB)."""
    cls, cfg, labels, feats = _case("cfg2")
    labels = labels.to(dev)
    leaves = [f.to(dev).to(torch.bfloat16).requires_grad_(True) for f in feats]
    del feats
    mod = cls(dict(cfg))

    def step():
        loss = mod(labels, leaves)
        grads = torch.autograd.grad(loss, leaves)
        del loss, grads

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    step()
    torch.cuda.synchronize()
    grew = torch.cuda.max_memory_allocated(dev) - base
    assert grew < 534.8e6, f"{grew / 1e6:.1f} MB"


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_half_maps_second_backward_and_no_grad(layout, dev):
    cls, cfg, labels, feats = _case("ms")
    labels = labels.to(dev)
    maps = [_layout(f.to(dev).to(torch.bfloat16), layout) for f in feats]
    mod = cls(dict(cfg))
    leaves = [m.detach().requires_grad_(True) for m in maps]
    torch.manual_seed(3)
    loss = mod(labels, leaves)
    g1 = torch.autograd.grad(loss, leaves, retain_graph=True)
    g2 = torch.autograd.grad(loss, leaves)
    for m, a, b in zip(maps, g1, g2):
        assert b.dtype == m.dtype and b.stride() == m.stride()
        assert torch.equal(_nonzero_pixels(a), _nonzero_pixels(b))
        _close_grad(b, a.float(), m.dtype)
    with torch.no_grad():
        torch.manual_seed(3)
        l_ng = mod(labels, maps)
        torch.manual_seed(3)
        l_32 = cls(dict(cfg))(labels, [m.float() for m in maps])
    assert abs(float(l_ng) - float(l_32)) <= 2e-6 * abs(float(l_32))
    assert abs(float(l_ng) - float(loss.detach())) <= 2e-6 * abs(float(loss.detach()))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_half_maps_partial_needs(layout, dev):
    """One scale detached: the backward allocates the gradients of the others itself, in the maps' dtype."""
    cls, cfg, labels, feats = _case("ms")
    labels = labels.to(dev)
    maps = [_layout(f.to(dev).to(torch.float16), layout) for f in feats]
    mask = [True, False, True]
    nat = _run(cls, cfg, labels, maps, 5, grad_mask=mask)
    ref = _run(cls, cfg, labels, [m.float() for m in maps], 5, grad_mask=mask)
    _compare(nat, ref, maps)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_mixed_fp32_and_bf16_maps(layout, dev):
    import mscs_b200
    from mscs_b200 import synth
    cfg = dict(MS_CFG, scales=2, weights=[1.0, 0.7])
    labels = synth.synth_labels(2, 128, 256, 19, 6, 16, 0.05, 1).to(dev)
    f0, f1 = synth.synth_features(2, 128, 128, 256, [4, 8], 2)
    maps = [_layout(f0.to(dev), layout), _layout(f1.to(dev).to(torch.bfloat16), layout)]
    cls = mscs_b200.DenseContrastiveLossV2_ms
    nat = _run(cls, cfg, labels, maps, 9)
    ref = _run(cls, cfg, labels, [m.float() for m in maps], 9)
    assert nat["grads"][0].dtype == torch.float32 and nat["grads"][1].dtype == torch.bfloat16
    _compare(nat, ref, maps)


# ---- cross entropy ---------------------------------------------------------------------------------------------
def _ce_inputs(dev, n=2, H=128, W=256):
    from mscs_b200 import synth
    g = torch.Generator().manual_seed(21)
    labels = synth.synth_labels(n, H, W, 19, 7, 16, 0.05, 22).to(dev)
    logits = (2.0 * torch.randn(n, 19, H, W, generator=g)).to(dev)
    return labels, logits


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_fused_ce_half_logits(dtype, dev):
    import mscs_b200
    from mscs_b200.coloss import CITYSCAPES_CLASS_WEIGHTS
    labels, logits = _ce_inputs(dev)
    x = logits.to(dtype)
    ce = mscs_b200.CrossEntropyLabelPass(20, 19, CITYSCAPES_CLASS_WEIGHTS).to(dev)
    compact = mscs_b200.label_pass(labels, 20)
    xh, x32 = x.clone().requires_grad_(True), x.float().requires_grad_(True)
    lh, l32 = ce(xh, compact), ce(x32, compact)
    dh, = torch.autograd.grad(lh, xh)
    d32, = torch.autograd.grad(l32, x32)
    assert dh.dtype == dtype and dh.shape == x.shape
    assert torch.equal(dh, d32.to(dtype))
    assert abs(float(lh) - float(l32)) <= 1e-7 * abs(float(l32))


@pytest.mark.gpu
def test_fused_ce_half_forward_allocates_no_copy(dev):
    import mscs_b200
    labels, logits = _ce_inputs(dev, 2, 256, 512)          # an fp32 copy of these logits would be 19.9 MB
    x = logits.to(torch.bfloat16).requires_grad_(True)
    ce = mscs_b200.CrossEntropyLabelPass(20, 19)
    compact = mscs_b200.label_pass(labels, 20)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    loss = ce(x, compact)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated(dev) - base < 1e6
    del loss


@pytest.mark.gpu
def test_fused_colosses_bf16(dev):
    import mscs_b200
    from mscs_b200 import synth
    cfg = dict(MS_CFG, losses={"CrossEntropyLoss": 1.0, "DenseContrastiveLossV2_ms": 0.1})
    labels, logits = _ce_inputs(dev)
    feats = [f.to(dev).to(torch.bfloat16) for f in synth.synth_features(2, 128, 128, 256, [4, 8, 16], 2)]
    vals = []
    for cast in (lambda t: t, lambda t: t.float()):
        w = mscs_b200.FusedCoLosses(dict(cfg))
        torch.manual_seed(4)
        total = w(cast(logits.to(torch.bfloat16)), labels, deep_features=[cast(f) for f in feats])
        vals.append({k: float(v) for k, v in w.loss_vals.items()} | {"total": float(total.detach())})
    nat, ref = vals
    assert nat.keys() == ref.keys()
    for k in ref:
        tol = 1e-7 if k == "CrossEntropyLoss" else 2e-6
        assert abs(nat[k] - ref[k]) <= tol * abs(ref[k]) + 1e-12, k


# ---- argument validation (no device) ---------------------------------------------------------------------------
_FAKE = 0x100000        # a 1 MiB-aligned address that is never dereferenced: validation fails first


def _expect_bad(rc, lib):
    assert rc < 0 and b"dtype" in lib.mscs_last_error()


@pytest.mark.parametrize("bad", [-1, 3])
def test_bad_dtype_in_batched_items_is_rejected(bad):
    import mscs_b200
    from mscs_b200 import _lib
    lib = mscs_b200.load()
    g = (_lib.GatherItem * 1)()
    g[0].feat = g[0].slot = g[0].n_rows_dev = g[0].anc_bf16 = g[0].anc_f32 = g[0].inv_norm = _FAKE
    g[0].n, g[0].C, g[0].plane, g[0].dtype = 1, 64, 8, bad
    _expect_bad(lib.mscs_gather_normalize_sectors_batch(g, 1, None), lib)
    r = (_lib.RowsItem * 1)()
    r[0].feat = r[0].pix = r[0].anc_bf16 = r[0].anc_f32 = r[0].inv_norm = r[0].dF = r[0].dfeat = _FAKE
    r[0].rows, r[0].C, r[0].ldF, r[0].dtype = 1, 64, 64, bad
    _expect_bad(lib.mscs_gather_rows_nhwc_batch(r, 1, None), lib)
    _expect_bad(lib.mscs_scatter_rows_nhwc_batch(r, 1, None), lib)
    sc = (_lib.ScatterItem * 1)()
    sc[0].dF = sc[0].anc_f32 = sc[0].inv_norm = sc[0].slot = sc[0].dfeat = _FAKE
    sc[0].ldF, sc[0].n, sc[0].C, sc[0].plane, sc[0].dtype = 64, 1, 64, 8, bad
    rows = (C.c_int32 * 1)(1)
    _expect_bad(lib.mscs_scatter_dense_batch(sc, rows, 1, None), lib)
    _expect_bad(lib.mscs_scatter_sectors_batch(sc, 1, None), lib)


@pytest.mark.parametrize("bad", [-1, 3])
def test_bad_dtype_in_ce_is_rejected(bad):
    import mscs_b200
    lib = mscs_b200.load()
    _expect_bad(lib.mscs_ce_forward(_FAKE, _FAKE, 1, 19, 8, None, 19, _FAKE, 20, _FAKE, _FAKE, None, bad), lib)
    _expect_bad(lib.mscs_ce_backward(_FAKE, _FAKE, 1, 19, 8, None, 19, _FAKE, _FAKE, _FAKE, None, bad), lib)


def test_half_items_rejected_by_fp32_sector_scatter():
    import mscs_b200
    from mscs_b200 import _lib
    lib = mscs_b200.load()
    sc = (_lib.ScatterItem * 1)()
    sc[0].dF = sc[0].anc_f32 = sc[0].inv_norm = sc[0].slot = sc[0].dfeat = _FAKE
    sc[0].ldF, sc[0].n, sc[0].C, sc[0].plane, sc[0].dtype = 64, 1, 64, 8, _lib.DTYPE_F16
    assert lib.mscs_scatter_sectors_batch(sc, 1, None) < 0 and b"fp32" in lib.mscs_last_error()
