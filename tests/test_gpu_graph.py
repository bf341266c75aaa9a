"""CUDA-graph capture of the loss with sampler='philox': a captured forward + backward, replayed with fresh inputs copied
into the static tensors, against eager calls of a module of the same configuration whose host call index is set to the
replay's device call index (2**62 + r).

Sampling is compared exactly (the same Philox words, the same selection kernel).  The loss, logged terms and gradients
go through the similarity kernels, whose atomics accumulate in an order that changes from run to run: loss and terms
within 2e-6 relative, gradients within 3e-4 of their maximum plus one ulp of their type (as test_gpu_half_io.py)."""
import pytest
import torch

BASE = 2 ** 62
MS_CFG = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, scales=3, weights=[1.0, 0.7, 0.4],
              cross_scale_contrast=True, min_views_per_class=5, max_views_per_class=40, max_features_total=600,
              sampler="philox", sampler_seed=7)
SS_CFG = dict(dataset="CITYSCAPES", experiment=1, temperature=0.1, min_views_per_class=5, max_views_per_class=100,
              max_features_total=1000, sampler="philox", sampler_seed=3)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    import mscs_b200
    assert mscs_b200.load().mscs_device_ok() == 1, "libmscs.so needs a compute-capability 10.x device"
    return torch.device("cuda:0")


def _inputs(r, dev, dtype=torch.float32, layout="nchw", name="small"):
    """Labels and maps of replay r (fresh features every replay, labels from a seed of their own)."""
    from mscs_b200 import synth
    if name == "cfg2":
        labels, feats = synth.make_inputs("cfg2")
        g = torch.Generator().manual_seed(100 + r)
        feats = [f + 0.05 * torch.randn(f.shape, generator=g) for f in feats]
    else:
        labels = synth.synth_labels(2, 128, 256, 19, 6, 16, 0.05, 1 + r)
        feats = synth.synth_features(2, 128, 128, 256, [4, 8, 16], 10 + r)
    fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
    return labels.to(dev), [f.to(dev, dtype).contiguous(memory_format=fmt) for f in feats]


def _cfg(name):
    if name == "cfg2":
        from mscs_b200 import synth
        return dict(synth.CONFIGS["cfg2"]["loss"], sampler="philox", sampler_seed=11)
    return dict(MS_CFG)


def _capture(mod, labels, maps, grad=True):
    """One eager warm-up call on a side stream, then the capture of forward (+ backward).  Returns (graph, static
    labels, static maps, static loss, static gradients)."""
    st_lab = labels.clone()
    st_maps = [m.detach().clone().requires_grad_(grad) for m in maps]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.set_grad_enabled(grad):
        loss = mod(st_lab, st_maps)
        if grad:
            torch.autograd.grad(loss, st_maps)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    grads = None
    with torch.cuda.graph(g), torch.set_grad_enabled(grad):
        loss = mod(st_lab, st_maps)
        if grad:
            grads = torch.autograd.grad(loss, st_maps)
    return g, st_lab, st_maps, loss, grads


def _replay(g, st_lab, st_maps, labels, maps):
    with torch.no_grad():
        st_lab.copy_(labels)
        for s, m in zip(st_maps, maps):
            s.copy_(m)
    g.replay()


def _eager(cls, cfg, call, labels, maps, grad=True):
    mod = cls(dict(cfg))
    mod._sampler_calls = call
    leaves = [m.detach().clone().requires_grad_(grad) for m in maps]
    with torch.set_grad_enabled(grad):
        loss = mod(labels, leaves)
        grads = torch.autograd.grad(loss, leaves) if grad else None
    return mod, loss, grads


def _close_grad(g, ref, rel=3e-4):
    mant = {torch.float32: 23, torch.bfloat16: 7, torch.float16: 10}[ref.dtype]
    r = ref.float()
    tol = rel * r.abs().max().item() + r.abs() * 2.0 ** -mant
    assert bool(((g.float() - r).abs() <= tol).all()), float((g.float() - r).abs().max())


def _check_replay(mod, eager_mod, loss, eager_loss, grads, eager_grads, grad_rel=3e-4):
    got, want = mod.fetch_samples(), eager_mod.fetch_samples()
    for a, b in zip(got, want):
        assert (a.T, a.V, a.N) == (b.T, b.V, b.N)
        assert torch.equal(a.idx_ref, b.idx_ref) and torch.equal(a.pair_ref, b.pair_ref) and torch.equal(a.pix, b.pix)
    lg, le = mod.fetch_logged(), eager_mod.fetch_logged()
    assert abs(float(loss) - float(eager_loss)) <= 2e-6 * abs(float(eager_loss))
    for k in ("ms_losses", "cs_losses"):
        assert len(lg[k]) == len(le[k])
        for x, y in zip(lg[k], le[k]):
            assert abs(x - y) <= 2e-6 * abs(y), (k, x, y)
    assert lg["has_inf_or_nan"] is False
    if grads is not None:
        for g, ge in zip(grads, eager_grads):
            assert g.dtype == ge.dtype and g.shape == ge.shape and g.stride() == ge.stride()
            _close_grad(g, ge, grad_rel)
    return [s.pix.clone() for s in got]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_replays_match_eager(layout, dtype, dev):
    import mscs_b200
    cls = mscs_b200.DenseContrastiveLossV2_ms
    mod = cls(dict(MS_CFG))
    labels, maps = _inputs(0, dev, dtype, layout)
    g, st_lab, st_maps, loss, grads = _capture(mod, labels, maps)
    assert mod._sampler_calls == 1 and int(mod.graph_call_index) == BASE       # the capture advanced neither
    rng = torch.get_rng_state()
    prev = None
    for r in range(3):
        _, fresh = _inputs(r + 1, dev, dtype, layout)       # same labels, fresh maps: the pixels must still change
        _replay(g, st_lab, st_maps, labels, fresh)
        em, el, eg = _eager(cls, MS_CFG, BASE + r, labels, fresh)
        pix = _check_replay(mod, em, loss, el, grads, eg)
        if prev is not None:
            assert any(not torch.equal(a, b) for a, b in zip(pix, prev)), "consecutive replays sampled the same pixels"
        prev = pix
    assert int(mod.graph_call_index) == BASE + 3
    assert torch.equal(rng, torch.get_rng_state())
    assert mod._sampler_calls == 1


@pytest.mark.gpu
def test_replay_matches_eager_cfg2(dev):
    import mscs_b200
    cls = mscs_b200.DenseContrastiveLossV2_ms
    cfg = _cfg("cfg2")
    mod = cls(dict(cfg))
    labels, maps = _inputs(0, dev, name="cfg2")
    g, st_lab, st_maps, loss, grads = _capture(mod, labels, maps)
    _, fresh = _inputs(1, dev, name="cfg2")
    _replay(g, st_lab, st_maps, labels, fresh)
    em, el, eg = _eager(cls, cfg, BASE, labels, fresh)
    _check_replay(mod, em, loss, el, grads, eg)


@pytest.mark.gpu
def test_whole_training_step_captured(dev):
    """1x1 projector + loss + backward + SGD step in one graph, against the eager sequence with the same call indices."""
    import mscs_b200
    torch.manual_seed(5)
    proj = torch.nn.Conv2d(32, 64, 1).to(dev)
    ref = torch.nn.Conv2d(32, 64, 1).to(dev)
    mod = mscs_b200.DenseContrastiveLossV2_ms(dict(MS_CFG))
    emod = mscs_b200.DenseContrastiveLossV2_ms(dict(MS_CFG))
    # (the parameter difference is lr x the run-to-run variation of the weight gradients: lr 0.5 gave 2.3e-4 relative)
    opt = torch.optim.SGD(proj.parameters(), lr=0.1)
    eopt = torch.optim.SGD(ref.parameters(), lr=0.1)
    gen = torch.Generator().manual_seed(0)

    def inputs():
        from mscs_b200 import synth
        lab = synth.synth_labels(2, 128, 256, 19, 6, 16, 0.05, 1).to(dev)
        return lab, [torch.randn(2, 32, 128 // s, 256 // s, generator=gen).to(dev) for s in (4, 8, 16)]

    def step(m, o, loss_mod, lab, xs):
        o.zero_grad(set_to_none=False)
        loss = loss_mod(lab, [m(x) for x in xs])
        loss.backward()
        o.step()

    lab, xs = inputs()
    st_lab, st_xs = lab.clone(), [x.clone() for x in xs]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step(proj, opt, mod, st_lab, st_xs)      # warm-up (eager call index 0)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step(proj, opt, mod, st_lab, st_xs)
    ref.load_state_dict(proj.state_dict())
    for r in range(3):
        lab, xs = inputs()
        with torch.no_grad():
            st_lab.copy_(lab)
            for a, b in zip(st_xs, xs):
                a.copy_(b)
        g.replay()
        emod._sampler_calls = BASE + r
        step(ref, eopt, emod, lab, xs)
    torch.cuda.synchronize()
    for p, q in zip(proj.parameters(), ref.parameters()):
        assert float((p - q).abs().max()) <= 1e-4 * float(q.abs().max())
    assert int(mod.graph_call_index) == BASE + 3


@pytest.mark.gpu
def test_forward_only_capture_no_grad(dev):
    import mscs_b200
    cls = mscs_b200.DenseContrastiveLossV2_ms
    mod = cls(dict(MS_CFG))
    labels, maps = _inputs(0, dev)
    with torch.no_grad():
        g, st_lab, st_maps, loss, _ = _capture(mod, labels, maps, grad=False)
    _, fresh = _inputs(1, dev)
    _replay(g, st_lab, st_maps, labels, fresh)
    em, el, _ = _eager(cls, MS_CFG, BASE, labels, fresh, grad=False)
    _check_replay(mod, em, loss, el, None, None)


@pytest.mark.gpu
def test_plan_error_during_replay(dev):
    """Labels that keep no pair: NaN loss, nan_flag 1, zero gradients, fetch_logged raises; the next replay is right."""
    import mscs_b200
    cls = mscs_b200.DenseContrastiveLossV2_ms
    mod = cls(dict(MS_CFG))
    labels, maps = _inputs(0, dev)
    g, st_lab, st_maps, loss, grads = _capture(mod, labels, maps)
    bad = torch.full_like(labels, 19)            # only the dropped last class: no (image, class) pair is kept
    _replay(g, st_lab, st_maps, bad, maps)
    torch.cuda.synchronize()
    assert torch.isnan(loss).item() and float(mod.nan_flag) == 1.0
    assert all(int((x != 0).sum()) == 0 for x in grads)
    with pytest.raises(RuntimeError, match="no \\(image, class\\) pair"):
        mod.fetch_logged()
    _, fresh = _inputs(1, dev)
    _replay(g, st_lab, st_maps, labels, fresh)
    em, el, eg = _eager(cls, MS_CFG, BASE + 1, labels, fresh)
    # (this checks recovery, not the accumulation order: the gradients of this small case carry more cancellation, and
    # the atomics' run-to-run variation has been seen at 4e-4 of their maximum)
    _check_replay(mod, em, loss, el, grads, eg, grad_rel=1e-3)
    assert float(mod.nan_flag) == 0.0


def _refused(fn):
    g = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="cannot be captured"):
        with torch.cuda.graph(g):
            fn()
    torch.cuda.synchronize()                      # the capture ended cleanly: the device is usable
    assert float(torch.ones(4, device="cuda").sum()) == 4.0


@pytest.mark.gpu
def test_refusals(dev):
    import mscs_b200
    from mscs_b200 import synth
    labels, maps = _inputs(0, dev)
    ref_cfg = {k: v for k, v in MS_CFG.items() if k not in ("sampler", "sampler_seed")}
    mod = mscs_b200.DenseContrastiveLossV2_ms(ref_cfg)
    mod(labels, maps)
    _refused(lambda: mod(labels, maps))                                      # reference sampler
    odd = mscs_b200.DenseContrastiveLossV2(dict(SS_CFG))
    lab_odd = synth.synth_labels(2, 60, 100, 19, 6, 4, 0.05, 1).to(dev)
    f_odd = torch.randn(2, 16, 15, 25, device=dev)
    _refused(lambda: odd(lab_odd, f_odd))                                    # planes not a multiple of 8 pixels
    cs = mscs_b200.DenseContrastiveLossV2(dict(SS_CFG, cross_scale_contrast=True))
    cs(labels, maps[0])
    _refused(lambda: cs(labels, maps[0]))                                    # single-scale cross-scale 4-tuple
    fresh = mscs_b200.DenseContrastiveLossV2_ms(dict(MS_CFG))
    _refused(lambda: fresh(labels, maps))                                    # no eager call before the capture


@pytest.mark.gpu
def test_graph_workspace_is_isolated(dev):
    import mscs_b200
    cls = mscs_b200.DenseContrastiveLossV2_ms
    mod = cls(dict(MS_CFG))
    labels, maps = _inputs(0, dev)
    g, st_lab, st_maps, loss, grads = _capture(mod, labels, maps)
    gstate = mod.last_state
    _, fresh = _inputs(1, dev)
    _replay(g, st_lab, st_maps, labels, fresh)
    logged = mod.fetch_logged()
    pix = [s.pix.clone() for s in mod.fetch_samples()]
    for _ in range(2):                      # eager calls on the same module: workspaces of the eager pool
        leaves = [m.detach().clone().requires_grad_(True) for m in maps]
        torch.autograd.grad(mod(labels, leaves), leaves)
        assert mod.last_state.entry.slab.data_ptr() != gstate.entry.slab.data_ptr()
    torch.cuda.synchronize()
    again = mod.fetch_logged(gstate)
    assert {k: v for k, v in again.items() if k != "log_this_step"} == \
        {k: v for k, v in logged.items() if k != "log_this_step"}
    assert all(torch.equal(a.pix, b) for a, b in zip(mod.fetch_samples(gstate), pix))
